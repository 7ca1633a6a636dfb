"""Cost and outcomes of the model-based robots (robot.policy = orca / social_force, cn_env_robot_act, kernel K8).

* Kernel time at c3 (16384 envs x 20 humans, robot FOV 0.5 pi, holonomic): CUDA events around `--reps` back-to-back
  launches of cn_env_robot_act after warm-up, for both policies, on the state of a running rollout.
* Step cost: the crowd step (auto-reset on) with a fixed action tensor, and cn_env_robot_act + the same step, the two arms
  alternating `--rounds` times in the same process, `--steps` steps per round; device time from CUDA events.
* Outcomes: evaluate_batched over `--episodes` test episodes for the ORCA robot, the social-force robot and DS-RNN with the
  shipped checkpoint 27776.pt (tests/golden/weights_holonomic_27776.npz), at the defaults (5 humans, FOV 2 pi) and at
  20 humans with FOV 0.5 pi.

    python tools/bench_robot_act.py > profiles/r3_robot_act.txt
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from crowdnav_dsrnn_b200 import Config  # noqa: E402
from crowdnav_dsrnn_b200.engine import CrowdEngine  # noqa: E402
from crowdnav_dsrnn_b200.evaluation import evaluate_batched  # noqa: E402
from crowdnav_dsrnn_b200.model import Policy  # noqa: E402
from crowdnav_dsrnn_b200.spaces import crowd_spaces  # noqa: E402

DEV = torch.device("cuda:0")


def config(H, fov, policy="srnn"):
    cfg = Config(human_num=H)
    cfg.robot.FOV = fov
    cfg.robot.policy = policy
    return cfg


def timed(fn, reps):
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    for _ in range(reps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / reps


def kernel_and_step(reps, steps, rounds):
    n = 16384
    eng = CrowdEngine(config(20, 0.5), n, DEV, phase="train", seed=1)
    eng.reset()
    act = torch.empty(n, 2, device=DEV)
    for _ in range(50):                     # a running rollout: episodes at every stage, spares in flight
        eng.step(eng.robot_act("orca", out=act), auto_reset=True)
    print("kernel: cn_env_robot_act at c3 (16384 envs x 20 humans, FOV 0.5 pi), CUDA events over %d launches after 20 warm-up"
          % reps)
    for policy in ("orca", "social_force"):
        for _ in range(20):
            eng.robot_act(policy, out=act)
        ms = [timed(lambda: eng.robot_act(policy, out=act), reps) for _ in range(3)]
        print("  %-13s us/launch %.2f  (3 repeats: %s)" % (policy, 1e3 * np.median(ms), " ".join("%.2f" % (1e3 * m) for m in ms)))
    fixed = act.clone()
    arms = {"step": lambda: eng.step(fixed, auto_reset=True),
            "robot_act + step": lambda: eng.step(eng.robot_act("orca", out=act), auto_reset=True)}
    for fn in arms.values():
        for _ in range(20):
            fn()
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(timed(fn, steps))
    eng.join()
    torch.cuda.synchronize()
    eng.close()
    print("step: crowd step with auto-reset at c3, %d steps per round, %d rounds alternating" % (steps, rounds))
    for k, t in times.items():
        t = np.array(t)
        print("  %-18s ms/step median %.4f  min %.4f  max %.4f" % (k, np.median(t), t.min(), t.max()))
    d = np.median(times["robot_act + step"]) - np.median(times["step"])
    print("  robot_act cost per step (median difference): %.4f ms = %.2f %% of a step" % (d, 100.0 * d / np.median(times["step"])))


def outcomes(episodes):
    w = np.load(os.path.join(ROOT, "tests", "golden", "weights_holonomic_27776.npz"))
    sd = {k: torch.from_numpy(w[k]) for k in w.files}
    print("outcomes: evaluate_batched, %d test episodes each (default test scenarios; path length: mean over all episodes)" % episodes)
    print("  %-28s %-22s %8s %9s %8s %13s %12s" % ("setting", "robot", "success", "collision", "timeout", "nav time [s]",
                                                  "path len [m]"))
    for label, H, fov in (("defaults (5 humans, FOV 2)", 5, 2.0), ("20 humans, FOV 0.5", 20, 0.5)):
        for robot in ("orca", "social_force", "srnn"):
            cfg = config(H, fov, robot)
            policy = None
            if robot == "srnn":
                obs, act = crowd_spaces(H)
                policy = Policy(obs.spaces, act, base="srnn", base_kwargs=cfg)
                policy.load_state_dict(sd)
                policy = policy.to(DEV)
            r = evaluate_batched(policy, cfg, DEV, episodes=episodes)
            assert r["unfinished"] == 0
            name = "DS-RNN (27776.pt)" if robot == "srnn" else {"orca": "ORCA", "social_force": "social force"}[robot]
            print("  %-28s %-22s %8.3f %9.3f %8.3f %13.2f %12.2f" % (label, name, r["success"], r["collision"], r["timeout"],
                                                                   r["mean_nav_time_success"], r["mean_path_length"]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2000)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--episodes", type=int, default=2000)
    args = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    print("card: %s" % card)
    kernel_and_step(args.reps, args.steps, args.rounds)
    outcomes(args.episodes)


if __name__ == "__main__":
    main()
