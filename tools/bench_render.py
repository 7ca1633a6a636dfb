"""Cost of cn_env_render (K7, csrc/render.cu) on one GPU, at the c3 config (20 humans, robot FOV 0.5 pi, holonomic).

* Kernel time: CUDA events around `--reps` back-to-back launches into one preallocated output, for k in {64, 1024, 16384}
  frames x S in {128, 256}.  Frames/s and the achieved write rate (3 S^2 bytes per frame) against the data sheet's
  7.7 TB/s of HBM3e.  The outputs of the large cases (>= 805 MB) do not fit the 126 MB L2, so those writes reach HBM.
* Rollout cost: a GraphedRollout at c3 (16384 envs) stepped `--steps` times with and without rendering 64 envs at
  S = 256 after every step, the two arms alternating `--rounds` times in the same process; device time from CUDA events.

    python tools/bench_render.py > profiles/r3_render.txt
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from crowdnav_dsrnn_b200 import Config  # noqa: E402
from crowdnav_dsrnn_b200.envs import CrowdVecEnv  # noqa: E402
from crowdnav_dsrnn_b200.model import Policy  # noqa: E402
from crowdnav_dsrnn_b200.rollout import GraphedRollout  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def c3_config():
    cfg = Config(human_num=20)
    cfg.robot.FOV = 0.5
    return cfg


def kernel_table(eng, reps):
    print("kernel: cn_env_render, CUDA events over %d launches after %d warm-up launches" % (reps, 3))
    print("%7s %5s %10s %12s %12s %10s" % ("k", "S", "ms/launch", "frames/s", "write GB/s", "of 7.7TB/s"))
    for k in (64, 1024, 16384):
        ids = (torch.arange(k, device=eng.device, dtype=torch.int32) * 7919 % eng.n).to(torch.int32)
        for S in (128, 256):
            out = torch.empty(k, S, S, 3, dtype=torch.uint8, device=eng.device)
            for _ in range(3):
                eng.render(ids, size=S, out=out)
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            t0.record()
            for _ in range(reps):
                eng.render(ids, size=S, out=out)
            t1.record()
            torch.cuda.synchronize()
            ms = t0.elapsed_time(t1) / reps
            rate = 3.0 * S * S * k / (ms * 1e-3)
            print("%7d %5d %10.4f %12.4g %12.1f %9.1f%%" % (k, S, ms, k / (ms * 1e-3), rate / 1e9, 100.0 * rate / HBM_BYTES_PER_S))
            del out


def rollout_cost(cfg, steps, rounds):
    dev = torch.device("cuda:0")
    n = 16384
    venv = CrowdVecEnv(cfg, n, dev, seed=1, phase="train")
    policy = Policy(venv.observation_space.spaces, venv.action_space, base="srnn", base_kwargs=cfg)
    w = np.load(os.path.join(GOLDEN, "weights_holonomic_27776.npz"))
    policy.load_state_dict({k: torch.from_numpy(w[k]) for k in w.files})
    policy = policy.to(dev)
    policy.precision = "bf16x3"
    obs = venv.reset()
    roll = GraphedRollout(policy, venv, obs)
    ids = torch.arange(64, device=dev, dtype=torch.int32)
    out = torch.empty(64, 256, 256, 3, dtype=torch.uint8, device=dev)
    for _ in range(20):                    # warm-up of both arms
        roll.step()
        venv.engine.render(ids, size=256, out=out)
    times = {False: [], True: []}
    for _ in range(rounds):
        for render in (False, True):
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            t0.record()
            for _ in range(steps):
                roll.step()
                if render:
                    venv.engine.render(ids, size=256, out=out)
            t1.record()
            torch.cuda.synchronize()
            times[render].append(t0.elapsed_time(t1) / steps)
    roll.close()
    venv.close()
    print("rollout: GraphedRollout c3 (16384 envs x 20 humans, bf16x3), %d steps per round, %d rounds alternating" % (steps, rounds))
    for render in (False, True):
        t = np.array(times[render])
        print("  %-34s ms/step median %.4f  min %.4f  max %.4f" % ("with render of 64 envs at S=256" if render else "without render",
                                                                     np.median(t), t.min(), t.max()))
    d = np.median(times[True]) - np.median(times[False])
    print("  render cost per step (median difference): %.4f ms = %.2f %% of a step" % (d, 100.0 * d / np.median(times[False])))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    print("card: %s" % card)
    cfg = c3_config()
    from crowdnav_dsrnn_b200.engine import CrowdEngine
    eng = CrowdEngine(cfg, 16384, torch.device("cuda:0"), phase="train", seed=1)
    eng.reset()
    kernel_table(eng, args.reps)
    eng.close()
    rollout_cost(cfg, args.steps, args.rounds)


if __name__ == "__main__":
    main()
