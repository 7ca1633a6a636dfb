"""Record test episodes of a checkpoint (or of a model-based robot) as PNG frames drawn on the GPU (CrowdEngine.render, K7).

Plays `--episodes k` test episodes in one batch, deterministically, the way `evaluate_batched` starts them (env k plays
test case k), and renders every step of every env until that env's first episode ends, the last frame showing the end
(collision, goal or timeout).  Writes <out>/env<k>/<step>.png (step 0 is the reset) and, with --tile, <out>/tile/<step>.png
with all envs in baselines' tile_images layout.  PNGs are written with stdlib zlib; nothing else is needed.

    python tools/render_episodes.py --checkpoint tests/golden/weights_holonomic_27776.npz --episodes 16 --out frames
    python tools/render_episodes.py --robot_policy orca --episodes 16 --out frames_orca      # no checkpoint: robot.policy
"""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from crowdnav_dsrnn_b200 import Config  # noqa: E402
from crowdnav_dsrnn_b200.envs import CrowdVecEnv  # noqa: E402
from crowdnav_dsrnn_b200.model import Policy  # noqa: E402
from crowdnav_dsrnn_b200.render import check_size, tile_images, write_png  # noqa: E402


def load_weights(path):
    if path.endswith(".npz"):
        w = np.load(path)
        return {k: torch.from_numpy(w[k]) for k in w.files}
    return torch.load(path, map_location="cpu", weights_only=True)


@torch.no_grad()
def record(config, state_dict, episodes, out, size=256, tile=False, device="cuda:0", seed=None, max_steps=None):
    """Returns {env: number of frames written}.  `state_dict` is None for a model-based robot (config.robot.policy
    'orca' / 'social_force'), whose action comes from CrowdEngine.robot_act."""
    dev = torch.device(device)
    n = int(episodes)
    venv = CrowdVecEnv(config, n, dev, seed=config.env.seed if seed is None else seed, phase="test", nenv=1)
    eng = venv.engine
    policy = None
    if venv.robot_policy is None:
        policy = Policy(venv.observation_space.spaces, venv.action_space, base="srnn", base_kwargs=config)
        policy.load_state_dict(state_dict)
        policy = policy.to(dev)
    st = eng.get_state()                    # env k plays test case k (evaluate_batched with no warm-up episode)
    ks = torch.arange(n, dtype=torch.int64, device=dev)
    st["counters"][:, 1] = (ks % 4).to(torch.int32)
    st["counters"][:, 2] = (ks % max(1, int(eng.cfg.case_size))).to(torch.int32)
    eng.set_state(counters=st["counters"])
    obs = eng.reset().obs()
    H = config.sim.human_num
    hx = {"human_node_rnn": torch.zeros(n, 1, 128, device=dev), "human_human_edge_rnn": torch.zeros(n, H + 1, 256, device=dev)}
    masks = torch.zeros(n, 1, device=dev)
    live = np.ones(n, dtype=bool)
    written = {k: 0 for k in range(n)}
    for k in range(n):
        os.makedirs(os.path.join(out, "env%d" % k), exist_ok=True)
    if tile:
        os.makedirs(os.path.join(out, "tile"), exist_ok=True)
    limit = int(eng.cfg.timeout_step) + 2 if max_steps is None else int(max_steps)

    def write(step, ids):
        for f, k in zip(eng.render(ids.tolist(), size=size).cpu().numpy(), ids):
            write_png(os.path.join(out, "env%d" % k, "%04d.png" % step), f)
            written[int(k)] += 1
        if tile:
            write_png(os.path.join(out, "tile", "%04d.png" % step), tile_images(eng.render(size=size).cpu().numpy()))

    step = 0
    write(step, np.arange(n))                             # the reset
    while live.any() and step < limit:
        if policy is None:
            action = eng.robot_act(venv.robot_policy)
        else:
            _, action, _, hx = policy.act(obs, hx, masks, deterministic=True)
        buf = eng.step(action, auto_reset=False)           # a finished env keeps its last state: its final frame shows it
        obs, masks = buf.obs(), buf.not_done
        step += 1
        write(step, np.nonzero(live)[0])                  # every env that was still playing, the ones ending now included
        live &= ~buf.done.cpu().numpy().astype(bool)
    venv.close()
    return written


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--checkpoint", default=os.path.join(ROOT, "tests", "golden", "weights_holonomic_27776.npz"),
                    help="state_dict .pt or weights .npz")
    ap.add_argument("--episodes", type=int, default=16)
    ap.add_argument("--out", required=True)
    ap.add_argument("--size", type=int, default=256)
    ap.add_argument("--tile", action="store_true")
    ap.add_argument("--kinematics", default="holonomic", choices=["holonomic", "unicycle"])
    ap.add_argument("--humans", type=int, default=None)
    ap.add_argument("--fov", type=float, default=None, help="robot.FOV (multiples of pi)")
    ap.add_argument("--seed", type=int, default=None)
    ap.add_argument("--robot_policy", default=None, choices=["orca", "social_force"],
                    help="record a model-based robot instead of the checkpoint")
    args = ap.parse_args(argv)
    check_size(args.size)
    cfg = Config(kinematics=args.kinematics, human_num=args.humans)
    if args.fov is not None:
        cfg.robot.FOV = args.fov
    if args.robot_policy is not None:
        cfg.robot.policy = args.robot_policy
    written = record(cfg, None if args.robot_policy else load_weights(args.checkpoint), args.episodes, args.out, size=args.size, tile=args.tile,
                     seed=args.seed)
    print("wrote %d frames of %d episodes to %s (frames per episode: %s)" % (
        sum(written.values()), len(written), args.out, " ".join(str(written[k]) for k in sorted(written))))
    return 0


if __name__ == "__main__":
    sys.exit(main())
