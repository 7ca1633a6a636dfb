"""Cost of a training-state file (train_state.py, `training.save_train_state`) at the c5 shape: 65536 envs x 20 humans,
T = 30, on one GPU.  Builds what `train()` holds between updates (envs after a reset, the policy, Adam with its moments,
the rollout storage with slot 0 filled) and times, with a host clock around work that ends in a device synchronise:

* one save: `train_state.save` (device -> host copies, torch.save, fsync, rename) of the shared file and rank 0's shard;
* one load: `train_state.load` (both files) + `train_state.restore` into a second set of objects.

Files go to a temporary directory (`--dir` to choose its parent), which is removed at the end.

    python tools/bench_train_state.py --envs 65536 --humans 20 --reps 3 > train_state.txt
"""
import argparse
import os
import shutil
import subprocess
import sys
import tempfile
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from crowdnav_dsrnn_b200 import Config, train_state  # noqa: E402
from crowdnav_dsrnn_b200.envs import CrowdVecEnv  # noqa: E402
from crowdnav_dsrnn_b200.model import Policy  # noqa: E402
from crowdnav_dsrnn_b200.storage import SRNNRolloutStorage  # noqa: E402


def build(cfg, n, dev):
    envs = CrowdVecEnv(cfg, n, dev, seed=cfg.env.seed, phase="train")
    policy = Policy(envs.observation_space.spaces, envs.action_space, base="srnn", base_kwargs=cfg).to(dev)
    opt = torch.optim.Adam(policy.parameters(), lr=cfg.training.lr, eps=cfg.training.eps)
    for p in policy.parameters():
        p.grad = torch.randn_like(p) * 1e-3
    opt.step()                                        # Adam's moments exist, as after the first update
    rollouts = SRNNRolloutStorage(cfg.ppo.num_steps, n, envs.observation_space.spaces, envs.action_space, 128, 256,
                                  device=dev, keep_hidden_history=False)
    obs = envs.reset()
    for k in rollouts.obs:
        rollouts.obs[k][0].copy_(obs[k])
    for v in rollouts.recurrent_hidden_states.values():
        v[0].normal_()
    return envs, policy, opt, rollouts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--humans", type=int, default=20)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--dir", default=None, help="parent of the temporary directory the files are written to")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    print("card: %s" % card)
    cfg = Config(human_num=args.humans)
    cfg.training.num_processes = args.envs
    cfg.ppo.num_steps = args.steps
    torch.manual_seed(0)
    keys = train_state.run_keys(cfg, args.envs, 1, False)
    src = build(cfg, args.envs, dev)
    dst = build(cfg, args.envs, dev)
    hidden = sum(v[0].numel() * 4 for v in src[3].recurrent_hidden_states.values())
    print("%d envs x %d humans, T = %d: hidden-state slot 0 %.3f GB (from shapes)" % (args.envs, args.humans, args.steps, hidden / 1e9))
    root = tempfile.mkdtemp(prefix="train_state_", dir=args.dir)
    try:
        for rep in range(args.reps):
            ckpt = os.path.join(root, "checkpoints")
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            path = train_state.save(ckpt, rep, (rep + 1) * args.envs * args.steps, keys, src[1], src[2], src[0].engine, src[3], dev)
            t1 = time.perf_counter()
            kind, shared, shard = train_state.load(path)
            train_state.restore(shared, shard, dst[1], dst[2], dst[0].engine, dst[3], dev)
            torch.cuda.synchronize(dev)
            t2 = time.perf_counter()
            sizes = [os.path.getsize(path), os.path.getsize(train_state.rank_path(path, 0))]
            same = all(torch.equal(src[3].recurrent_hidden_states[k][0], dst[3].recurrent_hidden_states[k][0])
                       for k in src[3].recurrent_hidden_states)
            print("rep %d: shared file %.1f MB, rank-0 shard %.1f MB; save %.2f s, load + restore %.2f s; hidden state restored "
                  "bit for bit: %s" % (rep, sizes[0] / 1e6, sizes[1] / 1e6, t1 - t0, t2 - t1, same))
            del shared, shard
            for name in os.listdir(ckpt):
                os.remove(os.path.join(ckpt, name))
    finally:
        shutil.rmtree(root, ignore_errors=True)
        for envs in (src[0], dst[0]):
            envs.close()


if __name__ == "__main__":
    main()
