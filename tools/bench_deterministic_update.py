"""Cost of the bit-reproducible native update (PPO(deterministic=True), training.cuda_deterministic): one native forward +
backward pass of `Policy.evaluate_actions` over a [T, n] rollout chunk (the pass the c5 update runs 10 times per cycle) in
the default mode (split-K atomics) and in ordered mode, alternating in one process, timed with CUDA events.  Also reports
the extra partial-product bytes of one pass, taken from the workspace queries of every ordered launch (shapes only).

    python tools/bench_deterministic_update.py --envs 4096 --humans 20 --steps 30 --reps 30 > deterministic_update.txt
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from crowdnav_dsrnn_b200 import Config, _lib, native  # noqa: E402
from crowdnav_dsrnn_b200.model import Policy  # noqa: E402
from crowdnav_dsrnn_b200.spaces import crowd_spaces  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--humans", type=int, default=20)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--reps", type=int, default=30, help="timed passes per mode (alternating)")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    n, H, T = args.envs, args.humans, args.steps
    obs_space, act_space = crowd_spaces(H)
    torch.manual_seed(0)
    policy = Policy(obs_space.spaces, act_space, base="srnn", base_kwargs=Config(human_num=H)).to(dev)
    policy.sequence_impl = "native"
    g = torch.Generator(device=dev).manual_seed(0)
    obs = {"robot_node": torch.randn(T * n, 1, 7, device=dev, generator=g),
           "temporal_edges": torch.randn(T * n, 1, 2, device=dev, generator=g),
           "spatial_edges": torch.randn(T * n, H, 2, device=dev, generator=g) * 3}
    masks = (torch.rand(T * n, 1, device=dev, generator=g) > 0.03).float()
    action = torch.randn(T * n, 2, device=dev, generator=g)
    hx0 = {"human_node_rnn": torch.randn(n, 1, 128, device=dev, generator=g) * 0.3,
           "human_human_edge_rnn": torch.randn(n, H + 1, 256, device=dev, generator=g) * 0.3}

    def one_pass():
        policy.zero_grad(set_to_none=True)
        value, logp, ent, _ = policy.evaluate_actions(obs, {k: v.clone() for k, v in hx0.items()}, masks, action)
        (value.mean() + logp.mean() - 0.01 * ent).backward()

    # partial-product bytes and reduction launches of one ordered pass, from the workspace queries (no timing involved)
    extra = {"gemm_bytes": 0, "gemm_reductions": 0, "encoder_bytes": 0, "encoder_reductions": 0}
    gemm, enc = native.gemm, native.encoder_grad

    def gemm_count(problems):
        nbytes, _ = native.ordered_workspace(problems)
        extra["gemm_bytes"] += nbytes
        extra["gemm_reductions"] += 1 if nbytes else 0
        return gemm(problems)

    def enc_count(de, e_hi, ld_e, x, dw, db):
        extra["encoder_bytes"] += _lib.load().cn_encoder_grad_ordered_workspace_bytes(x.shape[0])
        extra["encoder_reductions"] += 1
        return enc(de, e_hi, ld_e, x, dw, db)

    native.gemm, native.encoder_grad = gemm_count, enc_count
    native.DETERMINISTIC = True
    one_pass()
    native.DETERMINISTIC = False
    native.gemm, native.encoder_grad = gemm, enc

    for mode in (False, True, False, True):          # warm-up of both modes (allocator pools, module loads)
        native.DETERMINISTIC = mode
        one_pass()
    torch.cuda.synchronize()
    times = {False: [], True: []}
    for _ in range(args.reps):
        for mode in (False, True):
            native.DETERMINISTIC = mode
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            one_pass()
            e1.record()
            torch.cuda.synchronize()
            times[mode].append(e0.elapsed_time(e1))
    native.DETERMINISTIC = False
    med = {m: sorted(t)[len(t) // 2] for m, t in times.items()}
    mean = {m: sum(t) / len(t) for m, t in times.items()}
    print("card: %s" % card)
    print("native forward + backward pass of %d envs x %d humans x T = %d, %d alternating passes per mode (CUDA events)" % (
        n, H, T, args.reps))
    for m, name in ((False, "default (split-K atomics)"), (True, "ordered (deterministic)")):
        t = times[m]
        print("  %-26s median %.3f ms  mean %.3f ms  min %.3f ms  max %.3f ms" % (name, med[m], mean[m], min(t), max(t)))
    print("  overhead of ordered mode: %+.2f %% (median), %+.2f %% (mean)" % (100 * (med[True] / med[False] - 1),
                                                                            100 * (mean[True] / mean[False] - 1)))
    print("  extra partial-product bytes per pass: %.1f MB in %d split-K GEMM launches (+%d reduction launches), "
          "%.2f MB in %d encoder-gradient calls (+%d reduction launches)" % (
              extra["gemm_bytes"] / 1e6, extra["gemm_reductions"], extra["gemm_reductions"], extra["encoder_bytes"] / 1e6,
              extra["encoder_reductions"], extra["encoder_reductions"]))


if __name__ == "__main__":
    main()
