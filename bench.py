#!/usr/bin/env python
"""bench.py -- env-steps/s of the rollout hot path (crowd step + DS-RNN forward) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c2|c1] [--precision fp32|bf16x3|bf16] [--dump-outputs DIR]
    python bench.py --impl reference ...      # the CPU arm: the oracle port on the box's host cores

One "step" = Policy.act (DS-RNN forward, deterministic) + CrowdSimDict.step for every env of the batch
(+ the device-side reset of finished episodes).  Workload (BASELINE.json):
  c3 (default, the config the metric's 1e7 env-steps/s target is quoted on): 20 humans, robot FOV 90 deg,
     16384 envs per GPU, inference-only rollout, weights of the shipped holonomic checkpoint (27776.pt);
  c2: unicycle robot, 10 humans, mixed scenarios, dt 0.1, 1024 envs;  c1: reference defaults, 5 humans, 16 envs.
Prints ONE JSON line (see the task contract): value = whole-job env-steps/s with everything resident in HBM,
e2e = the same metric through the reference-facing API with host buffers (actions, masks, rewards, dones cross
PCIe every step, as in train.py:243-292), roofline for the dominant kernel, cpu_baseline for the oracle port.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "c3": dict(human_num=20, envs_per_gpu=16384, kinematics="holonomic", over={"robot.FOV": 0.5},
               weights="holonomic_27776", label="c3: 20 humans, robot FOV 0.5*pi, 16384 envs/GPU, inference rollout"),
    "c2": dict(human_num=10, envs_per_gpu=1024, kinematics="unicycle",
               over={"env.time_step": 0.1, "reward.discomfort_penalty_factor": 1.0},
               weights="unicycle_55554", label="c2: unicycle, 10 humans, mixed scenarios, dt 0.1, 1024 envs"),
    "c1": dict(human_num=5, envs_per_gpu=16, kinematics="holonomic", over={"sim.train_val_sim": ["circle_crossing"]},
               weights="holonomic_27776", label="c1: reference defaults, 5 humans circle_crossing, 16 envs"),
    # BASELINE.json configs[4]: PPO training, 65536 envs x 20 humans in total, sharded over the GPUs (strong scaling)
    "c5": dict(human_num=20, envs_total=65536, kinematics="holonomic", over={}, weights="holonomic_27776", train=True,
               label="c5: PPO training, 65536 envs x 20 humans in total, T=30, 5 epochs x 2 minibatches, native update"),
}


# dram__bytes_read.sum + dram__bytes_write.sum per launch.  NOT sampled in this run: constants copied from ONE earlier
# `ncu --set full` capture of the same kernels at the default sizes (the file named in `traffic_source`); only reported for that
# workload / batch, null otherwise
# edge kernel: the resident-image instantiation the graph rollout runs (reads the 352 MB split-bf16 image, writes the fp32 state
# and the next image: 358 MB + 658 MB, profiles/r2_ncu_edge_image.txt); step kernel: profiles/r2_ncu_final_other_kernels.txt
NCU_TRAFFIC_BYTES = {("c3", 16384): {"edge_gru_tc_kernel": 358.48e6 + 657.58e6, "crowd_step_kernel": 18.12e6 + 3.58e6}}
NCU_TRAFFIC_SOURCE = ("profiles/r2_ncu_edge_image.txt / profiles/r2_ncu_final_other_kernels.txt (one ncu --set full capture each, "
                      "end of round 2; not re-measured by this run)")


def reference_python_baseline(workload):
    """The BASELINE.md section-3 CPU path -- the reference's own Python env under its own ShmemVecEnv + Policy.act, rvo2
    restated -- cannot travel to the GPU box (it is Python from /root/reference); it is timed in the build container by
    oracle/bench_reference_python.py and its committed result is quoted here, labelled as such."""
    path = os.path.join(ROOT, "profiles", "r2_reference_python_cpu.json")
    if not os.path.exists(path):
        return None
    try:
        with open(path) as f:
            doc = json.load(f)
    except ValueError:
        return None
    for r in doc.get("results", []):
        if r.get("workload") == workload and r.get("did_not_finish"):
            return {"value": None, "unit": "env-steps/s", "cores": r["processes"], "kind": "reference-python",
                    "sample": "did not finish: " + r["note"], "measured_on": doc.get("where"),
                    "source": "profiles/r2_reference_python_cpu.json (oracle/bench_reference_python.py)"}
        if r.get("workload") == workload:
            return {"value": r["env_steps_per_s"], "unit": "env-steps/s", "cores": r["processes"], "kind": "reference-python",
                    "sample": "%d lock-step steps of %d reference CrowdSimDict processes under ShmemVecEnv + reference Policy.act in %.0f s%s"
                              % (r["timed_steps"], r["processes"], r["elapsed_s"], " (wall-capped)" if r.get("wall_capped") else ""),
                    "measured_on": doc.get("where"), "source": "profiles/r2_reference_python_cpu.json (oracle/bench_reference_python.py)"}
    return None


def step_bytes(H):          # SURVEY 8(d): algorithmic HBM bytes of the step kernel per env-step
    return 96 * H + 188


def forward_flops(H):       # SURVEY 8(d): algorithmic FLOPs of the DS-RNN forward per env-step
    return 2 * ((H + 1) * 262272 + 320 * H + 426965)


def edge_stage_flops(H):    # encoder + GRU(64->256) per edge row: 2*(2*64 + 768*64 + 768*256) FLOP
    return 2 * (H + 1) * (2 * 64 + 768 * 64 + 768 * 256)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops"], bf16_tflops_sustained=p["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def make_config(wl):
    from crowdnav_dsrnn_b200 import Config

    cfg = Config(kinematics=wl["kinematics"], human_num=wl["human_num"])
    for k, v in wl["over"].items():
        sec, _, attr = k.partition(".")
        setattr(getattr(cfg, sec), attr, v)
    return cfg


def load_weights(name):
    path = os.path.join(ROOT, "tests", "golden", "weights_%s.npz" % name)
    w = np.load(path)
    return {k: w[k] for k in w.files}


DUMP_BYTES = 64 * 10 ** 6      # --dump-outputs writes at most this much in all


def dump_outputs(path, arrays, n_envs=None):
    """--dump-outputs: write each array (torch tensor or numpy) as <path>/<name>.npy, float64 as float64 and everything else as
    float32.  If they would exceed DUMP_BYTES together, every array whose first axis is the env axis (length n_envs) keeps
    the same fixed, seeded sample of envs, so that two runs with the same arguments write the same rows."""
    out = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        out[name] = a if a.dtype == np.float64 else a.astype(np.float32)
    per_env = lambda a: n_envs is not None and a.ndim > 0 and a.shape[0] == n_envs
    env_bytes = sum(a.nbytes for a in out.values() if per_env(a))
    budget = DUMP_BYTES - 128 * len(out) - sum(a.nbytes for a in out.values() if not per_env(a))     # 128 B: .npy header
    if env_bytes > budget:
        keep = max(1, int(budget // (env_bytes // n_envs)))
        rows = np.sort(np.random.default_rng(0).choice(n_envs, keep, replace=False))
        out = {k: a[rows] if per_env(a) else a for k, a in out.items()}
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:  # noqa: BLE001 - nvidia-smi missing: report no clocks rather than fail the bench
            pass

    def begin(self, timeout=3.0):
        """Start sampling and return once nvidia-smi delivers (its start-up can take longer than a short timed region); the
        samples taken from here on are the ones reported."""
        self.start()
        t_end = time.time() + timeout
        while not self.rows and time.time() < t_end and self.is_alive():
            time.sleep(0.02)
        self.first = len(self.rows)

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        first = getattr(self, "first", 0)
        rows = self.rows[first:] if len(self.rows) > first else self.rows      # a region shorter than one period: what there is
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_port_rate(wl, n_envs, steps, warmup, threads):
    """env-steps/s of the ORACLE PORT on the host cores: C crowd step (pthreads over envs) + torch fp32 forward."""
    import torch

    from crowdnav_dsrnn_b200 import abi
    from oracle import crowd_oracle, dsrnn_oracle

    torch.set_num_threads(threads)
    cfg_obj = make_config(wl)
    cfg = abi.flatten_config(cfg_obj, n_envs, phase="train")
    H = cfg.human_num
    sd = {k: torch.from_numpy(v) for k, v in load_weights(wl["weights"]).items()}
    st = crowd_oracle.OracleState(n_envs, H)
    out = crowd_oracle.reset(cfg, st, n_threads=threads)
    hn, he = torch.zeros(n_envs, 1, 128), torch.zeros(n_envs, H + 1, 256)
    masks = torch.ones(n_envs, 1)
    t0 = None
    with torch.no_grad():
        for it in range(warmup + steps):
            if it == warmup:
                t0 = time.perf_counter()
            r = dsrnn_oracle.forward(sd, torch.from_numpy(out.robot_node), torch.from_numpy(out.temporal_edges),
                                     torch.from_numpy(out.spatial_edges), hn, he, masks)
            hn, he = r["h_node"], r["h_edge"]
            out = crowd_oracle.step(cfg, st, r["action_mean"].numpy(), auto_reset=True, n_threads=threads)
            masks = torch.from_numpy(1.0 - out.done.astype(np.float32)).unsqueeze(1)
    dt = time.perf_counter() - t0
    return n_envs * steps / dt, dt


def run_reference_arm(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n_cpu = max(64, min(wl["envs_per_gpu"], 32 * threads))
    rate, dt = cpu_port_rate(wl, n_cpu, args.steps, args.warmup, threads)
    line = {
        "impl": "reference", "metric": "env_steps_per_sec_incl_dsrnn_forward", "value": rate, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["label"], "human_num": wl["human_num"], "envs_per_step": n_cpu},
        "cpu_baseline": {"value": rate, "unit": "env-steps/s", "cores": threads, "kind": "port",
                         "sample": "%d envs x %d steps of the same workload (oracle C crowd step on %d pthreads + torch fp32 "
                                   "DS-RNN forward on %d threads)" % (n_cpu, args.steps, threads, threads)},
        "e2e": {"value": rate, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------ GPU arm
def run_ours(args, wl):
    import torch
    import torch.distributed as dist

    from crowdnav_dsrnn_b200 import _lib
    from crowdnav_dsrnn_b200.envs import CrowdVecEnv
    from crowdnav_dsrnn_b200.model import Policy
    from crowdnav_dsrnn_b200.spaces import crowd_spaces

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    N = args.envs_per_gpu or wl["envs_per_gpu"]
    H = wl["human_num"]
    cfg_obj = make_config(wl)
    cfg_obj.training.num_processes = N * world
    # envs shard by global id: rank r owns [r*N, (r+1)*N); RNG is keyed by global env id, no data-path collective
    venv = CrowdVecEnv(cfg_obj, N, dev, seed=0, phase="train", env_id_offset=rank * N, nenv=N * world)
    obs_space, act_space = crowd_spaces(H)
    policy = Policy(obs_space.spaces, act_space, base="srnn", base_kwargs=cfg_obj)
    policy.load_state_dict({k: torch.from_numpy(v) for k, v in load_weights(wl["weights"]).items()})
    policy = policy.to(dev)
    policy.precision = args.precision
    eng = venv.engine

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident rollout (value)
    last = {}       # what the last step of the last rollout() call returned (--dump-outputs of the eager loop)

    def rollout(steps, obs, hx, masks):
        for _ in range(steps):
            value, action, _, hx = policy.act(obs, hx, masks, deterministic=True)
            obs, reward, done, _ = venv.step_device(action)
            masks = (1.0 - done.to(torch.float32)).unsqueeze(1)
        if steps:
            last.update(obs, reward=reward, done=done, value=value, action=action, **hx)
        return obs, hx, masks

    obs = venv.reset()
    hx = {"human_node_rnn": torch.zeros(N, 1, 128, device=dev), "human_human_edge_rnn": torch.zeros(N, H + 1, 256, device=dev)}
    masks = torch.zeros(N, 1, device=dev)
    obs, hx, masks = rollout(args.prime, obs, hx, masks)      # de-phase the episodes (untimed)
    obs, hx, masks = rollout(args.warmup, obs, hx, masks)     # warm-up (untimed)
    import ctypes as C
    from crowdnav_dsrnn_b200.rollout import GraphedRollout

    sampler = ClockSampler(local)
    if args.no_graph:
        launches0 = eng.launches + policy.gpu_launches
        if rank == 0:
            sampler.begin()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        obs, hx, masks = rollout(args.steps, obs, hx, masks)
        ev1.record()
        barrier()
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, last, N)
        launches = eng.launches + policy.gpu_launches - launches0
    else:
        # the timed loop replays the rollout step (crowd step incl. swap-in of spare episodes -> forward on the new observation,
        # with the refill of the consumed spares forked beside the attention kernel) as a CUDA graph: the kernels and the
        # data flow are those of the eager loop (tests/test_gpu_rollout_graph.py), only the launch path differs
        roll = GraphedRollout(policy, venv, obs, hx, masks)
        for _ in range(max(3, args.warmup)):
            roll.step()
        if rank == 0:
            sampler.begin()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(args.steps):
            buf = roll.step()
        ev1.record()
        barrier()
        if args.dump_outputs and rank == 0:
            # the last replay stepped the envs into `buf`, then ran the forward on that observation: it wrote action and value to
            # sets[parity] and the hidden state it produced to sets[parity ^ 1] (GraphedRollout._one_step)
            fw, h = roll.sets[roll.parity], roll.sets[roll.parity ^ 1]
            dump_outputs(args.dump_outputs, dict(buf.obs(), reward=buf.reward, done=buf.done, value=fw["value"], action=fw["mean"],
                                                 human_node_rnn=h["h_node"], human_human_edge_rnn=h["h_edge"]), N)
        launches = args.steps * roll.launches_per_step
        # per-kernel durations for the roofline: CUDA events recorded by the library around the dominant kernels on the
        # launching stream, over a short EAGER continuation of the same step schedule (events cannot be read back from a
        # graph replay; the eager launches keep the refill where the graph has it, beside the attention kernel)
        lib.cn_dsrnn_enable_timing(policy._handle, 1)
        lib.cn_env_enable_timing(eng.handle, 1)
        for _ in range(min(args.steps, 50)):
            buf = roll.step_eager()
        torch.cuda.synchronize()
        obs = buf.obs()
        hx, masks = roll.hidden()
        roll.close()
        hx = {k: v.clone() for k, v in hx.items()}
        masks = masks.clone()
    clocks = sampler.stop() if rank == 0 else None
    ms = ev0.elapsed_time(ev1)
    if args.no_graph:
        lib.cn_dsrnn_enable_timing(policy._handle, 1)
        lib.cn_env_enable_timing(eng.handle, 1)
        obs, hx, masks = rollout(min(args.steps, 50), obs, hx, masks)
        torch.cuda.synchronize()
    edge_ms, n_fw, step_ms, n_st = C.c_float(), C.c_int(), C.c_float(), C.c_int()
    lib.cn_dsrnn_time_ms(policy._handle, C.byref(edge_ms), C.byref(n_fw))
    lib.cn_env_time_ms(eng.handle, C.byref(step_ms), C.byref(n_st))
    lib.cn_dsrnn_enable_timing(policy._handle, 0)
    lib.cn_env_enable_timing(eng.handle, 0)
    resets = float(eng.get_state()["counters"][:, 1].float().mean().item())

    # ---------------- end-to-end through the reference-facing API with HOST buffers (e2e)
    e2e_steps = max(3, min(args.steps, args.e2e_steps))
    pin_action = torch.empty(N, 2, dtype=torch.float32).pin_memory()
    pin_masks = torch.empty(N, 1, dtype=torch.float32).pin_memory()

    def e2e_rollout(steps, obs, hx, masks):
        for _ in range(steps):
            _, action, _, hx = policy.act(obs, hx, masks, deterministic=True)
            pin_action.copy_(action, non_blocking=True)            # action.cpu() of VecPyTorch.step_async (envs.py:224-229)
            # the env API is driven from the pinned HOST buffer; the H2D copy is ordered after the D2H copy on the stream
            obs, reward, done, infos = venv.step(pin_action.to(dev, non_blocking=True))    # reward CPU tensor, done numpy
            pin_masks.copy_(torch.from_numpy(1.0 - done.astype(np.float32)).unsqueeze(1))  # train.py:279
            masks = pin_masks.to(dev, non_blocking=True)
        return obs, hx, masks

    obs, hx, masks = e2e_rollout(3, obs, hx, masks)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    obs, hx, masks = e2e_rollout(e2e_steps, obs, hx, masks)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    h2d = N * 2 * 4 + N * 4                 # actions + masks
    d2h = N * 2 * 4 + N * 4 + N             # actions + reward + done

    if world > 1:
        t = torch.tensor([ms, e2e_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = float(t[0]), float(t[1])
        lt = torch.tensor([float(launches)], device=dev)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
        launches = int(lt[0])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    value = N * world * args.steps / (ms * 1e-3)
    e2e_value = N * world * e2e_steps / (e2e_ms * 1e-3)
    edge_avg_ms = edge_ms.value / max(1, n_fw.value)
    step_avg_ms = step_ms.value / max(1, n_st.value)
    roof_step = {"bound": "hbm", "achieved": N * step_bytes(H) / (step_avg_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"],
                 "unit": "GB/s", "kernel": "crowd_step_kernel", "ms_per_launch": step_avg_ms, "traffic": None,
                 "algorithmic_bytes_per_env_step": step_bytes(H), "share_of_step": step_avg_ms / (ms / args.steps)}
    roof_step["frac"] = roof_step["achieved"] / roof_step["peak"]
    roof_step["note"] = ("nominally HBM-bound (SURVEY 8(d)); measured: instruction-issue bound at every H (H=1..20: 0.015-0.026 of "
                         "the HBM peak, profiles/r2_k1_sweep.txt; ncu at H=20: the ORCA solves keep 83 % of the issue slots busy, dram 0.4 %)")
    traffic = NCU_TRAFFIC_BYTES.get((args.workload, N), {})
    roof_step["traffic"] = traffic.get("crowd_step_kernel")
    roof_step["traffic_source"] = NCU_TRAFFIC_SOURCE if traffic else None
    edge_kernel = "edge_gru_simt_kernel" if args.precision == "fp32" else "edge_gru_tc_kernel"
    passes = 3 if args.precision == "bf16x3" else 1
    roof_edge = {"bound": "tensor", "achieved": N * edge_stage_flops(H) / (edge_avg_ms * 1e-3) / 1e12,
                 "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s", "kernel": edge_kernel,
                 "ms_per_launch": edge_avg_ms, "traffic": None, "algorithmic_flops_per_env_step": edge_stage_flops(H),
                 "tensor_passes": passes, "share_of_step": edge_avg_ms / (ms / args.steps)}
    roof_edge["frac"] = roof_edge["achieved"] / roof_edge["peak"]
    # `frac` counts ALGORITHMIC FLOPs (one product per weight); the kernel issues `tensor_passes` bf16 MMAs per product to reach
    # fp32-level accuracy, so the tensor pipe itself runs at frac_issued of the measured sustained bf16 peak
    roof_edge["frac_issued"] = passes * roof_edge["frac"]
    roof_edge["traffic"] = traffic.get(edge_kernel)
    roof_edge["traffic_source"] = NCU_TRAFFIC_SOURCE if traffic.get(edge_kernel) else None
    dominant = roof_edge if edge_avg_ms >= step_avg_ms else roof_step
    other = roof_step if dominant is roof_edge else roof_edge

    cpu = None
    if not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        n_cpu = max(64, min(N, 32 * threads))
        _, probe = cpu_port_rate(wl, n_cpu, 2, 1, threads)                 # size the sample for ~args.cpu_seconds of CPU work
        cpu_steps = int(max(3, min(2000, args.cpu_seconds / max(probe / 2, 1e-4))))
        rate, dt = cpu_port_rate(wl, n_cpu, cpu_steps, 2, threads)
        cpu = {"value": rate, "unit": "env-steps/s", "cores": threads, "kind": "port",
               "sample": "%d envs x %d steps of the same workload in %.1f s (oracle C crowd step on %d pthreads + torch fp32 "
                         "DS-RNN forward)" % (n_cpu, cpu_steps, dt, threads)}

    line = {
        "metric": "env_steps_per_sec_incl_dsrnn_forward", "value": value, "unit": "env-steps/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": {"fp32": "f32", "bf16x3": "bf16x3 (3-pass split bf16, fp32 accumulate)", "bf16": "bf16", "fp16": "fp16 (fp32 accumulate)"}[args.precision],
        "data": "synthetic scenarios (device reset, counter-based RNG); weights of the shipped checkpoint %s" % wl["weights"],
        "config": {"workload": wl["label"] if N == wl["envs_per_gpu"] else wl["label"] + " (overridden: %d envs/GPU)" % N,
                   "human_num": H, "envs_per_gpu": N, "global_envs": N * world,
                   "parallelism": "env-sharded x%d, no data-path collective" % world, "precision": args.precision,
                   "l2": "inputs larger than L2 (hidden state %.0f MB + env state %.0f MB per step vs 126 MB L2)" % (
                       N * (H + 1) * 256 * 4 * 2 / 1e6, N * step_bytes(H) / 1e6),
                   "launch": "eager" if args.no_graph else "cuda-graph replay of the rollout step", "prime_steps": args.prime, "resets_per_env_total": resets, "peaks": peaks["source"]},
        "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps},
        "gpu_launches": launches, "clocks": clocks, "roofline": dominant, "roofline_other": other, "cpu_baseline": cpu,
        "cpu_baseline_reference_python": reference_python_baseline(args.workload),
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ training workload (c5)
def run_train(args, wl):
    """One "step" = one PPO update cycle: T = ppo.num_steps rollout steps of every env (CUDA crowd step + DS-RNN forward,
    device resident), bootstrap value, returns, and the PPO update (5 epochs x 2 minibatches) on the library's native
    kernels, gradients averaged over the ranks with NCCL.  value = env-steps/s of the whole job."""
    import ctypes as C

    import torch
    import torch.distributed as dist

    from crowdnav_dsrnn_b200 import _lib, native
    from crowdnav_dsrnn_b200.envs import CrowdVecEnv
    from crowdnav_dsrnn_b200.model import Policy
    from crowdnav_dsrnn_b200.ppo import PPO
    from crowdnav_dsrnn_b200.spaces import crowd_spaces
    from crowdnav_dsrnn_b200.storage import SRNNRolloutStorage

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (there is no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    total = args.envs_total or wl["envs_total"]
    N = total // world
    H = wl["human_num"]
    cfg = make_config(wl)
    cfg.training.num_processes = N
    T = int(cfg.ppo.num_steps)
    torch.manual_seed(1234 + rank)
    venv = CrowdVecEnv(cfg, N, dev, seed=0, phase="train", env_id_offset=rank * N, nenv=N * world)
    obs_space, act_space = crowd_spaces(H)
    policy = Policy(obs_space.spaces, act_space, base="srnn", base_kwargs=cfg)
    policy.load_state_dict({k: torch.from_numpy(v) for k, v in load_weights(wl["weights"]).items()})
    policy = policy.to(dev)
    rollouts = SRNNRolloutStorage(T, N, obs_space.spaces, act_space, 128, 256, "GRU", device=dev, keep_hidden_history=False)
    per_pass = min(args.envs_per_pass, N // cfg.ppo.num_mini_batch)
    agent = PPO(policy, cfg.ppo.clip_param, cfg.ppo.epoch, cfg.ppo.num_mini_batch, cfg.ppo.value_loss_coef, cfg.ppo.entropy_coef,
                lr=cfg.training.lr, eps=cfg.training.eps, max_grad_norm=cfg.training.max_grad_norm, max_envs_per_pass=per_pass,
                native=True)
    obs = venv.reset()
    for k in rollouts.obs:
        rollouts.obs[k][0].copy_(obs[k])
    timing = {"rollout": [], "update": []}

    def cycle(record=False):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)] if record else None
        if record:
            ev[0].record()
        for step in range(T):
            value, action, log_prob, hx = policy.act(rollouts.obs_at(step), dict(rollouts.hidden_at(step)), rollouts.masks[step])
            o, reward, done, buf = venv.step_device(action)
            rollouts.insert(o, hx, action, log_prob, value, reward, buf.not_done, None)
        next_value = policy.get_value(rollouts.obs_at(-1), dict(rollouts.hidden_at(-1)), rollouts.masks[-1]).detach()
        rollouts.compute_returns(next_value, cfg.ppo.use_gae, cfg.reward.gamma, cfg.ppo.gae_lambda, cfg.training.use_proper_time_limits)
        if record:
            ev[1].record()
        losses = agent.update(rollouts, sync=False)
        rollouts.after_update()
        if record:
            ev[2].record()
            timing["pending"] = ev
        return losses

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        cycle()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.begin()
    launches0 = venv.engine.launches + policy.gpu_launches + native.COUNTERS["gemm_launches"] + native.COUNTERS["kernel_launches"]
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        losses = cycle()
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        # the last update cycle returned the averaged losses (value, action, entropy) and left the updated weights in the policy
        dump_outputs(args.dump_outputs, dict(losses=losses, **{"param." + k: v for k, v in policy.state_dict().items()}))
    ms = e0.elapsed_time(e1)
    launches = venv.engine.launches + policy.gpu_launches + native.COUNTERS["gemm_launches"] + native.COUNTERS["kernel_launches"] - launches0
    clocks = sampler.stop() if rank == 0 else None
    # one more cycle with the library's GEMM timing on: the roofline of the dominant kernel and the rollout / update split
    lib.cn_gemm_enable_timing(1)
    cycle(record=True)
    torch.cuda.synchronize()
    gemm_ms, gemm_n, gemm_flops = C.c_float(), C.c_int(), C.c_double()
    lib.cn_gemm_time_ms(C.byref(gemm_ms), C.byref(gemm_n), C.byref(gemm_flops))
    lib.cn_gemm_enable_timing(0)
    ev = timing["pending"]
    rollout_ms, update_ms = ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])
    # end to end through the public training API (train.train): same loop plus its per-update host reads (episode
    # statistics and losses cross PCIe once per update)
    from crowdnav_dsrnn_b200.train import train as train_api

    cfg.training.num_env_steps = 10 ** 12
    cfg.training.log_interval = 1
    cfg.training.save_interval = 10 ** 9
    e2e_updates = max(1, min(args.steps, 2))
    barrier()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    # train() writes its run artefacts (configs, log, progress.csv, checkpoint) like a user's run does, but not into the tree
    with tempfile.TemporaryDirectory() as run_dir:
        train_api(cfg, dev, num_updates=1, output_dir=run_dir, actor_critic=policy, log=None, max_envs_per_pass=per_pass, native_update=True)
        barrier()
        t0.record()
        train_api(cfg, dev, num_updates=e2e_updates, output_dir=run_dir, actor_critic=policy, log=None, max_envs_per_pass=per_pass, native_update=True)
        t1.record()
        barrier()
    e2e_ms = t0.elapsed_time(t1)
    if world > 1:
        t = torch.tensor([ms, e2e_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms = float(t[0]), float(t[1])
        lt = torch.tensor([float(launches)], device=dev)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
        launches = int(lt[0])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = measured_peaks()
    value = N * world * T * args.steps / (ms * 1e-3)
    e2e_value = N * world * T * e2e_updates / (e2e_ms * 1e-3)
    roof = {"bound": "tensor", "kernel": "gemm_bf16x3_kernel", "achieved": gemm_flops.value / (gemm_ms.value * 1e-3) / 1e12,
            "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s", "ms_per_launch": gemm_ms.value / max(1, gemm_n.value),
            "launches_per_step": gemm_n.value, "ms_per_step": gemm_ms.value, "traffic": None, "tensor_passes": 3,
            "algorithmic_flops_per_step": gemm_flops.value, "share_of_step": gemm_ms.value / (rollout_ms + update_ms),
            "note": "all cn_gemm_bf16x3 launches of one update cycle (recurrent products, weight gradients, linears); algorithmic "
                    "FLOPs = 2 m n k, three bf16 tensor passes are issued per product"}
    roof["frac"] = roof["achieved"] / roof["peak"]
    line = {
        "metric": "env_steps_per_sec_ppo_training", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "bf16x3 (3-pass split bf16, fp32 accumulate) for every contraction; fp32 elsewhere",
        "data": "synthetic scenarios (device reset, counter-based RNG); initial weights of the shipped checkpoint %s" % wl["weights"],
        "config": {"workload": wl["label"], "human_num": H, "global_envs": N * world, "envs_per_gpu": N, "num_steps": T,
                   "ppo_epoch": cfg.ppo.epoch, "num_mini_batch": cfg.ppo.num_mini_batch, "envs_per_pass": per_pass,
                   "parallelism": "env-sharded x%d, NCCL all-reduce of the gradients (2 buckets, the first overlapped with backward)" % world,
                   "l2": "inputs larger than L2 (activations of one pass: %.1f GB)" % (per_pass * (H + 1) * T * 11.3e3 / 1e9),
                   "rollout_ms": rollout_ms, "update_ms": update_ms, "peaks": peaks["source"]},
        "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 5 * 8 + 3 * 4,
                "steps": e2e_updates, "ms_per_step": e2e_ms / e2e_updates,
                "note": "crowdnav_dsrnn_b200.train.train(): the same cycle through the public API, with its per-update host reads"},
        "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cpu_baseline": None,
    }
    emit(line)
    if world > 1:
        dist.destroy_process_group()


_RESULT_FD = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner to stdout when the
    communicator is created lazily), so everything the process writes to fd 1 during the run goes to stderr and only the
    result line is written to the real stdout."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    text = json.dumps(line) + "\n"
    if _RESULT_FD is None:
        sys.stdout.write(text)
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, text.encode())


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 200; 3 update cycles for c5)")
    ap.add_argument("--warmup", type=int, default=None, help="untimed steps (default 20; 3 for c5)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="bf16x3", choices=["fp32", "bf16x3", "bf16", "fp16"])
    ap.add_argument("--envs-per-gpu", type=int, default=0)
    ap.add_argument("--prime", type=int, default=150, help="untimed steps before warm-up so episodes are de-phased")
    ap.add_argument("--e2e-steps", type=int, default=50)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU work of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time the eager loop instead of the CUDA-graph replay")
    ap.add_argument("--envs-total", type=int, default=0, help="c5: total envs over all GPUs (default 65536)")
    ap.add_argument("--envs-per-pass", type=int, default=4096, help="c5: env trajectories per forward/backward pass of the update")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32 / float64, at most "
                         "64 MB: a fixed sample of envs when larger; rank 0's envs): c1-c3 the observation, reward, done, value, "
                         "action and hidden state of the step, c5 the losses and the updated weights")
    args = ap.parse_args()
    wl = WORKLOADS[args.workload]
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this project's GPU path; --impl reference has none")
    if args.steps is None:
        args.steps = 3 if wl.get("train") else 200
    if args.warmup is None:
        args.warmup = 3 if wl.get("train") else 20
    if args.warmup < 3:
        args.warmup = 3
    if wl.get("train"):
        if args.impl == "reference":
            raise SystemExit("--impl reference times the rollout workloads (c1/c2/c3); the training workload has no CPU arm")
        run_train(args, wl)
    elif args.impl == "reference":
        run_reference_arm(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
