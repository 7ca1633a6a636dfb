"""TEST INFRASTRUCTURE -- host mirror of the launch shapes the env launchers pick, of the env state blob's layout, and
the tiling of a small sampled state to a benchmark-sized batch.

  * step_shape: cn_launch_crowd_step (csrc/crowd_step.cu): lane-group width G, envs per CTA E (the production rule, the
    small-batch rule below E * 4 * SMs envs, the CN_STEP_ENVS_PER_CTA knob and its clamp to the 48 KB shared-memory
    default), grid and the size of the last CTA, for the group form (also the two-launch form) and the thread-per-human
    form (CN_STEP_SEQ=1);
  * reset_grid: cn_launch_crowd_reset (csrc/crowd_reset.cu): one CTA per env, except the synchronous fall-back (at most
    592 CTAs) and the refill of the listed envs (at most 1184 CTAs), which stride over their envs;
  * robot_act_shape: cn_launch_robot_act: one G-lane group per env, 256 / G envs per CTA;
  * state_layout: cn_carve (csrc/env_common.cuh), the byte offset of every array inside the caller's state buffer;
  * tile_state: a state_sampler.sample() batch repeated to N envs, each tile with its own counters.

The GPU tests take the SM count from torch.cuda.get_device_properties and assert that every case runs the path it is
named after; tests/test_env_launch_shapes_host.py pins the mirror at the B200's 148 SMs.
"""
import numpy as np

STEP_THREADS = 256
SMEM_DEFAULT = 48 * 1024                   # dynamic shared memory a kernel may use without cudaFuncSetAttribute
STEP_SMEM_PER_HUMAN = 16 + 16 + 8 + 4      # float4 pv + float4 gr + float2 nv + float th
STEP_SMEM_SCRATCH = 2 * STEP_THREADS * 16  # ranked + projected lines of every lane group
STEP_SMEM_STATIC = 2560                    # static shared memory of crowd_step_kernel (cuobjdump --dump-resource-usage)
RESET_SYNC_CTAS = 592
RESET_LIST_CTAS = 1184
B200_SMS = 148
MAX_GROUPS = 8


def pick_group(m):
    """Lanes per ORCA solve: the next power of two >= the neighbour count m, at least 4."""
    return 4 if m <= 4 else (8 if m <= 8 else (16 if m <= 16 else 32))


def step_envs_per_cta_limit(H):
    """Largest E whose E * H humans fit the group form's 48 KB of shared memory beside its static shared memory (the
    launcher clamps CN_STEP_ENVS_PER_CTA to it)."""
    return (SMEM_DEFAULT - STEP_SMEM_STATIC - STEP_SMEM_SCRATCH) // (H * STEP_SMEM_PER_HUMAN)


def step_shape(n_envs, H, num_sms, robot_visible=False, form="group", envs_per_cta=None):
    """dict(G, E, grid, last, smem, small_batch) of one crowd step.  form: "group" (the default launch; "split", the
    two-launch form, runs its ORCA kernel with the same shape) or "seq" (CN_STEP_SEQ=1).  envs_per_cta: the value of
    CN_STEP_ENVS_PER_CTA (None: unset).  `last` = envs of the last CTA (== E unless the last CTA is partial)."""
    M = H - 1 + (1 if robot_visible else 0)
    G = pick_group(max(M, 1))
    knob = envs_per_cta if envs_per_cta is not None and 1 <= envs_per_cta <= 64 else None
    if form == "seq" and 1 <= M <= 32:
        E = max(1, min(64, STEP_THREADS // H))
        small = n_envs < E * 2 * num_sms
        if small:
            E = max(1, n_envs // (2 * num_sms))
        if knob is not None:
            E = knob
        S = min((E * H + 31) & ~31, STEP_THREADS)
        smem = E * H * STEP_SMEM_PER_HUMAN + S * M * (16 + 4)
    else:
        E = min(64, max(8, (2 * (STEP_THREADS // G) + H - 1) // H))
        small = n_envs < E * 4 * num_sms
        if small:
            E = max(1, n_envs // (4 * num_sms))
        if knob is not None:
            E = min(knob, step_envs_per_cta_limit(H))
        smem = E * H * STEP_SMEM_PER_HUMAN + STEP_SMEM_SCRATCH + STEP_SMEM_STATIC
    grid = -(-n_envs // E)
    return dict(G=G, E=E, grid=grid, last=n_envs - (grid - 1) * E, smem=smem, small_batch=small)


def reset_grid(n_envs, mode):
    """CTAs of one reset launch.  mode: "live" (cn_env_reset), "spare" (the refill after a reset), "sync" (the fall-back
    after a step) or "list" (the refill of the envs a step appended to the refill list)."""
    if mode == "sync":
        return min(n_envs, RESET_SYNC_CTAS)
    if mode == "list":
        return min(n_envs, RESET_LIST_CTAS)
    assert mode in ("live", "spare"), mode
    return n_envs


def strided_iterations(entries, grid):
    """Envs the busiest CTA of a grid-stride loop over `entries` envs handles."""
    return -(-entries // grid) if entries > 0 else 0


def robot_act_shape(n_envs, H):
    """dict(G, per_cta, grid, last) of cn_env_robot_act."""
    G = pick_group(H)
    per = STEP_THREADS // G
    grid = -(-n_envs // per)
    return dict(G=G, per_cta=per, grid=grid, last=n_envs - (grid - 1) * per)


def state_layout(n_envs, H):
    """(offsets, total): byte offset of every array of the state buffer carved by cn_env_create, and its size
    (= cn_env_state_bytes).  Every array starts on a 256-byte boundary."""
    nh = n_envs * H
    arrays = (("hum_pv", 16 * nh), ("hum_gr", 16 * nh), ("hum_bel", 16 * nh), ("hum_br", 4 * nh), ("hum_th", 4 * nh),
              ("rob_pv", 16 * n_envs), ("rob_gr", 16 * n_envs), ("rob_x", 16 * n_envs), ("rob_acc", 8 * n_envs),
              ("ctr", 16 * n_envs), ("sp_pv", 16 * nh), ("sp_gr", 16 * nh), ("sp_th", 4 * nh), ("sp_rob_pv", 16 * n_envs),
              ("sp_rob_gr", 16 * n_envs), ("sp_theta", 4 * n_envs), ("sp_meta", 16 * n_envs), ("need_spare", n_envs),
              ("need_sync", n_envs), ("sync_count", 16), ("refill_list", 4 * n_envs), ("hum_nv", 8 * nh),
              ("grp", 16 * MAX_GROUPS * n_envs), ("sp_grp", 16 * MAX_GROUPS * n_envs))
    offsets, off = {}, 0
    for name, nbytes in arrays:
        offsets[name] = off
        off = (off + nbytes + 255) & ~255
    return offsets, off


def tile_state(inp, n_envs, case_stride=100003):
    """Repeat the envs of a sampled state (dict of arrays with a leading env axis, as state_sampler.sample returns) to
    n_envs envs.  Tile k (envs k * n0 .. (k + 1) * n0 - 1) gets case_counter + k * case_stride and scenario_counter + k,
    so every tile draws its own random numbers (goal re-sampling, the next episode)."""
    n0 = next(iter(inp.values())).shape[0]
    idx = np.arange(n_envs) % n0
    tile = (np.arange(n_envs) // n0).astype(np.int64)
    out = {k: np.ascontiguousarray(v[idx]) for k, v in inp.items()}
    if "counters" in out:
        c = out["counters"].astype(np.int64)
        c[:, 2] += tile * case_stride
        c[:, 1] += tile
        assert c.max() < 2 ** 31
        out["counters"] = np.ascontiguousarray(c, np.int32)
    return out
