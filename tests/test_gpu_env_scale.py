"""GPU: the env half of the hot path (crowd step, reset, spare-episode refill and its join, observe, state convert, robot
act) at the benchmark shapes, against the C oracle.

test_gpu_crowd_step.py runs at most 4096 envs: at H = 20 that is the small-batch launch rule (E = 3 envs per CTA), one env
per CTA in the fall-back and the refill, and a refill that finishes at once.  Here every case runs the path the benchmark
runs, and asserts that it does with the host mirror of the launchers (env_launch_shapes.py):
  * one step at c3 (16384 x 20, FOV 0.5), c5 (65536 x 20), c2 (1024 x 10, unicycle), c1 (16 x 5) and c3 with a partial
    last CTA, in all three step forms, with and without auto-reset;
  * CN_STEP_ENVS_PER_CTA from 1 to 64 (the launcher clamps what does not fit 48 KB of shared memory);
  * resets at scale, full and masked, and the group environment;
  * the synchronous fall-back and the refill striding over more envs than they have CTAs, and the refill list
    overflowing, in lock-step with the oracle;
  * guard rows around every output and a sentinel tail behind the state buffer;
  * the robot-act kernel with a partial last CTA;
  * the graphed and pipelined rollouts against the eager loop at c3, and a refill that really overlaps other work.
Comparison rules (gpu_helpers.compare): flags, indices, masks and counters bit-exact; floats after one step within 2e-6;
multi-step positions and velocities within 1e-4; rewards within 1e-5.  Every check prints its worst error beside its
tolerance (run with -s)."""
import ctypes as C
import functools
import os

import numpy as np
import pytest
import torch

from crowdnav_dsrnn_b200 import Config, _lib, abi
from oracle import crowd_oracle, state_sampler
import env_launch_shapes as S
import gpu_helpers as G
import robot_oracle

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL_STEP, TOL_TRAJ, TOL_REWARD = 2e-6, 1e-4, 1e-5
LAUNCH_SWITCHES = ("CN_STEP_SEQ", "CN_STEP_SPLIT", "CN_STEP_ENVS_PER_CTA", "CN_REFILL_THREADS")
FORMS = {"group": {}, "seq": {"CN_STEP_SEQ": "1"}, "split": {"CN_STEP_SPLIT": "1"}}


@pytest.fixture(autouse=True)
def _default_launch(monkeypatch):
    for k in LAUNCH_SWITCHES:
        monkeypatch.delenv(k, raising=False)


def _set_form(monkeypatch, form):
    monkeypatch.delenv("CN_STEP_SEQ", raising=False)
    monkeypatch.delenv("CN_STEP_SPLIT", raising=False)
    for k, v in FORMS[form].items():
        monkeypatch.setenv(k, v)


@pytest.fixture(params=list(FORMS))
def step_form(request, monkeypatch):
    """The three forms of the step: lane group per human in one launch (default), thread per human (CN_STEP_SEQ=1), ORCA
    kernel + env-tail kernel (CN_STEP_SPLIT=1).  The launcher reads the switches at every call."""
    _set_form(monkeypatch, request.param)
    return request.param


def _sms():
    return torch.cuda.get_device_properties(DEV).multi_processor_count


def _cfg(human_num, kinematics="holonomic", **over):
    c = Config(kinematics=kinematics, human_num=human_num)
    for k, v in over.items():
        sec, _, attr = k.partition(".")
        setattr(getattr(c, sec), attr, v)
    return c


def _report(where, errs):
    """errs: name -> (worst error, tolerance).  Prints and asserts."""
    for name, (err, tol) in errs.items():
        print("%-34s %-22s worst %.3g  tol %.0e" % (where, name, err, tol))
    for name, (err, tol) in errs.items():
        assert err <= tol, "%s %s: worst error %g > %g" % (where, name, err, tol)


def _report_compare(where, rep, tol=TOL_STEP):
    _report(where, {k: (v, tol) for k, v in rep.items() if k != "bit_exact_humans"})


def _max_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max()) if a.size else 0.0


# ---------------------------------------------------------------------------------------------------- inputs
C3 = dict(human_num=20, **{"robot.FOV": 0.5})
CASES = {            # name -> (config overrides, envs, sample key)
    "c3": (C3, 16384, "h20"),
    "c3_partial": (C3, 16384 + 5, "h20"),
    "c2": (dict(human_num=10, kinematics="unicycle", **{"env.time_step": 0.1, "reward.discomfort_penalty_factor": 1.0}), 1024, "c2"),
    "c1": (dict(human_num=5, **{"sim.train_val_sim": ["circle_crossing"]}), 16, "c1"),
    "c5": (dict(human_num=20), 65536, "h20"),
}
SAMPLE_ENVS = 4096


@functools.lru_cache(maxsize=None)
def _sample(key):
    """state_sampler.sample is a per-human Python loop: sample at most 4096 envs once and tile them to N."""
    kw, n = {"h20": (C3, SAMPLE_ENVS), "c2": (CASES["c2"][0], 1024), "c1": (CASES["c1"][0], 16)}[key]
    cfg = abi.flatten_config(_cfg(**kw), n, phase="train")
    return state_sampler.sample(cfg, n, seed=4242 + n)


def _inputs(name):
    kw, n, key = CASES[name]
    inp = S.tile_state(_sample(key), n)
    act = inp.pop("action")
    return kw, n, inp, act


_ORACLE_STEPS = {}


def _oracle_step(name, cfg, inp, act, auto_reset):
    """One oracle step of a case (cached: every step form and envs-per-CTA value is compared with the same result)."""
    key = (name, bool(auto_reset))
    if key not in _ORACLE_STEPS:
        ost = G.oracle_state_from(inp, act.shape[0], cfg.human_num)
        oout = crowd_oracle.step(cfg, ost, act, auto_reset=auto_reset, n_threads=8)
        _ORACLE_STEPS[key] = (G.oracle_out_to_numpy(oout), ost)
    return _ORACLE_STEPS[key]


def _gpu_step(kw, n, inp, act, auto_reset):
    eng = G.make_engine(_cfg(**kw), n)
    eng.set_state(**inp)
    buf = eng.step(torch.from_numpy(act).to(DEV), auto_reset=auto_reset)
    out, st = G.buf_to_numpy(buf), G.state_to_numpy(eng.get_state())
    cfg = eng.cfg
    eng.close()
    return cfg, out, st


def _step_vs_oracle(name, auto_reset, where):
    kw, n, inp, act = _inputs(name)
    cfg, out, st = _gpu_step(kw, n, inp, act, auto_reset)
    oout, ost = _oracle_step(name, cfg, inp, act, auto_reset)
    rep = G.compare(out, st, oout, ost, where=where)
    _report_compare(where, rep)
    assert out["done"].sum() > 0
    return out, st


def _assert_same_bits(a, b, where):
    for k in a:
        x, y = np.ascontiguousarray(a[k]), np.ascontiguousarray(b[k])
        assert x.shape == y.shape and x.tobytes() == y.tobytes(), "%s: %s differs" % (where, k)


def _assert_step_shape(name, form):
    kw, n, _ = CASES[name]
    sh = S.step_shape(n, kw["human_num"], _sms(), form="seq" if form == "seq" else "group")
    if name in ("c3", "c3_partial", "c5") and form != "seq":
        assert (sh["G"], sh["E"], sh["small_batch"]) == (32, 8, False), sh          # the production rule, not small-batch
    if name == "c3_partial":
        assert n % sh["E"] != 0 and sh["last"] < sh["E"], sh
    return sh


# ---------------------------------------------------------------------------------------------------- 1. one step
@pytest.mark.parametrize("auto_reset", [False, True])
@pytest.mark.parametrize("name", ["c3", "c3_partial", "c2", "c1"])
def test_one_step_at_benchmark_shapes(name, auto_reset, step_form):
    sh = _assert_step_shape(name, step_form)
    out, _ = _step_vs_oracle(name, auto_reset, "%s %s ar=%d E=%d" % (name, step_form, auto_reset, sh["E"]))
    if auto_reset and name.startswith("c3"):
        # a fresh engine has no spares: every finished env takes the synchronous fall-back, more than its 592 CTAs
        n_done = int(out["done"].sum())
        assert S.strided_iterations(n_done, S.reset_grid(CASES[name][1], "sync")) >= 2, n_done


def test_c5_step_and_reset_at_65536(monkeypatch):
    """All 65536-env cases in one test: one step in the three forms with and without auto-reset, then the reset."""
    kw, n, _ = CASES["c5"]
    for form in FORMS:
        _set_form(monkeypatch, form)
        sh = _assert_step_shape("c5", form)
        for auto_reset in (False, True):
            _step_vs_oracle("c5", auto_reset, "c5 %s ar=%d E=%d" % (form, auto_reset, sh["E"]))
    _set_form(monkeypatch, "group")
    _reset_vs_oracle(kw, n, "c5 reset")


# ---------------------------------------------------------------------------------------------------- 2. envs per CTA
_DEFAULT_BITS = {}


@pytest.mark.parametrize("envs_per_cta", [1, 3, 7, 8, 13, 32, 43, 44, 64])
def test_envs_per_cta_sweep(envs_per_cta, monkeypatch):
    """c3 with a partial last CTA at every CN_STEP_ENVS_PER_CTA: oracle parity and the default's bits.  44 and 64 ask for
    more than the 48 KB of shared memory the kernel may use and are clamped by the launcher to 43 (E = 44 and 64 failed
    to launch before the clamp)."""
    name = "c3_partial"
    kw, n, inp, act = _inputs(name)
    if "bits" not in _DEFAULT_BITS:
        _, out0, st0 = _gpu_step(kw, n, inp, act, True)
        _DEFAULT_BITS["bits"] = (out0, st0)
    sh = S.step_shape(n, kw["human_num"], _sms(), envs_per_cta=envs_per_cta)
    assert sh["E"] == min(envs_per_cta, 43) and sh["smem"] <= S.SMEM_DEFAULT, sh
    monkeypatch.setenv("CN_STEP_ENVS_PER_CTA", str(envs_per_cta))
    cfg, out, st = _gpu_step(kw, n, inp, act, True)
    oout, ost = _oracle_step(name, cfg, inp, act, True)
    where = "%s E=%d (knob %d) last CTA %d" % (name, sh["E"], envs_per_cta, sh["last"])
    _report_compare(where, G.compare(out, st, oout, ost, where=where))
    out0, st0 = _DEFAULT_BITS["bits"]
    _assert_same_bits(out, out0, where)
    _assert_same_bits(st, st0, where)


# ---------------------------------------------------------------------------------------------------- 3. reset at scale
def _reset_vs_oracle(kw, n, where, seed=7):
    eng = G.make_engine(_cfg(**kw), n, seed=seed)
    cfg, H = eng.cfg, eng.h
    out = G.buf_to_numpy(eng.reset())
    ost = crowd_oracle.OracleState(n, H)
    oout = G.oracle_out_to_numpy(crowd_oracle.reset(cfg, ost, n_threads=8))

    def check(rows, label):
        st = G.state_to_numpy(eng.get_state())
        errs = {}
        for f in ("robot_node", "temporal_edges", "spatial_edges"):
            errs[f] = (_max_err(out[f][rows], oout[f][rows]), TOL_STEP)
        assert np.array_equal(out["visible_mask"][rows], oout["visible_mask"][rows]), label
        for f in G.STATE_FIELDS:
            if f == "counters":
                assert np.array_equal(st[f], ost.counters), label
            else:
                errs["state." + f] = (_max_err(st[f], getattr(ost, f)), TOL_STEP)
        _report(label, errs)

    check(np.arange(n), where)
    for mname, mask in (("every 3rd", np.arange(n) % 3 == 0), ("tail", np.arange(n) >= n - n // 5 - 3)):
        mask = mask.astype(np.uint8)
        out = G.buf_to_numpy(eng.reset(torch.from_numpy(mask).to(DEV)))
        oout = G.oracle_out_to_numpy(crowd_oracle.reset(cfg, ost, mask=mask, n_threads=8))
        check(mask.astype(bool), "%s mask %s" % (where, mname))
    eng.close()


@pytest.mark.parametrize("kw,n", [(C3, 16384), (dict(human_num=9, **{"sim.group_human": True}), 16384)],
                         ids=["c3_16384x20", "group_16384x9"])
def test_reset_at_scale(kw, n):
    _reset_vs_oracle(kw, n, "reset %dx%d" % (n, kw["human_num"]))


# ---------------------------------------------------------------------------------------------------- 4. fall-back / refill
def _blob(eng, layout, name, dtype, count):
    off = layout[name]
    item = torch.tensor([], dtype=dtype).element_size()
    return eng.state[off:off + count * item].view(dtype)


def _spare_valid(eng, layout):
    """Per env: does its spare episode match its counters (the step kernel would swap it in)?"""
    n = eng.n
    meta = _blob(eng, layout, "sp_meta", torch.int32, 4 * n).view(n, 4).cpu().numpy()
    ctr = _blob(eng, layout, "ctr", torch.int32, 4 * n).view(n, 4).cpu().numpy()
    return (meta[:, 0] == 1) & (meta[:, 1] == ctr[:, 2]) & (meta[:, 2] == ctr[:, 1])


def _sync_count(eng, layout):
    return _blob(eng, layout, "sync_count", torch.int32, 4).cpu().numpy()


def _refill(eng):
    _lib.check(eng.lib.cn_env_refill(eng.handle, eng._stream()), "cn_env_refill")


def _force_timeout(eng, ost, rows):
    ctr = eng.get_state()["counters"]
    ctr[torch.from_numpy(rows).to(DEV), 0] = eng.cfg.timeout_step
    eng.set_state(counters=ctr)
    ost.counters[rows, 0] = eng.cfg.timeout_step


def _lockstep(eng, ost, act, t, where):
    """One deferred-refill step on both sides; flags and counters bit-exact, rewards to 1e-5.  Returns (out, reward err)."""
    out = G.buf_to_numpy(eng.step(torch.from_numpy(act).to(DEV), auto_reset=True, defer_refill=True))
    oout = crowd_oracle.step(eng.cfg, ost, act, auto_reset=True, n_threads=8)
    for f in ("done", "event"):
        assert np.array_equal(out[f], getattr(oout, f)), "%s step %d: %s" % (where, t, f)
    assert np.array_equal(out["visible_mask"], oout.visible_mask.astype(np.int64)), "%s step %d" % (where, t)
    assert np.array_equal(G.state_to_numpy(eng.get_state())["counters"], ost.counters), "%s step %d: counters" % (where, t)
    return out, _max_err(out["reward"], oout.reward)


def _final_state(eng, ost, where, rew):
    st = G.state_to_numpy(eng.get_state())
    assert np.array_equal(st["counters"], ost.counters)
    _report(where, {"reward (all steps)": (rew, TOL_REWARD), "humans": (_max_err(st["humans"], ost.humans), TOL_TRAJ),
                    "robot": (_max_err(st["robot"], ost.robot), TOL_TRAJ)})


def test_fallback_and_refill_strides_track_oracle():
    """16384 x 20 for 30 steps of a fixed action tape.  Even envs get stale spares (case counter moved behind their back),
    every third env is forced to time out at the first step: more envs take the fall-back in one step than its 592 CTAs
    and more are appended to the refill list than the refill's 1184 CTAs.  After every refill each listed env must hold a
    spare that matches its counters, and the counters of both launches must be re-armed."""
    n = 16384
    eng = G.make_engine(_cfg(**C3), n, seed=11)
    layout, total = S.state_layout(n, eng.h)
    assert total == eng.state.numel()
    cfg = eng.cfg
    eng.reset()
    ost = crowd_oracle.OracleState(n, cfg.human_num)
    crowd_oracle.reset(cfg, ost, n_threads=8)
    st = eng.get_state()
    st["counters"][::2, 2] += 7
    eng.set_state(counters=st["counters"])
    ost.counters[:] = st["counters"].cpu().numpy()
    _force_timeout(eng, ost, np.arange(0, n, 3))
    rng = np.random.default_rng(9)
    max_sync = max_list = 0
    rew = 0.0
    listed = np.zeros(0, np.int64)
    for t in range(30):
        eng.join()
        torch.cuda.synchronize()
        assert (_sync_count(eng, layout) == 0).all(), "step %d: sync_count not re-armed" % t
        valid = _spare_valid(eng, layout)
        assert valid[listed].all(), "step %d: %d listed envs without a spare" % (t, int((~valid[listed]).sum()))
        act = rng.normal(0, 0.7, (n, 2)).astype(np.float32)
        out, r = _lockstep(eng, ost, act, t, "strides")
        rew = max(rew, r)
        torch.cuda.synchronize()
        done = out["done"].astype(bool)
        n_sync, n_swap = int((done & ~valid).sum()), int((done & valid).sum())
        sc = _sync_count(eng, layout)
        assert sc[0] == 0 and sc[1] == 0, "step %d: fall-back counter not re-armed %s" % (t, sc)
        assert sc[2] == n_sync + n_swap, "step %d: %d list entries for %d + %d resets" % (t, sc[2], n_sync, n_swap)
        assert not _blob(eng, layout, "need_sync", torch.uint8, n).any()
        lst = _blob(eng, layout, "refill_list", torch.int32, n)[:sc[2]].cpu().numpy()
        assert np.array_equal(np.sort(lst), np.flatnonzero(done)), "step %d: refill list" % t
        listed = lst.astype(np.int64)
        max_sync, max_list = max(max_sync, n_sync), max(max_list, int(sc[2]))
        _refill(eng)
    _final_state(eng, ost, "strides 16384x20 30 steps", rew)
    print("strides: most fall-back resets in one step %d (%d CTAs), most list entries %d (%d CTAs)"
          % (max_sync, S.reset_grid(n, "sync"), max_list, S.reset_grid(n, "list")))
    assert S.strided_iterations(max_sync, S.reset_grid(n, "sync")) >= 2
    assert S.strided_iterations(max_list, S.reset_grid(n, "list")) >= 2
    eng.close()


def test_refill_list_overflow_tracks_oracle():
    """512 x 5, episodes of five steps.  Steps with the refill deferred and nobody starting it: envs 0..299 end twice (their
    second reset goes through the fall-back and lands past the list's 512 entries, a duplicate of their first), envs
    300..511 end after the list is full (dropped).  cn_env_refill then makes spares for the listed envs only; a dropped
    env must take the fall-back at its next reset.  The oracle's plain reset tracks every step."""
    n = 512
    kw = dict(human_num=5, **{"env.time_limit": 2})
    eng = G.make_engine(_cfg(**kw), n, seed=13)
    layout, _ = S.state_layout(n, eng.h)
    cfg = eng.cfg
    assert cfg.timeout_step <= 6
    eng.reset()
    ost = crowd_oracle.OracleState(n, cfg.human_num)
    crowd_oracle.reset(cfg, ost, n_threads=8)
    rng = np.random.default_rng(17)
    tape = lambda: rng.normal(0, 0.7, (n, 2)).astype(np.float32)
    rew, t = 0.0, 0
    for rows in (np.arange(300), np.arange(300), np.arange(300, n)):
        _force_timeout(eng, ost, rows)
        out, r = _lockstep(eng, ost, tape(), t, "overflow")
        rew, t = max(rew, r), t + 1
        assert out["done"][rows].all()
    torch.cuda.synchronize()
    sc = _sync_count(eng, layout)
    assert sc[2] > n, "the list did not overflow: %s" % sc
    lst = _blob(eng, layout, "refill_list", torch.int32, n).cpu().numpy()
    dropped = np.setdiff1d(np.arange(n), lst)
    print("overflow: %d entries for a list of %d, %d distinct envs listed, %d dropped" % (sc[2], n, len(np.unique(lst)), len(dropped)))
    assert len(np.unique(lst)) < n and len(dropped) > 0
    _refill(eng)
    eng.join()
    torch.cuda.synchronize()
    assert (_sync_count(eng, layout) == 0).all()
    valid = _spare_valid(eng, layout)
    assert valid[lst].all() and not valid[dropped].any()
    first_reset = np.zeros(n, bool)
    for k in range(3 * cfg.timeout_step):
        eng.join()
        torch.cuda.synchronize()
        valid = _spare_valid(eng, layout)
        out, r = _lockstep(eng, ost, tape(), t, "overflow")
        rew, t = max(rew, r), t + 1
        done = out["done"].astype(bool)
        new = done & ~first_reset
        assert not valid[np.intersect1d(np.flatnonzero(new), dropped)].any()      # dropped envs: fall-back first
        first_reset |= done
        _refill(eng)
    assert first_reset[dropped].all()
    _final_state(eng, ost, "overflow 512x5", rew)
    eng.close()


# ---------------------------------------------------------------------------------------------------- 5. write guards
GUARD = 128


class Guarded:
    """A [GUARD + n + GUARD, ...] device tensor: NaN (floats) / 0xFF (integers) guard rows around the rows a call may write."""

    def __init__(self, shape, dtype):
        n = shape[0]
        self.full = torch.empty((n + 2 * GUARD,) + tuple(shape[1:]), dtype=dtype, device=DEV)
        if dtype.is_floating_point:
            self.full.fill_(float("nan"))
        else:
            self.full.view(torch.uint8).fill_(0xFF)
        self.inner = self.full[GUARD:GUARD + n]
        self.ref = self.full.clone()

    def ptr(self):
        return C.c_void_p(self.inner.data_ptr())

    def intact(self):
        b = lambda x: x.contiguous().view(torch.uint8)
        return (torch.equal(b(self.full[:GUARD]), b(self.ref[:GUARD])) and
                torch.equal(b(self.full[-GUARD:]), b(self.ref[-GUARD:])))


def _check_guards(bufs, what):
    torch.cuda.synchronize()
    bad = [k for k, g in bufs.items() if not g.intact()]
    assert not bad, "%s wrote outside its outputs: %s" % (what, bad)
    for k, g in bufs.items():
        if g.inner.dtype == torch.float32 and what != "cn_env_robot_act":
            assert not torch.isnan(g.inner).any(), "%s left %s unwritten" % (what, k)


@pytest.mark.parametrize("n", [16384 + 5, 3])
def test_env_calls_write_only_their_outputs(n):
    """cn_env_reset / step / observe / get_state / robot_act through the C ABI on caller-owned buffers with guard rows, and
    a state buffer with a sentinel head and tail: nothing outside the outputs changes."""
    lib = _lib.load()
    H = 20
    cfg = abi.flatten_config(_cfg(**C3), n, phase="train", seed=3)
    nbytes = lib.cn_env_state_bytes(C.byref(cfg), n)
    assert nbytes == S.state_layout(n, H)[1]
    head, tail = 4096, 1 << 16
    blob = torch.full((head + nbytes + tail,), 0xA5, dtype=torch.uint8, device=DEV)
    handle = C.c_void_p()
    _lib.check(lib.cn_env_create(C.byref(cfg), n, DEV.index or 0, C.c_void_p(blob.data_ptr() + head), nbytes, C.byref(handle)),
               "cn_env_create")
    stream = lambda: C.c_void_p(torch.cuda.current_stream(DEV).cuda_stream)
    f32, i32, u8 = torch.float32, torch.int32, torch.uint8
    obs = {"robot_node": Guarded((n, 1, 7), f32), "temporal_edges": Guarded((n, 1, 2), f32),
           "spatial_edges": Guarded((n, H, 2), f32), "visible_mask": Guarded((n,), i32)}
    obs_struct = lambda: abi.CnObsOut(*[obs[k].ptr() for k in ("robot_node", "temporal_edges", "spatial_edges", "visible_mask")])
    try:
        _lib.check(lib.cn_env_reset(handle, None, C.byref(obs_struct()), stream()), "cn_env_reset")
        _check_guards(obs, "cn_env_reset")
        mask = Guarded((n,), u8)
        mask.inner.copy_((torch.arange(n, device=DEV) % 2).to(u8))
        mask.ref = mask.full.clone()
        _lib.check(lib.cn_env_reset(handle, mask.ptr(), C.byref(obs_struct()), stream()), "cn_env_reset (masked)")
        _check_guards(dict(obs, mask=mask), "cn_env_reset (masked)")
        rng = np.random.default_rng(1)
        for t in range(3):
            outs = dict(obs, reward=Guarded((n,), f32), done=Guarded((n,), u8), event=Guarded((n,), i32),
                        scenario=Guarded((n,), i32), info=Guarded((n, abi.INFO_DIM), f32), episode_return=Guarded((n,), f32),
                        episode_length=Guarded((n,), i32), goal_changed=Guarded((n,), i32), not_done=Guarded((n, 1), f32))
            act = Guarded((n, 2), f32)
            act.inner.copy_(torch.from_numpy(rng.normal(0, 0.7, (n, 2)).astype(np.float32)))
            act.ref = act.full.clone()
            so = abi.CnStepOut(obs_struct(), *[outs[k].ptr() for k in ("reward", "done", "event", "scenario", "info",
                                                                       "episode_return", "episode_length", "goal_changed", "not_done")])
            _lib.check(lib.cn_env_step(handle, act.ptr(), C.byref(so), 1 + (t % 2), stream()), "cn_env_step")
            _check_guards(dict(outs, action=act), "cn_env_step")
            if t % 2:
                _lib.check(lib.cn_env_refill(handle, stream()), "cn_env_refill")
        _lib.check(lib.cn_env_observe(handle, C.byref(obs_struct()), stream()), "cn_env_observe")
        _check_guards(obs, "cn_env_observe")
        view = {"robot": Guarded((n, 9), f32), "humans": Guarded((n, H, 9), f32), "belief": Guarded((n, H, 5), f32),
                "extras": Guarded((n, 4), f32), "counters": Guarded((n, 4), i32), "episode_return": Guarded((n,), f32),
                "groups": Guarded((n, abi.MAX_GROUPS, 4), f32)}
        sv = abi.CnStateView(*[view[k].ptr() for k in G.STATE_FIELDS])
        _lib.check(lib.cn_env_get_state(handle, C.byref(sv), stream()), "cn_env_get_state")
        _check_guards(view, "cn_env_get_state")
        for policy in (abi.POLICY_ORCA, abi.POLICY_SOCIAL_FORCE):
            a = {"action": Guarded((n, 2), f32)}
            _lib.check(lib.cn_env_robot_act(handle, policy, a["action"].ptr(), stream()), "cn_env_robot_act")
            _check_guards(a, "cn_env_robot_act")
        _lib.check(lib.cn_env_join(handle, stream()), "cn_env_join")
        torch.cuda.synchronize()
        assert (blob[:head] == 0xA5).all() and (blob[head + nbytes:] == 0xA5).all(), "the state buffer's sentinels changed"
    finally:
        lib.cn_env_destroy(handle)
    torch.cuda.synchronize()
    assert (blob[:head] == 0xA5).all() and (blob[head + nbytes:] == 0xA5).all()


# ---------------------------------------------------------------------------------------------------- 6. robot act
@pytest.mark.parametrize("policy", ["orca", "social_force"])
@pytest.mark.parametrize("H,n", [(20, 16384 + 3), (5, 1027)])
def test_robot_act_partial_last_cta(H, n, policy):
    sh = S.robot_act_shape(n, H)
    assert sh["last"] < sh["per_cta"], sh
    c = _cfg(H)
    c.robot.FOV = 0.5
    eng = G.make_engine(c, n, seed=31 + H)
    eng.reset()
    for _ in range(3):
        eng.step(eng.robot_act(policy), auto_reset=True)
    got = eng.robot_act(policy).cpu().numpy()
    ost = crowd_oracle.OracleState(n, H)
    for f, v in G.state_to_numpy(eng.get_state()).items():
        getattr(ost, f)[...] = v
    want = robot_oracle.robot_act(eng.cfg, ost, policy)
    where = "robot_act %s %dx%d last CTA %d of %d" % (policy, n, H, sh["last"], sh["per_cta"])
    if policy == "orca":
        bad = got.view(np.uint32) != want.view(np.uint32)
        _report(where, {"action (bits)": (float(bad.any(axis=1).sum()), 0)})
    else:
        ok = np.isfinite(want).all(axis=1)
        assert np.array_equal(np.isfinite(got).all(axis=1), ok)
        _report(where, {"action": (_max_err(got[ok], want[ok]), 1e-6)})
    assert np.abs(got[-sh["last"]:]).sum() > 0
    eng.close()


# ---------------------------------------------------------------------------------------------------- 7. graphed rollout
@pytest.fixture(scope="module")
def policy_27776():
    from crowdnav_dsrnn_b200.model import Policy
    from crowdnav_dsrnn_b200.spaces import crowd_spaces

    w = np.load(os.path.join(GOLDEN, "weights_holonomic_27776.npz"))
    obs_space, act_space = crowd_spaces(20)
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(0)
        policy = Policy(obs_space.spaces, act_space, base="srnn", base_kwargs=_cfg(**C3))
    policy.load_state_dict({k: torch.as_tensor(w[k]) for k in w.files})
    policy = policy.to(DEV)
    yield policy
    if policy._handle is not None:
        policy.start_refill_of(None)
        policy.set_edge_image(None, None)


def _eager_loop(policy, cfg, n, steps):
    from crowdnav_dsrnn_b200.envs import CrowdVecEnv

    venv = CrowdVecEnv(cfg, n, DEV, seed=5, phase="train")
    obs = venv.reset()
    hx = {"human_node_rnn": torch.zeros(n, 1, 128, device=DEV), "human_human_edge_rnn": torch.zeros(n, 21, 256, device=DEV)}
    masks = torch.zeros(n, 1, device=DEV)
    trace = []
    for _ in range(steps):
        value, action, _, hx = policy.act(obs, hx, masks, deterministic=True)
        obs, reward, done, buf = venv.step_device(action)
        masks = (1.0 - done.float()).unsqueeze(1)
        trace.append((reward.clone(), done.clone(), buf.event.clone()))
    st = {k: v.clone() for k, v in venv.engine.get_state().items()}
    venv.close()
    return trace, st, hx, masks, obs, value, action


def test_graphed_rollout_equals_eager_at_c3(policy_27776):
    from crowdnav_dsrnn_b200.envs import CrowdVecEnv
    from crowdnav_dsrnn_b200.rollout import GraphedRollout

    n, steps, cfg = 16384, 20, _cfg(**C3)
    trace, st_e, hx_e, _, _, _, _ = _eager_loop(policy_27776, cfg, n, steps)
    venv = CrowdVecEnv(cfg, n, DEV, seed=5, phase="train")
    obs = venv.reset()
    roll = GraphedRollout(policy_27776, venv, obs, edge_image=True)
    assert roll.use_image
    for _ in range(steps - roll.steps):
        buf = roll.step()
    torch.cuda.synchronize()
    st_g = {k: v.clone() for k, v in venv.engine.get_state().items()}
    hx_g, _ = roll.hidden()
    for a, b in zip(trace[-1], (buf.reward, buf.done, buf.event)):
        assert torch.equal(a, b)
    for k in st_e:
        assert torch.equal(st_e[k], st_g[k]), k
    assert torch.equal(hx_e["human_human_edge_rnn"], hx_g["human_human_edge_rnn"])
    assert torch.equal(hx_e["human_node_rnn"], hx_g["human_node_rnn"])
    n_done = int(sum(t[1].sum() for t in trace))
    print("graphed c3: %d episodes ended in %d steps, state / hidden state bit-identical to the eager loop" % (n_done, steps))
    assert n_done > 0
    roll.close()
    venv.close()


def test_pipelined_rollout_equals_eager_at_c3(policy_27776):
    from crowdnav_dsrnn_b200.rollout import PipelinedRollout

    n, cycles, cfg = 16384, 20, _cfg(**C3)
    _, st_e, hx, masks, obs, _, _ = _eager_loop(policy_27776, cfg, n, cycles)
    he_c, hn_c = hx["human_human_edge_rnn"].clone(), hx["human_node_rnn"].clone()
    value, action, _, hx1 = policy_27776.act(obs, hx, masks, deterministic=True)      # half 1 is one forward ahead
    roll = PipelinedRollout(policy_27776, cfg, n, DEV, seed=5, phase="train")
    for _ in range(cycles - roll.steps):
        roll.step()
    torch.cuda.synchronize()
    halves = roll.state()
    n_a = roll.sizes[0]
    for k in st_e:
        got = torch.cat([h["engine"].get_state()[k] for h in halves], 0)
        assert torch.equal(st_e[k], got), k
    assert torch.equal(halves[0]["hidden"]["human_human_edge_rnn"], he_c[:n_a])
    assert torch.equal(halves[0]["hidden"]["human_node_rnn"], hn_c[:n_a])
    assert torch.equal(halves[1]["hidden"]["human_human_edge_rnn"], hx1["human_human_edge_rnn"][n_a:])
    assert torch.equal(halves[1]["hidden"]["human_node_rnn"], hx1["human_node_rnn"][n_a:])
    assert torch.equal(halves[1]["action"], action[n_a:]) and torch.equal(halves[1]["value"], value[n_a:])
    print("pipelined c3: split %d + %d, env and hidden state bit-identical to the eager loop" % roll.sizes)
    roll.close()


def test_refill_beside_gemm_tracks_oracle():
    """30 eager c3 steps with the refill deferred and started by cn_env_refill right before a long GEMM on the caller's
    stream, so the refill runs while the GEMM does; the next step joins it.  In lock-step with the oracle."""
    n = 16384
    eng = G.make_engine(_cfg(**C3), n, seed=23)
    cfg = eng.cfg
    eng.reset()
    ost = crowd_oracle.OracleState(n, cfg.human_num)
    crowd_oracle.reset(cfg, ost, n_threads=8)
    g = torch.Generator(device=DEV).manual_seed(0)
    a = torch.randn(4096, 4096, device=DEV, generator=g)
    rng = np.random.default_rng(29)
    rew, n_done = 0.0, 0
    for t in range(30):
        out, r = _lockstep(eng, ost, rng.normal(0, 0.7, (n, 2)).astype(np.float32), t, "refill beside gemm")
        rew, n_done = max(rew, r), n_done + int(out["done"].sum())
        _refill(eng)
        for _ in range(4):
            a = torch.tanh(a @ a * (1.0 / 64))
    _final_state(eng, ost, "refill beside gemm 16384x20 30 steps", rew)
    print("refill beside gemm: %d episodes ended" % n_done)
    assert n_done > 0
    eng.close()
