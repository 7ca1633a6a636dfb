"""GPU: the model-based robots (robot.policy = 'orca' / 'social_force', kernel K8 behind cn_env_robot_act).
  * the kernel against the host restatement (tests/robot_oracle.py) on injected and rolled-out states: ORCA bit for bit, social force to 1e-6;
  * a vectorised env with a model-based robot steps exactly like an 'srnn' env fed with CrowdEngine.robot_act, and
    tracks the oracle's rollout;
  * robot_act + step captured in a CUDA graph replay the eager calls;
  * evaluate_batched(None, cfg) and `python -m crowdnav_dsrnn_b200.test --robot_policy ...`."""
import json

import numpy as np
import pytest
import torch

from crowdnav_dsrnn_b200 import Config
from crowdnav_dsrnn_b200 import test as test_cli
from crowdnav_dsrnn_b200.envs import CrowdVecEnv, make_vec_envs
from crowdnav_dsrnn_b200.evaluation import evaluate_batched
from oracle import crowd_oracle, state_sampler
import gpu_helpers as G
import robot_oracle

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
HS = [1, 2, 5, 10, 16, 17, 20, 31]           # group widths 4, 4, 8, 16, 16, 32, 32, 32


def _cfg(H, fov=2.0, policy="srnn"):
    c = Config(human_num=H)
    c.robot.FOV = fov
    c.robot.policy = policy
    return c


def _oracle_state(st, n, H):
    ost = crowd_oracle.OracleState(n, H)
    for f, v in G.state_to_numpy(st).items():
        getattr(ost, f)[...] = v
    return ost


def _check(eng, n, H, policy):
    got = eng.robot_act(policy).cpu().numpy()
    want = robot_oracle.robot_act(eng.cfg, _oracle_state(eng.get_state(), n, H), policy)
    if policy == "orca":
        bad = got.view(np.uint32) != want.view(np.uint32)
        assert not bad.any(), "%d of %d envs differ, first %s" % (bad.any(axis=1).sum(), n, np.argwhere(bad)[:3].tolist())
    else:
        ok = np.isfinite(want).all(axis=1)
        assert np.array_equal(np.isfinite(got).all(axis=1), ok)
        assert np.abs(got[ok].astype(np.float64) - want[ok]).max() <= 1e-6


@pytest.mark.parametrize("policy", ["orca", "social_force"])
@pytest.mark.parametrize("fov", [2.0, 0.5])
@pytest.mark.parametrize("H", HS)
def test_robot_act_matches_oracle_on_rolled_out_beliefs(H, fov, policy):
    """Beliefs after a reset and a few steps: with FOV 0.5 some rows are parked at (15, 15) or dead-reckoned."""
    n = 1024
    eng = G.make_engine(_cfg(H, fov), n, seed=17 + H)
    eng.reset()
    _check(eng, n, H, policy)
    for _ in range(4):
        eng.step(eng.robot_act(policy), auto_reset=True)
        _check(eng, n, H, policy)
    if fov < 2.0:
        bel = eng.get_state()["belief"].cpu().numpy()
        assert (bel[:, :, 0] == 15.0).any()


@pytest.mark.parametrize("policy", ["orca", "social_force"])
@pytest.mark.parametrize("H", HS)
def test_robot_act_matches_oracle_on_injected_states(H, policy):
    """The state sampler's branches (robot overlapping a human, far rows, zero velocities), then the same envs with the
    robot surrounded by its belief rows within 1.2 m, so that linearProgram2 fails and linearProgram3 runs."""
    n = 2048
    eng = G.make_engine(_cfg(H), n)
    inp = state_sampler.sample(eng.cfg, n, seed=300 + H)
    inp.pop("action")
    inp["belief"][:, 0, 0:2] = inp["robot"][:, 0:2] + np.float32(0.2)          # every robot overlaps belief row 0
    eng.set_state(**inp)
    _check(eng, n, H, policy)
    rng = np.random.default_rng(H)
    dense = inp["belief"].copy()
    r = rng.uniform(0.3, 1.2, (n, H))
    a = rng.uniform(0, 2 * np.pi, (n, H))
    dense[:, :, 0] = inp["robot"][:, None, 0] + r * np.cos(a)
    dense[:, :, 1] = inp["robot"][:, None, 1] + r * np.sin(a)
    dense[:, :, 2:4] = -0.5 * np.stack([np.cos(a), np.sin(a)], -1)           # walking towards the robot
    inp["belief"] = np.ascontiguousarray(dense, np.float32)
    eng.set_state(**inp)
    _check(eng, n, H, policy)


def _run(venv, steps, feed):
    venv.reset()
    trace = []
    for _ in range(steps):
        _, _, _, buf = venv.step_device(feed(venv))
        trace.append(G.buf_to_numpy(buf))
    return trace, G.state_to_numpy(venv.engine.get_state())


@pytest.mark.parametrize("policy", ["orca", "social_force"])
def test_model_based_env_equals_srnn_env_fed_with_robot_act(policy):
    n, H, steps = 512, 10, 200
    a = CrowdVecEnv(_cfg(H, 0.5, policy), n, DEV, seed=4, phase="train")
    b = CrowdVecEnv(_cfg(H, 0.5, "srnn"), n, DEV, seed=4, phase="train")
    ta, sa = _run(a, steps, lambda v: None)
    tb, sb = _run(b, steps, lambda v: v.engine.robot_act(policy))
    for t, (x, y) in enumerate(zip(ta, tb)):
        for f in G.OUT_FIELDS:
            assert np.array_equal(x[f], y[f]), "step %d %s" % (t, f)
    for f in G.STATE_FIELDS:
        assert np.array_equal(sa[f], sb[f]), f
    assert sum(int(x["done"].sum()) for x in ta) > n          # auto-resets happened
    a.close()
    b.close()


def test_model_based_rollout_tracks_oracle():
    n, H, steps = 512, 5, 100
    eng = G.make_engine(_cfg(H, 0.5), n, seed=3)
    cfg = eng.cfg
    eng.reset()
    ost = crowd_oracle.OracleState(n, H)
    crowd_oracle.reset(cfg, ost, n_threads=8)
    n_done = 0
    for t in range(steps):
        act = eng.robot_act("orca")
        oact = robot_oracle.robot_act(cfg, ost, "orca")
        assert np.abs(act.cpu().numpy() - oact).max() <= 1e-4, "step %d" % t
        buf = eng.step(act, auto_reset=True)
        oout = crowd_oracle.step(cfg, ost, oact, auto_reset=True, n_threads=8)
        out = G.buf_to_numpy(buf)
        for f in ("done", "event", "visible_mask", "goal_changed"):
            assert np.array_equal(out[f], G.oracle_out_to_numpy(oout)[f]), "step %d %s" % (t, f)
        assert np.abs(out["reward"] - oout.reward).max() <= 1e-5
        n_done += int(out["done"].sum())
    st = G.state_to_numpy(eng.get_state())
    assert np.abs(st["humans"] - ost.humans).max() <= 1e-4
    assert np.abs(st["robot"] - ost.robot).max() <= 1e-4
    assert np.abs(st["belief"] - ost.belief).max() <= 1e-4
    assert n_done > 0


def test_robot_act_and_step_replay_in_a_cuda_graph():
    n, H, steps = 1024, 5, 40
    cfg = _cfg(H, 0.5, "orca")
    va = CrowdVecEnv(cfg, n, DEV, seed=8, phase="train")
    trace, st_e = _run(va, steps, lambda v: None)
    va.close()

    vb = CrowdVecEnv(cfg, n, DEV, seed=8, phase="train")
    vb.reset()
    eng = vb.engine
    action = torch.empty(n, 2, device=DEV)

    def one_step():
        eng.robot_act("orca", out=action)
        eng.step(action, auto_reset=True)
        eng.join()

    side = torch.cuda.Stream(device=DEV)
    side.wait_stream(torch.cuda.current_stream(DEV))
    with torch.cuda.stream(side):
        one_step()                                    # two eager warm-up steps, one per output buffer
        one_step()
    torch.cuda.current_stream(DEV).wait_stream(side)
    torch.cuda.synchronize(DEV)
    graphs = []
    for _ in range(2):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            one_step()                                # flips eng.cur: the two graphs write the two buffers in turn
        graphs.append(g)
    for t in range(2, steps):
        graphs[t % 2].replay()
        eng.cur ^= 1
    torch.cuda.synchronize(DEV)
    out = G.buf_to_numpy(eng.bufs[eng.cur])
    for f in G.OUT_FIELDS:
        assert np.array_equal(out[f], trace[-1][f]), f
    st_g = G.state_to_numpy(eng.get_state())
    for f in G.STATE_FIELDS:
        assert np.array_equal(st_g[f], st_e[f]), f
    vb.close()


@pytest.mark.parametrize("policy", ["orca", "social_force"])
def test_evaluate_batched_model_based_robot(policy):
    cfg = _cfg(5, 2.0, policy)
    r1 = evaluate_batched(None, cfg, DEV, episodes=2000)
    r2 = evaluate_batched(None, cfg, DEV, episodes=2000)
    print(policy, {k: r1[k] for k in ("success", "collision", "timeout", "mean_nav_time_success", "mean_path_length")})
    assert r1["unfinished"] == 0
    assert abs(r1["success"] + r1["collision"] + r1["timeout"] - 1.0) < 1e-6          # float32 means
    assert json.dumps(r1, sort_keys=True) == json.dumps(r2, sort_keys=True)
    assert r1["success"] > 0.3                                # the robot does walk to its goal
    assert {"episodes", "success", "collision", "timeout", "unfinished", "mean_steps", "mean_nav_time_success",
            "mean_path_length", "mean_return", "per_scenario", "side_left_episodes"} <= set(r1)


def test_test_driver_runs_a_model_based_robot(tmp_path, monkeypatch):
    (tmp_path / "data" / "m").mkdir(parents=True)
    monkeypatch.chdir(tmp_path)
    assert test_cli.main(["--model_dir", "data/m", "--robot_policy", "orca", "--test_name", "cli"]) == 0
    log = (tmp_path / "data" / "m" / "test" / "model_orca_test_cli_.log").read_text()
    for must in ("Using robot policy orca", "robot FOV", "humans FOV", "success rate: ", "collision rate: ", "timeout rate: ",
                 "SCENARIO BREAKDOWN: ", "navigation time ======", "path length ======"):
        assert must in log, must
    assert "Using model" not in log
    envs = make_vec_envs("CrowdSimDict-v0", 0, 2, 0.99, None, DEV, False, config=_cfg(5, 2.0, "social_force"))
    envs.reset()
    obs, reward, done, infos = envs.step(None)
    assert reward.shape == (2, 1) and len(infos) == 2
    envs.close()
