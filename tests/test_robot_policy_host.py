"""CPU: the model-based robots (robot.policy = 'orca' / 'social_force').  The reference's step never asks a robot policy for
an action, so there is no reference fixture: the host restatement of the robot's action (tests/robot_oracle.py) is pinned
here against the RVO2 stand-in driven with ORCA.predict's call sequence (orca.py:85-136), against the C oracle's human
social-force branch (itself pinned on the reference's social-force step fixtures), against a numpy restatement of
SOCIAL_FORCE.predict (social_force.py:11-63) and against known answers.  The refusals need no GPU."""
import numpy as np
import pytest
import torch

from crowdnav_dsrnn_b200 import Config, abi
from crowdnav_dsrnn_b200.envs import CrowdVecEnv, make_vec_envs
from crowdnav_dsrnn_b200.evaluation import evaluate_batched
from crowdnav_dsrnn_b200.model import Policy
from crowdnav_dsrnn_b200.spaces import crowd_spaces
from crowdnav_dsrnn_b200.test import log_file_name
from oracle import crowd_oracle, state_sampler
import robot_oracle

PX, PY, VX, VY, RAD, GX, GY, VPREF = range(8)


def _state(H, n, seed, fov=2.0):
    c = Config(human_num=H)
    c.robot.FOV = fov
    cfg = abi.flatten_config(c, n, phase="train")
    inp = state_sampler.sample(cfg, n, seed=seed)
    st = crowd_oracle.OracleState(n, H)
    for f in ("robot", "humans", "belief", "extras", "counters"):
        getattr(st, f)[...] = inp[f]
    return cfg, st


def _rvo2_predict(cfg, self9, others5):
    """ORCA.predict (orca.py:85-136) on the RVO2 stand-in: a fresh simulator, the robot as agent 0, the others after it."""
    from oracle.refshim import rvo2

    params = (float(cfg.orca_neighbor_dist), len(others5), float(cfg.orca_time_horizon), float(cfg.orca_time_horizon))
    sim = rvo2.PyRVOSimulator(float(cfg.time_step), *params, 0.3, 1.0)
    s = [float(x) for x in self9]
    safety = float(cfg.orca_safety_space)
    sim.addAgent((s[PX], s[PY]), *params, s[RAD] + 0.01 + safety, s[VPREF], (s[VX], s[VY]))
    for o in others5:
        o = [float(x) for x in o]
        sim.addAgent((o[0], o[1]), *params, o[4] + 0.01 + safety, 1.0, (o[2], o[3]))
    velocity = np.array((s[GX] - s[PX], s[GY] - s[PY]))
    speed = np.linalg.norm(velocity)
    pref_vel = velocity / speed if speed > 1 else velocity
    sim.setAgentPrefVelocity(0, tuple(pref_vel))
    for i in range(len(others5)):
        sim.setAgentPrefVelocity(i + 1, (0, 0))
    sim.doStep()
    return np.array(sim.getAgentVelocity(0), np.float32)


def _social_force_np(cfg, self9, others5):
    """SOCIAL_FORCE.predict (social_force.py:11-63) in numpy float64."""
    s = self9.astype(np.float64)
    o = others5.astype(np.float64)
    dx, dy = s[GX] - s[PX], s[GY] - s[PY]
    dist_to_goal = np.sqrt(dx ** 2 + dy ** 2)
    desired_vx, desired_vy = (dx / dist_to_goal) * s[VPREF], (dy / dist_to_goal) * s[VPREF]
    curr_vx, curr_vy = cfg.sf_KI * (desired_vx - s[VX]), cfg.sf_KI * (desired_vy - s[VY])
    ivx = ivy = 0.0
    for k in range(len(o)):
        ddx, ddy = s[PX] - o[k, 0], s[PY] - o[k, 1]
        d = np.sqrt(ddx ** 2 + ddy ** 2)
        ivx += cfg.sf_A * np.exp((s[RAD] + o[k, 4] - d) / cfg.sf_B) * (ddx / d)
        ivy += cfg.sf_A * np.exp((s[RAD] + o[k, 4] - d) / cfg.sf_B) * (ddy / d)
    nvx = s[VX] + (curr_vx + ivx) * cfg.time_step
    nvy = s[VY] + (curr_vy + ivy) * cfg.time_step
    nrm = np.linalg.norm([nvx, nvy])
    if nrm > s[VPREF]:
        return np.array([nvx / nrm * s[VPREF], nvy / nrm * s[VPREF]], np.float32)
    return np.array([nvx, nvy], np.float32)


@pytest.mark.parametrize("H", [1, 5, 20])
def test_robot_social_force_is_the_oracle_human_social_force(H):
    """Human i of a social-force crowd (humans.policy = social_force, robot invisible to humans, full human FOV) sees the
    other humans in index order: one C-oracle step leaves its social-force action in its velocity.  The same self row and
    others through the robot's restatement must give the same float32 bits."""
    c = Config(human_num=H)
    c.humans.policy = "social_force"
    n = 64
    cfg = abi.flatten_config(c, n, phase="train")
    inp = state_sampler.sample(cfg, n, seed=120 + H)
    st = crowd_oracle.OracleState(n, H)
    for f in ("robot", "humans", "belief", "extras", "counters"):
        getattr(st, f)[...] = inp[f]
    pre = st.humans.copy()
    crowd_oracle.step(cfg, st, inp["action"], auto_reset=False)
    checked = 0
    for e in range(n):
        for i in range(H):
            others = np.concatenate([pre[e, :i, 0:5], pre[e, i + 1:, 0:5]])
            want = robot_oracle.social_force(cfg, pre[e, i], others)
            if not np.isfinite(want).all():
                continue
            assert np.array_equal(st.humans[e, i, 2:4].view(np.uint32), want.view(np.uint32)), (e, i)
            checked += 1
    assert checked > 0.8 * n * H


@pytest.mark.parametrize("H", [1, 5, 16])
def test_oracle_robot_orca_equals_the_rvo2_call_sequence_of_orca_predict(H):
    cfg, st = _state(H, 96, seed=70 + H)
    got = robot_oracle.robot_act(cfg, st, abi.POLICY_ORCA)
    for e in range(st.n):
        want = _rvo2_predict(cfg, st.robot[e], st.belief[e])
        assert np.array_equal(got[e].view(np.uint32), want.view(np.uint32)), (e, got[e], want)


@pytest.mark.parametrize("H", [1, 5, 20])
def test_oracle_robot_social_force_equals_numpy_restatement(H):
    cfg, st = _state(H, 128, seed=90 + H)
    got = robot_oracle.robot_act(cfg, st, "social_force")
    want = np.stack([_social_force_np(cfg, st.robot[e], st.belief[e]) for e in range(st.n)])
    ok = np.isfinite(want).all(axis=1)          # a robot standing exactly on its goal divides by zero, as the reference does
    assert ok.mean() > 0.9
    assert np.abs(got[ok].astype(np.float64) - want[ok]).max() <= 1e-6


def _one_env(robot, belief):
    c = Config(human_num=len(belief))
    cfg = abi.flatten_config(c, 1, phase="train")
    st = crowd_oracle.OracleState(1, len(belief))
    st.robot[0] = robot
    st.belief[0] = belief
    return cfg, st


def test_known_answers():
    far = [[30.0, 30.0, 0.0, 0.0, 0.3], [-25.0, 12.0, 0.5, 0.0, 0.3]]      # beyond orca.neighbor_dist = 10 m
    # no neighbour in range, goal within 1 m: the action is exactly the raw g - p
    cfg, st = _one_env([1.0, 2.0, 0.3, -0.2, 0.3, 1.5, 2.25, 1.0, 0.0], far)
    got = robot_oracle.robot_act(cfg, st, "orca")[0]
    want = np.array([np.float32(1.5 - 1.0), np.float32(2.25 - 2.0)], np.float32)
    assert np.array_equal(got, want)
    # no neighbour in range, goal far away: the preferred velocity (unit vector to the goal)
    cfg, st = _one_env([1.0, 2.0, 0.0, 0.0, 0.3, -3.0, 5.0, 1.0, 0.0], far)
    got = robot_oracle.robot_act(cfg, st, "orca")[0]
    d = np.array([-4.0, 3.0]) / 5.0
    assert np.abs(got - d).max() <= 1e-6
    # robot on its goal: zero
    cfg, st = _one_env([1.0, 2.0, 0.4, 0.1, 0.3, 1.0, 2.0, 1.0, 0.0], far)
    got = robot_oracle.robot_act(cfg, st, "orca")[0]
    assert np.array_equal(got, np.zeros(2, np.float32))


def test_unicycle_and_unknown_robot_policies_are_refused_before_any_cuda_work():
    for name in ("orca", "social_force"):
        c = Config(kinematics="unicycle")
        c.robot.policy = name
        with pytest.raises(NotImplementedError, match="holonomic"):
            abi.robot_policy_of(c)
        with pytest.raises(NotImplementedError):
            CrowdVecEnv(c, 4, "cpu")
        with pytest.raises(NotImplementedError):
            make_vec_envs("CrowdSimDict-v0", 0, 4, 0.99, None, "cpu", False, config=c)
    c = Config()
    c.robot.policy = "cadrl"
    with pytest.raises(NotImplementedError):
        abi.robot_policy_of(c)
    with pytest.raises(NotImplementedError):
        CrowdVecEnv(c, 4, "cpu")
    c.robot.policy = "srnn"
    assert abi.robot_policy_of(c) is None
    c.robot.policy = "orca"
    assert abi.robot_policy_of(c) == abi.POLICY_ORCA
    c.robot.policy = "social_force"
    assert abi.robot_policy_of(c) == abi.POLICY_SOCIAL_FORCE


def test_evaluate_batched_refuses_a_policy_for_a_model_based_robot():
    c = Config()
    obs, act = crowd_spaces(c.sim.human_num)
    policy = Policy(obs.spaces, act, base="srnn", base_kwargs=c)
    c.robot.policy = "orca"
    with pytest.raises(ValueError, match="actor_critic=None"):
        evaluate_batched(policy, c, "cpu")
    c.robot.policy = "srnn"
    with pytest.raises(ValueError):
        evaluate_batched(None, c, "cpu")
    with pytest.raises(NotImplementedError):
        Policy(obs.spaces, act, base="orca", base_kwargs=c)


def test_test_driver_names_the_log_after_the_robot_policy():
    assert log_file_name("orca", "test") == "model_orca_test_test_.log"
    assert log_file_name("social_force", "h20") == "model_social_force_test_h20_.log"
