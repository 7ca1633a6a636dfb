"""ctypes mirror of include/crowdnav_b200.h and the Config -> CnConfig flattening.

`flatten_config` reads the attribute tree of crowd_nav/configs/config.py:9-214
(the reference's `Config`, or this package's restatement of it) exactly where
CrowdSim.configure (crowd_sim/envs/crowd_sim.py:93-246) and Agent.__init__
(crowd_sim/envs/utils/agent.py:16-35) read it.
"""
import ctypes as C
import math

ABI_VERSION = 3
MAX_HUMANS = 32
MAX_SCENARIOS = 8
MAX_GROUPS = 8
STEP_TABLE_WORDS = 128
INFO_DIM = 12

HOLONOMIC, UNICYCLE = 0, 1
POLICY_ORCA, POLICY_SOCIAL_FORCE = 0, 1
HUMAN_POLICIES = {"orca": POLICY_ORCA, "social_force": POLICY_SOCIAL_FORCE}
# model-based robots (robot.policy, policy_factory.py:12-17): their action comes from cn_env_robot_act
ROBOT_POLICIES = {"orca": POLICY_ORCA, "social_force": POLICY_SOCIAL_FORCE}
PHASE_TRAIN, PHASE_VAL, PHASE_TEST = 0, 1, 2
PHASES = {"train": PHASE_TRAIN, "val": PHASE_VAL, "test": PHASE_TEST}
EV_NOTHING, EV_DANGER, EV_REACH_GOAL, EV_COLLISION, EV_TIMEOUT = 0, 1, 2, 3, 4
SCENARIOS = [
    "circle_crossing", "square_crossing", "parallel_traffic", "perpendicular_traffic",
    "side_pref_passing", "side_pref_overtaking", "side_pref_crossing",
]
SCENARIO_ID = {s: i for i, s in enumerate(SCENARIOS)}
INFO_COLUMNS = {
    "dmin": 0, "aggregate_nav_time": 1, "path_violation": 2, "personal_violation": 3, "jerk_cost": 4,
    "dist_to_goal": 5, "speed_violation": 6, "side_left": 7, "side_right": 8, "separation": 9,
}
PREC_FP32, PREC_BF16X3, PREC_BF16, PREC_FP16 = 0, 1, 2, 3
PRECISIONS = {"fp32": PREC_FP32, "bf16x3": PREC_BF16X3, "bf16": PREC_BF16, "fp16": PREC_FP16}
# cn_env_render: palette (0xRRGGBB), marker sizes (metres / radians) and the accepted frame sizes (CN_RENDER_*)
RENDER_RGB = {"background": 0xFFFFFF, "fov": 0xDCE9F7, "goal": 0xD62728, "human_in": 0x2CA02C, "human_out": 0x9E9E9E,
              "robot": 0xFFC20E, "heading": 0x8C5A00, "invalid": 0xFF00FF}
RENDER_GOAL_RADIUS = 0.15
RENDER_HEADING_HALF = 0.5
RENDER_MIN_SIZE, RENDER_MAX_SIZE, RENDER_SIZE_MULTIPLE = 32, 2048, 16


class CnConfig(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("human_num", C.c_int32), ("kinematics", C.c_int32),
        ("robot_visible", C.c_int32), ("randomize_attributes", C.c_int32), ("potential_based", C.c_int32),
        ("exponential", C.c_int32), ("time_factor", C.c_int32), ("random_goal_changing", C.c_int32),
        ("end_goal_changing", C.c_int32), ("side_preference", C.c_int32), ("social_metrics", C.c_int32),
        ("phase", C.c_int32), ("nenv", C.c_int32), ("n_scenarios", C.c_int32),
        ("scenarios", C.c_int32 * MAX_SCENARIOS),
        ("max_spawn_tries", C.c_int32), ("max_goal_tries", C.c_int32), ("max_robot_tries", C.c_int32),
        ("timeout_step", C.c_int32), ("env_id_offset", C.c_int32), ("reserved0", C.c_int32),
        ("goal_change_steps", C.c_uint32 * STEP_TABLE_WORDS),
        ("base_seed", C.c_uint64), ("seed_offset", C.c_uint64), ("case_size", C.c_uint64),
        ("time_step", C.c_double), ("time_limit", C.c_double), ("success_reward", C.c_double),
        ("collision_penalty", C.c_double), ("discomfort_dist", C.c_double),
        ("discomfort_penalty_factor", C.c_double), ("potential_factor", C.c_double), ("exp_factor", C.c_double),
        ("exp_denom", C.c_double), ("circle_radius", C.c_double), ("square_width", C.c_double),
        ("robot_fov", C.c_double), ("human_fov", C.c_double), ("robot_radius", C.c_double),
        ("robot_v_pref", C.c_double), ("human_radius", C.c_double), ("human_v_pref", C.c_double),
        ("min_personal_space", C.c_double), ("max_walking_speed", C.c_double),
        ("goal_change_chance", C.c_double), ("end_goal_change_chance", C.c_double),
        ("orca_neighbor_dist", C.c_float), ("orca_safety_space", C.c_float), ("orca_time_horizon", C.c_float),
        ("reserved1", C.c_float),
        ("human_policy", C.c_int32), ("random_policy_changing", C.c_int32), ("random_unobservability", C.c_int32),
        ("random_radii", C.c_int32), ("random_v_pref", C.c_int32), ("group_human", C.c_int32),
        ("unobservable_chance", C.c_double), ("sf_A", C.c_double), ("sf_B", C.c_double), ("sf_KI", C.c_double),
    ]


_fp = C.c_void_p


class CnStateView(C.Structure):
    _fields_ = [("robot", _fp), ("humans", _fp), ("belief", _fp), ("extras", _fp), ("counters", _fp),
                ("episode_return", _fp), ("groups", _fp)]


class CnObsOut(C.Structure):
    _fields_ = [("robot_node", _fp), ("temporal_edges", _fp), ("spatial_edges", _fp), ("visible_mask", _fp)]


class CnStepOut(C.Structure):
    _fields_ = [("obs", CnObsOut), ("reward", _fp), ("done", _fp), ("event", _fp), ("scenario", _fp),
                ("info", _fp), ("episode_return", _fp), ("episode_length", _fp), ("goal_changed", _fp),
                ("not_done", _fp)]


DSRNN_WEIGHT_FIELDS = [
    "t_enc_w", "t_enc_b", "t_w_ih", "t_w_hh", "t_b_ih", "t_b_hh",
    "s_enc_w", "s_enc_b", "s_w_ih", "s_w_hh", "s_b_ih", "s_b_hh",
    "att_t_w", "att_t_b", "att_s_w", "att_s_b",
    "robot_w", "robot_b",
    "n_enc_w", "n_enc_b", "n_att_w", "n_att_b", "n_w_ih", "n_w_hh", "n_b_ih", "n_b_hh", "n_out_w", "n_out_b",
    "actor0_w", "actor0_b", "actor2_w", "actor2_b",
    "critic0_w", "critic0_b", "critic2_w", "critic2_b",
    "critic_lin_w", "critic_lin_b", "mean_w", "mean_b",
]

# CnDsrnnWeights member -> key of the reference Policy.state_dict() (model.py:17-104; SURVEY 8(b))
DSRNN_STATE_DICT_KEYS = {
    "t_enc_w": "base.humanhumanEdgeRNN_temporal.encoder_linear.weight",
    "t_enc_b": "base.humanhumanEdgeRNN_temporal.encoder_linear.bias",
    "t_w_ih": "base.humanhumanEdgeRNN_temporal.gru.weight_ih_l0",
    "t_w_hh": "base.humanhumanEdgeRNN_temporal.gru.weight_hh_l0",
    "t_b_ih": "base.humanhumanEdgeRNN_temporal.gru.bias_ih_l0",
    "t_b_hh": "base.humanhumanEdgeRNN_temporal.gru.bias_hh_l0",
    "s_enc_w": "base.humanhumanEdgeRNN_spatial.encoder_linear.weight",
    "s_enc_b": "base.humanhumanEdgeRNN_spatial.encoder_linear.bias",
    "s_w_ih": "base.humanhumanEdgeRNN_spatial.gru.weight_ih_l0",
    "s_w_hh": "base.humanhumanEdgeRNN_spatial.gru.weight_hh_l0",
    "s_b_ih": "base.humanhumanEdgeRNN_spatial.gru.bias_ih_l0",
    "s_b_hh": "base.humanhumanEdgeRNN_spatial.gru.bias_hh_l0",
    "att_t_w": "base.attn.temporal_edge_layer.0.weight",
    "att_t_b": "base.attn.temporal_edge_layer.0.bias",
    "att_s_w": "base.attn.spatial_edge_layer.0.weight",
    "att_s_b": "base.attn.spatial_edge_layer.0.bias",
    "robot_w": "base.robot_linear.weight",
    "robot_b": "base.robot_linear.bias",
    "n_enc_w": "base.humanNodeRNN.encoder_linear.weight",
    "n_enc_b": "base.humanNodeRNN.encoder_linear.bias",
    "n_att_w": "base.humanNodeRNN.edge_attention_embed.weight",
    "n_att_b": "base.humanNodeRNN.edge_attention_embed.bias",
    "n_w_ih": "base.humanNodeRNN.gru.weight_ih_l0",
    "n_w_hh": "base.humanNodeRNN.gru.weight_hh_l0",
    "n_b_ih": "base.humanNodeRNN.gru.bias_ih_l0",
    "n_b_hh": "base.humanNodeRNN.gru.bias_hh_l0",
    "n_out_w": "base.humanNodeRNN.output_linear.weight",
    "n_out_b": "base.humanNodeRNN.output_linear.bias",
    "actor0_w": "base.actor.0.weight", "actor0_b": "base.actor.0.bias",
    "actor2_w": "base.actor.2.weight", "actor2_b": "base.actor.2.bias",
    "critic0_w": "base.critic.0.weight", "critic0_b": "base.critic.0.bias",
    "critic2_w": "base.critic.2.weight", "critic2_b": "base.critic.2.bias",
    "critic_lin_w": "base.critic_linear.weight", "critic_lin_b": "base.critic_linear.bias",
    "mean_w": "dist.fc_mean.weight", "mean_b": "dist.fc_mean.bias",
}


class CnDsrnnWeights(C.Structure):
    _fields_ = [(name, _fp) for name in DSRNN_WEIGHT_FIELDS]


class CnDsrnnIO(C.Structure):
    _fields_ = [(name, _fp) for name in (
        "robot_node", "temporal_edges", "spatial_edges", "h_node_in", "h_edge_in", "masks",
        "h_node_out", "h_edge_out", "value", "action_mean", "actor_features")]


class CnEdgeSeqStep(C.Structure):
    _fields_ = [("temporal_edges", _fp), ("spatial_edges", _fp), ("masks", _fp), ("h_in", _fp),
                ("in_row_spatial", C.c_longlong), ("in_row_temporal", C.c_longlong),
                ("out_row_spatial", C.c_longlong), ("out_row_temporal", C.c_longlong),
                ("h_out", _fp), ("ws", _fp), ("hm_hi", _fp), ("hm_lo", _fp), ("e_hi", _fp), ("e_lo", _fp)]


GEMM_MAX_PROBLEMS = 4


class CnGemmOperand(C.Structure):
    _fields_ = [("hi", _fp), ("lo", _fp), ("ld", C.c_longlong), ("mn_major", C.c_int), ("reserved", C.c_int)]


class CnGemm(C.Structure):
    _fields_ = [("a", CnGemmOperand), ("b", CnGemmOperand), ("c", _fp), ("ldc", C.c_longlong), ("bias", _fp),
                ("m", C.c_int), ("n", C.c_int), ("k", C.c_int), ("act", C.c_int), ("accumulate", C.c_int), ("split_k", C.c_int)]


def step_tables(time_step, time_limit):
    """Replay the reference's float64 `global_time += time_step` accumulation
    (crowd_sim_dict.py:253) and return (timeout_step, goal_change_bits):

    * timeout_step: first step index s whose calc_reward sees
      `global_time >= time_limit - 1` (crowd_sim.py:1032);
    * goal_change_bits[s] set iff after s steps `global_time % 5 == 0`
      (crowd_sim_dict.py:262).
    """
    words = [0] * STEP_TABLE_WORDS
    t = 0  # `self.global_time = 0` (int) at reset, then `+= time_step`
    timeout_step = None
    for s in range(32 * STEP_TABLE_WORDS - 1):
        if t >= time_limit - 1:
            timeout_step = s
        t += time_step
        if t % 5 == 0:
            words[(s + 1) >> 5] |= 1 << ((s + 1) & 31)
        if timeout_step is not None:  # the terminal step still runs its goal update before the reset
            break
    if timeout_step is None:
        raise ValueError("episode longer than %d steps is not supported" % (32 * STEP_TABLE_WORDS))
    return timeout_step, words


def robot_policy_of(config):
    """The CN_POLICY_* of a model-based robot (robot.policy = 'orca' / 'social_force'), None for the learned 'srnn' robot.
    Raises NotImplementedError for any other name, and for a model-based robot with unicycle kinematics."""
    name = config.robot.policy
    if name == "srnn":
        return None
    if name not in ROBOT_POLICIES:
        raise NotImplementedError("robot.policy=%r (the vectorised env runs 'srnn', 'orca' and 'social_force')" % (name,))
    if config.action_space.kinematics != "holonomic":
        raise NotImplementedError("robot.policy=%r outputs velocities: it needs action_space.kinematics='holonomic', not %r"
                                  % (name, config.action_space.kinematics))
    return ROBOT_POLICIES[name]


def flatten_config(config, n_envs, phase=None, seed=None, env_id_offset=0, nenv=None,
                   max_spawn_tries=1024, max_goal_tries=32, max_robot_tries=256):
    """Build the CnConfig the C ABI consumes from a reference-shaped Config object."""
    c = CnConfig()
    c.abi_version = ABI_VERSION
    if config.humans.policy not in HUMAN_POLICIES:      # crowd_sim.py:106-127 raises for anything else too
        raise NotImplementedError("humans.policy=%r (the reference's humans are 'orca' or 'social_force')" % (config.humans.policy,))
    # optional human behaviours (SURVEY 8(f) N4)
    c.human_policy = HUMAN_POLICIES[config.humans.policy]
    c.random_policy_changing = int(bool(getattr(config.humans, "random_policy_changing", False)))
    c.random_unobservability = int(bool(getattr(config.humans, "random_unobservability", False)))
    c.random_radii = int(bool(getattr(config.humans, "random_radii", False)))
    c.random_v_pref = int(bool(getattr(config.humans, "random_v_pref", False)))
    c.group_human = int(bool(getattr(config.sim, "group_human", False)) and not config.test.side_preference)   # crowd_sim.py:123-125
    c.unobservable_chance = float(getattr(config.humans, "unobservable_chance", 0.3))
    sf = getattr(config, "sf", None)
    c.sf_A = float(getattr(sf, "A", 2.0))
    c.sf_B = float(getattr(sf, "B", 1.0))
    c.sf_KI = float(getattr(sf, "KI", 1.0))
    # noise.add_noise is accepted and has no effect, exactly as in the reference: only the base CrowdSim.generate_ob applies
    # apply_noise (crowd_sim.py:1115-1116); CrowdSimDict overrides generate_ob without it (crowd_sim_dict.py:71-103)
    if getattr(config.reward, "norm_zones", False):
        raise NotImplementedError("reward.norm_zones is degenerate in the reference (DESIGN.md section 4) and not reproduced")
    if getattr(config.lidar, "enable", False):
        raise NotImplementedError("lidar is out of scope (SURVEY section 2 row 18)")
    c.human_num = int(config.sim.human_num)
    kin = config.action_space.kinematics
    if kin not in ("holonomic", "unicycle"):
        raise ValueError("unknown kinematics %r" % (kin,))
    c.kinematics = HOLONOMIC if kin == "holonomic" else UNICYCLE
    c.robot_visible = int(bool(config.robot.visible))
    if c.human_num < 1 or c.human_num + c.robot_visible > MAX_HUMANS:
        raise ValueError("human_num must be in 1..%d" % (MAX_HUMANS - c.robot_visible))
    c.randomize_attributes = int(bool(config.env.randomize_attributes))
    c.potential_based = int(bool(config.reward.potential_based))
    c.exponential = int(bool(config.reward.exponential))
    c.time_factor = int(bool(config.reward.time_factor))
    c.random_goal_changing = int(bool(config.humans.random_goal_changing))
    c.end_goal_changing = int(bool(config.humans.end_goal_changing))
    c.side_preference = int(bool(config.test.side_preference))
    c.social_metrics = int(bool(config.test.social_metrics))
    if phase is None:  # envs.py:70-73
        phase = "train" if n_envs > 1 else "test"
    c.phase = PHASES[phase]
    c.nenv = int(n_envs if nenv is None else nenv)
    scen = config.sim.test_sim if phase == "test" else config.sim.train_val_sim
    if isinstance(scen, str):  # crowd_sim.py:138-142
        raise TypeError("config.sim.train_val_sim or config.sim.test_sim should be a list of strings. "
                        "Update your config.py")
    if not 1 <= len(scen) <= MAX_SCENARIOS:
        raise ValueError("scenario list must have 1..%d entries" % MAX_SCENARIOS)
    if c.social_metrics:
        assert len(scen) == 4  # crowd_sim_dict.py:116
    c.n_scenarios = len(scen)
    for i, s in enumerate(scen):
        c.scenarios[i] = SCENARIO_ID[s]
    c.max_spawn_tries, c.max_goal_tries, c.max_robot_tries = max_spawn_tries, max_goal_tries, max_robot_tries
    timeout_step, words = step_tables(config.env.time_step, config.env.time_limit)
    c.timeout_step = timeout_step
    for i, w in enumerate(words):
        c.goal_change_steps[i] = w
    c.env_id_offset = int(env_id_offset)
    c.base_seed = int(config.env.seed if seed is None else seed)
    val_cap, test_cap = 1000, 1000  # case_capacity, crowd_sim.py:110-114
    c.seed_offset = {"train": val_cap + test_cap, "val": 0, "test": val_cap}[phase]
    c.case_size = {"train": 2 ** 32 - 1 - 2000, "val": int(config.env.val_size),
                   "test": int(config.env.test_size)}[phase]
    c.time_step = float(config.env.time_step)
    c.time_limit = float(config.env.time_limit)
    c.success_reward = float(config.reward.success_reward)
    c.collision_penalty = float(config.reward.collision_penalty)
    c.discomfort_dist = float(config.reward.discomfort_dist_back)
    c.discomfort_penalty_factor = float(config.reward.discomfort_penalty_factor)
    c.potential_factor = float(config.reward.potential_factor)
    c.exp_factor = float(config.reward.exp_factor)
    c.exp_denom = float(config.reward.exp_denom)
    c.circle_radius = float(config.sim.circle_radius)
    c.square_width = float(config.sim.square_width)
    c.robot_fov = math.pi * config.robot.FOV
    c.human_fov = math.pi * config.humans.FOV
    c.robot_radius = float(config.robot.radius)
    c.robot_v_pref = float(config.robot.v_pref)
    c.human_radius = float(config.humans.radius)
    c.human_v_pref = float(config.humans.v_pref)
    c.min_personal_space = float(config.social.min_personal_space)
    c.max_walking_speed = float(config.social.max_walking_speed)
    c.goal_change_chance = float(config.humans.goal_change_chance)
    c.end_goal_change_chance = float(config.humans.end_goal_change_chance)
    c.orca_neighbor_dist = float(config.orca.neighbor_dist)
    c.orca_safety_space = float(config.orca.safety_space)
    c.orca_time_horizon = float(config.orca.time_horizon)
    return c
