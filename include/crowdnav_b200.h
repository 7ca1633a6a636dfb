/*
 * crowdnav_b200.h -- C ABI of libcrowdnav_b200.so (B200 / sm_100a).
 *
 * Drop-in boundary for the rollout hot path of evan-tan/CrowdNav_DSRNN:
 *   crowd step  (CrowdSimDict.step,  crowd_sim/envs/crowd_sim_dict.py:205-271)
 *   reset       (CrowdSimDict.reset, crowd_sim/envs/crowd_sim_dict.py:105-203)
 *   DS-RNN fwd  (SRNN.forward,       pytorchBaselines/a2c_ppo_acktr/srnn_model.py:409-504)
 *
 * The reference has no FFI of its own for this path except the third-party
 * `rvo2` module (crowd_nav/policy/orca.py:87-136); the functions below are what
 * a binding for the whole batched path replaces it with.  Plain pointers and
 * sizes only; no torch types.  All pointers named *_dev are DEVICE pointers
 * owned by the caller.  Every call is asynchronous on `stream` (a
 * cudaStream_t passed as void*).  Every function returns CN_OK or a negative
 * error code; cn_last_error() returns the text for the calling thread.
 */
#ifndef CROWDNAV_B200_H
#define CROWDNAV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CN_ABI_VERSION 3
#define CN_MAX_HUMANS 32          /* one 32-lane group per ORCA solve */
#define CN_MAX_SCENARIOS 8
#define CN_MAX_GROUPS 8            /* circle groups per episode: every group takes at least 4 of the <= 32 humans */
#define CN_STEP_TABLE_WORDS 128   /* bit table over step indices: up to 4096 steps per episode */

enum { CN_OK = 0, CN_ERR_ARG = -1, CN_ERR_CUDA = -2, CN_ERR_UNSUPPORTED = -3, CN_ERR_STATE = -4 };

/* config.action_space.kinematics (crowd_nav/configs/config.py:136-138) */
enum { CN_HOLONOMIC = 0, CN_UNICYCLE = 1 };
/* scenario strings of config.sim.train_val_sim / test_sim (config.py:17-35; crowd_sim.py:306-354) */
enum {
    CN_SCN_CIRCLE_CROSSING = 0, CN_SCN_SQUARE_CROSSING = 1, CN_SCN_PARALLEL_TRAFFIC = 2,
    CN_SCN_PERPENDICULAR_TRAFFIC = 3, CN_SCN_SIDE_PREF_PASSING = 4, CN_SCN_SIDE_PREF_OVERTAKING = 5,
    CN_SCN_SIDE_PREF_CROSSING = 6
};
/* config.humans.policy (crowd_nav/policy/policy_factory.py): the humans' reactive policy */
enum { CN_POLICY_ORCA = 0, CN_POLICY_SOCIAL_FORCE = 1 };
/* event classes of crowd_sim/envs/utils/info.py:1-38 */
enum { CN_EV_NOTHING = 0, CN_EV_DANGER = 1, CN_EV_REACH_GOAL = 2, CN_EV_COLLISION = 3, CN_EV_TIMEOUT = 4 };
/* env.phase (pytorchBaselines/a2c_ppo_acktr/envs.py:70-73) */
enum { CN_PHASE_TRAIN = 0, CN_PHASE_VAL = 1, CN_PHASE_TEST = 2 };

/*
 * Flattened crowd_nav/configs/config.py (consumed by CrowdSim.configure,
 * crowd_sim/envs/crowd_sim.py:93-246, and Agent.__init__, utils/agent.py:16-35).
 * Doubles where the reference holds Python floats.
 */
typedef struct CnConfig {
    int32_t abi_version;              /* CN_ABI_VERSION */
    int32_t human_num;                /* sim.human_num, 1..CN_MAX_HUMANS */
    int32_t kinematics;               /* CN_HOLONOMIC / CN_UNICYCLE */
    int32_t robot_visible;            /* robot.visible: humans' ORCA sees the robot */
    int32_t randomize_attributes;     /* env.randomize_attributes */
    int32_t potential_based;          /* reward.potential_based */
    int32_t exponential;              /* reward.exponential */
    int32_t time_factor;              /* reward.time_factor */
    int32_t random_goal_changing;     /* humans.random_goal_changing */
    int32_t end_goal_changing;        /* humans.end_goal_changing */
    int32_t side_preference;          /* test.side_preference */
    int32_t social_metrics;           /* test.social_metrics */
    int32_t phase;                    /* CN_PHASE_* (selects scenario list, seed offset, case size) */
    int32_t nenv;                     /* env.nenv: case_counter stride (crowd_sim_dict.py:162-164) */
    int32_t n_scenarios;              /* length of the active scenario list */
    int32_t scenarios[CN_MAX_SCENARIOS];
    int32_t max_spawn_tries;          /* bounded rejection (DESIGN.md: deviation from the unbounded loops) */
    int32_t max_goal_tries;
    int32_t max_robot_tries;
    int32_t timeout_step;             /* first step index whose float64-accumulated global_time >= time_limit-1 */
    int32_t env_id_offset;            /* global id of local env 0 (multi-GPU sharding; RNG is keyed by global id) */
    int32_t reserved0;
    uint32_t goal_change_steps[CN_STEP_TABLE_WORDS]; /* bit s set: after s steps global_time % 5 == 0 (crowd_sim_dict.py:262) */
    uint64_t base_seed;               /* env.seed (thisSeed = base_seed + global env id, envs.py:66-68) */
    uint64_t seed_offset;             /* counter_offset[phase] (crowd_sim_dict.py:147-151) */
    uint64_t case_size;               /* case_size[phase] (crowd_sim.py:115-119) */
    double time_step;                 /* env.time_step */
    double time_limit;                /* env.time_limit */
    double success_reward;
    double collision_penalty;
    double discomfort_dist;           /* reward.discomfort_dist_back */
    double discomfort_penalty_factor; /* already multiplied by time_step (config.py:73-74) */
    double potential_factor;
    double exp_factor;
    double exp_denom;
    double circle_radius;
    double square_width;
    double robot_fov;                 /* radians = pi * robot.FOV */
    double human_fov;                 /* radians = pi * humans.FOV */
    double robot_radius;
    double robot_v_pref;
    double human_radius;              /* used when !randomize_attributes and for the dummy human */
    double human_v_pref;
    double min_personal_space;        /* social.min_personal_space */
    double max_walking_speed;         /* social.max_walking_speed */
    double goal_change_chance;
    double end_goal_change_chance;
    float orca_neighbor_dist;         /* orca.* are narrowed to float at the rvo2 boundary */
    float orca_safety_space;
    float orca_time_horizon;
    float reserved1;
    /* --- optional human behaviours (SURVEY 8(f) N4; all off in the reference's default config) --- */
    int32_t human_policy;             /* humans.policy: CN_POLICY_ORCA / CN_POLICY_SOCIAL_FORCE */
    int32_t random_policy_changing;   /* humans.random_policy_changing: each human is ORCA or social force, drawn per episode
                                         (crowd_sim.py:463-473, crowd_sim_dict.py:157-159) */
    int32_t random_unobservability;   /* humans.random_unobservability: human 0 misses each neighbour with unobservable_chance
                                         at every step (crowd_sim.py:1121-1153) */
    int32_t random_radii;             /* humans.random_radii / random_v_pref: radius / v_pref += U(-0.1, 0.1) whenever a human */
    int32_t random_v_pref;            /*   is given a new end goal (crowd_sim.py:779-786) */
    int32_t group_human;              /* sim.group_human (and not test.side_preference): the group environment, crowd_sim.py:476-622 */
    double unobservable_chance;       /* humans.unobservable_chance */
    double sf_A, sf_B, sf_KI;         /* sf.A, sf.B, sf.KI (crowd_nav/policy/social_force.py:22-27) */
} CnConfig;

/*
 * Canonical (test/injection) view of the env state, all DEVICE pointers,
 * row-major, n_envs rows.  Field order follows Agent.get_full_state_list
 * (utils/agent.py:116-127).  NULL members are skipped.
 */
typedef struct CnStateView {
    float *robot;      /* [N, 9]  px,py,vx,vy,radius,gx,gy,v_pref,theta */
    float *humans;     /* [N, H, 9] same field order */
    float *belief;     /* [N, H, 5] last_human_states px,py,vx,vy,r (crowd_sim.py:199,429-455) */
    float *extras;     /* [N, 4]  desiredVelocity[0], potential, last_acceleration x,y */
    int32_t *counters; /* [N, 4]  step_count, scenario_counter, case_counter, current_scenario */
    float *episode_return; /* [N]  running sum of rewards (bench.Monitor) */
    float *groups;     /* [N, CN_MAX_GROUPS, 4] group environment only (may be NULL): radius, centre x, centre y, valid (1/0) of the
                          static circle groups of the episode (self.circle_groups, crowd_sim.py:476-505) */
} CnStateView;

/* Observation dict of CrowdSimDict.generate_ob (crowd_sim_dict.py:72-103), float32. */
typedef struct CnObsOut {
    float *robot_node;      /* [N, 1, 7] px,py,r,gx,gy,v_pref,theta */
    float *temporal_edges;  /* [N, 1, 2] vx,vy */
    float *spatial_edges;   /* [N, H, 2] belief_p - robot_p */
    uint32_t *visible_mask; /* [N] bit i: human i inside the robot FOV (crowd_sim.py:851-865) */
} CnObsOut;

/* Per-step outputs of CrowdSimDict.step (crowd_sim_dict.py:205-271) + Monitor. */
typedef struct CnStepOut {
    CnObsOut obs;           /* post-step observation; the RESET observation where done (shmem_vec_env.py:165-168) */
    float *reward;          /* [N] */
    uint8_t *done;          /* [N] */
    int32_t *event;         /* [N] CN_EV_* */
    int32_t *scenario;      /* [N] CN_SCN_* of the episode the step belonged to */
    float *info;            /* [N, CN_INFO_DIM] see CN_INFO_* */
    float *episode_return;  /* [N] valid where done */
    int32_t *episode_length;/* [N] valid where done */
    uint32_t *goal_changed; /* [N] bit i: human i was given a new goal after this step (may be NULL) */
    float *not_done;        /* [N] 1.0f - done: the `masks` of the next Policy.act (train.py:279), may be NULL */
} CnStepOut;

/* columns of CnStepOut.info (step_info keys, crowd_sim.py:973-1030) */
enum {
    CN_INFO_DMIN = 0,            /* Danger.min_dist (inf when no human was scanned) */
    CN_INFO_AGGREGATE_NAV_TIME = 1,
    CN_INFO_PATH_VIOLATION = 2,
    CN_INFO_PERSONAL_VIOLATION = 3,
    CN_INFO_JERK_COST = 4,
    CN_INFO_DIST_TO_GOAL = 5,
    CN_INFO_SPEED_VIOLATION = 6,
    CN_INFO_SIDE_LEFT = 7,
    CN_INFO_SIDE_RIGHT = 8,
    CN_INFO_SEPARATION = 9,
    CN_INFO_DIM = 12
};

typedef struct CnEnv CnEnv;

const char *cn_last_error(void);
int cn_abi_version(void);

/* bytes of device memory the SoA state of n_envs needs; the caller allocates it */
size_t cn_env_state_bytes(const CnConfig *cfg, int n_envs);
int cn_env_create(const CnConfig *cfg, int n_envs, int device, void *state_dev, size_t state_bytes, CnEnv **out);
int cn_env_destroy(CnEnv *env);
/* CrowdSimDict.reset for the envs whose mask byte is non-zero (all when mask_dev == NULL) */
int cn_env_reset(CnEnv *env, const uint8_t *mask_dev, const CnObsOut *obs, void *stream);
/* CrowdSimDict.step on every env; action_dev [N,2] float32 raw policy output (clip_action is applied inside).
 * auto_reset != 0 reproduces the vec-env worker: done envs are reset and return the reset observation. */
int cn_env_step(CnEnv *env, const float *action_dev, const CnStepOut *out, int auto_reset, void *stream);
/* cn_env_reset / cn_env_step(auto_reset) also start generating the NEXT episode of the envs that were reset ("spare
 * episodes": the rejection-sampling spawn of the following reset, crowd_sim.py:359-393) on an internal stream that forks
 * from `stream`, so that the step kernel can swap a finished episode for its spare without waiting for the spawn.  The
 * next cn_env_* call joins that work automatically; cn_env_join makes `stream` wait for it explicitly (needed at the end
 * of a CUDA-graph capture, and before the caller frees or reads the state buffer on another stream). */
int cn_env_join(CnEnv *env, void *stream);
/* Start the refill at the current position of `stream` (what cn_env_step does by itself unless it was called with
 * auto_reset == 2 = "reset, but somebody else starts the refill"). */
int cn_env_refill(CnEnv *env, void *stream);
int cn_env_set_state(CnEnv *env, const CnStateView *view, void *stream);
int cn_env_get_state(CnEnv *env, const CnStateView *view, void *stream);
/* regenerate the observation from the current state without stepping (generate_ob(reset=True) semantics) */
int cn_env_observe(CnEnv *env, const CnObsOut *obs, void *stream);

/*
 * DS-RNN policy forward (SRNN.forward infer=True + DiagGaussian.fc_mean,
 * srnn_model.py:409-504, distributions.py:85-94).  Weights are DEVICE float32
 * tensors in the reference's own state_dict layout (row-major [out, in]).
 */
typedef struct CnDsrnnWeights {
    /* humanhumanEdgeRNN_temporal / _spatial: encoder_linear [64,2],[64]; gru weight_ih [768,64], weight_hh [768,256], biases [768] */
    const float *t_enc_w, *t_enc_b, *t_w_ih, *t_w_hh, *t_b_ih, *t_b_hh;
    const float *s_enc_w, *s_enc_b, *s_w_ih, *s_w_hh, *s_b_ih, *s_b_hh;
    /* attn.temporal_edge_layer.0 / spatial_edge_layer.0: [64,256],[64] */
    const float *att_t_w, *att_t_b, *att_s_w, *att_s_b;
    /* robot_linear [3,7],[3] */
    const float *robot_w, *robot_b;
    /* humanNodeRNN: encoder_linear [64,3],[64]; edge_attention_embed [64,512],[64]; gru [384,128],[384,128],[384],[384]; output_linear [256,128],[256] */
    const float *n_enc_w, *n_enc_b, *n_att_w, *n_att_b, *n_w_ih, *n_w_hh, *n_b_ih, *n_b_hh, *n_out_w, *n_out_b;
    /* actor.0, actor.2, critic.0, critic.2: [256,256],[256]; critic_linear [1,256],[1]; dist.fc_mean [2,256],[2] */
    const float *actor0_w, *actor0_b, *actor2_w, *actor2_b;
    const float *critic0_w, *critic0_b, *critic2_w, *critic2_b;
    const float *critic_lin_w, *critic_lin_b, *mean_w, *mean_b;
} CnDsrnnWeights;

typedef struct CnDsrnnIO {
    const float *robot_node;     /* [N,1,7] */
    const float *temporal_edges; /* [N,1,2] */
    const float *spatial_edges;  /* [N,H,2] */
    const float *h_node_in;      /* [N,1,128]   rnn_hxs["human_node_rnn"] */
    const float *h_edge_in;      /* [N,H+1,256] rnn_hxs["human_human_edge_rnn"] (row 0 temporal, 1..H spatial) */
    const float *masks;          /* [N,1] 0 where the episode just ended */
    float *h_node_out;           /* [N,1,128] */
    float *h_edge_out;           /* [N,H+1,256] */
    float *value;                /* [N,1] critic_linear output */
    float *action_mean;          /* [N,2] dist.fc_mean output */
    float *actor_features;       /* [N,256] hidden_actor (may be NULL) */
} CnDsrnnIO;

typedef struct CnDsrnn CnDsrnn;

/* precision of the tensor-core contractions */
/* FP32: CUDA cores, exact.  BF16X3: 3-pass split bf16 (operands ~2^-17).  BF16 / FP16: one tensor-core pass. */
enum { CN_PREC_FP32 = 0, CN_PREC_BF16X3 = 1, CN_PREC_BF16 = 2, CN_PREC_FP16 = 3 };

int cn_dsrnn_create(const CnDsrnnWeights *w, int device, void *stream, CnDsrnn **out);
int cn_dsrnn_destroy(CnDsrnn *m);
/* re-read (and re-pack) the weights after an optimiser step */
int cn_dsrnn_update_weights(CnDsrnn *m, const CnDsrnnWeights *w, void *stream);
size_t cn_dsrnn_workspace_bytes(int n_envs, int human_num);
int cn_dsrnn_forward(CnDsrnn *m, int n_envs, int human_num, const CnDsrnnIO *io, int precision,
                     void *workspace_dev, size_t workspace_bytes, void *stream);
/* A rollout that runs the forward right after the env step can let the FORWARD start the env's spare-episode refill, at
 * the point where it hurts least: next to the bandwidth-bound attention kernel (the refill's CTAs cannot share an SM with
 * the persistent tensor-core kernels, whose register / shared-memory footprint is a whole SM).  Pair
 * cn_dsrnn_set_refill_env(m, env) with cn_env_step(..., auto_reset = 2, ...); env == NULL clears it. */
int cn_dsrnn_set_refill_env(CnDsrnn *m, CnEnv *env);
/* Half-batch pipelining (rollout.PipelinedRollout): `event` (a cudaEvent_t owned by the caller, NULL clears it) is recorded on
 * the forward's stream right behind the edge-GRU stage -- the last part of a forward that fills the machine -- so another
 * stream can start the crowd step of an independent half batch beside the projection / attention / node kernels. */
int cn_dsrnn_set_edge_event(CnDsrnn *m, void *event);
/* Resident image of the edge hidden state for rollouts that feed a forward's output straight into the next forward
 * (rollout.GraphedRollout): bfloat16 hi / lo matrices [n_envs * (human_num + 1), 256] in LOGICAL row order (spatial rows
 * env * human_num + human first, then the temporal rows), x ~= hi + lo.  With out_hi / out_lo set, the next forwards (bf16x3)
 * also write the image of h_edge_out; with in_hi / in_lo set they read their A operand from it by TMA instead of converting
 * h_edge_in -- the caller guarantees that the image was written by the forward that produced exactly this h_edge_in and that
 * the masks are 0 or 1.  Same results bit for bit.  NULL pairs switch either half off. */
int cn_dsrnn_set_edge_image(CnDsrnn *m, void *in_hi, void *in_lo, void *out_hi, void *out_lo);
/* number of kernels the last forward / step call launched (bench.py's gpu_launches claim) */
int cn_dsrnn_last_launches(const CnDsrnn *m);
int cn_env_last_launches(const CnEnv *env);
/* Optional device timing of the dominant kernels (bench.py's roofline): when enabled the library brackets the
 * edge-GRU stage of every forward / the step kernel of every cn_env_step with CUDA events on the launching
 * stream.  *_time_ms() synchronises those events and returns the accumulated milliseconds and launch count
 * since the last call (and resets both). */
int cn_dsrnn_enable_timing(CnDsrnn *m, int enable);
int cn_dsrnn_time_ms(CnDsrnn *m, float *edge_stage_ms, int *n_forwards);
int cn_env_enable_timing(CnEnv *env, int enable);
int cn_env_time_ms(CnEnv *env, float *step_kernel_ms, int *n_steps);

/*
 * Training path (PPO update, SURVEY.md 8(f) N1): the gate math of ONE step of a masked GRU sequence
 * h_t = GRUCell(x_t, m_t * h_{t-1}) over R independent rows -- what nn.GRU does inside `_forward_gru`
 * (srnn_model.py:53-104) between two mask boundaries, and its gradient.  The recurrent GEMMs are the caller's
 * (cuBLAS); gate order r|z|n as in torch.nn.GRU.  All pointers are device float32, 16-byte aligned, hid % 4 == 0.
 *
 * forward:  gi = x_t W_ih^T, gh = hm W_hh^T [R,3 hid] (no biases), hm = m_t * h_{t-1} [R,hid], b_ih / b_hh [3 hid]
 *           -> h_out [R,hid]; ws [R,4 hid] = r | z | n | (W_hn hm + b_hn) for the backward;
 *              hm_next = m_next[row] * h_out (the next step's masked state) when hm_next != NULL.
 * backward: g = grad_h + (d_next ? m_next[row] * d_next : 0), where d_next = dL/d(hm of step t+1)
 *           -> dgi, dgh [R,3 hid] (gradients of gi and gh; bias gradients are their column sums), dhm = g * z
 *              (the direct part of dL/d(hm); the caller adds dgh W_hh).
 * Optional bfloat16 hi/lo copies (NULL = off; cn_split_bf16 below describes the pair) of what the NEXT GEMMs read, so that
 * the split-bf16 3-pass products need no separate pass over their operands: hm_next_hi/lo [R,hid] of hm_next;
 * dgi_hi/lo, dgh_hi/lo [R,3 hid] of dgi and dgh (all four or none).
 */
int cn_gru_gates_forward(const float *gi, const float *gh, const float *hm, const float *b_ih, const float *b_hh,
                         const float *m_next, float *h_out, float *hm_next, float *ws, void *hm_next_hi, void *hm_next_lo,
                         int rows, int hid, void *stream);
int cn_gru_gates_backward(const float *grad_h, const float *d_next, const float *m_next, const float *ws, const float *hm,
                          float *dgi, float *dgh, float *dhm, void *dgi_hi, void *dgi_lo, void *dgh_hi, void *dgh_lo,
                          int rows, int hid, void *stream);
/* a[n] float32 -> hi[n], lo[n] bfloat16 with hi = bf16(a), lo = bf16(a - hi): the operand pair of the split-bf16 3-pass
 * tensor-core products (A_hi B_hi + A_lo B_hi + A_hi B_lo, fp32 accumulation) the update can use for its recurrent GEMMs
 * (same arithmetic as the rollout's CN_PREC_BF16X3).  n % 4 == 0. */
int cn_split_bf16(const float *a, void *hi, void *lo, size_t n, void *stream);

/*
 * Native PPO-update path (SURVEY.md 8(f) N1; replaces the cuBLAS calls under `evaluate_actions` + autograd,
 * model.py:96-104, srnn_model.py:53-104, ppo.py:76-106).
 *
 * Sequence layout of every [T, rows, ...] array of the two edge GRUs: the T*S spatial rows (S = n_envs * human_num, step-major,
 * env-major, human-minor) come first, the T*n_envs temporal rows after them; "row" below is an index into that layout.
 */

/* One step t of both edge-GRU sequences: h_out = GRUCell(ReLU(W_enc x_t + b), m_t * h_in) on the tensor cores (the rollout's
 * edge kernel, CN_PREC_BF16X3), also writing what the backward reads. */
typedef struct CnEdgeSeqStep {
    const float *temporal_edges;   /* [n_envs, 2]    x_t of the temporal edges */
    const float *spatial_edges;    /* [S, 2]         x_t of the spatial edges */
    const float *masks;            /* [n_envs]       m_t */
    const float *h_in;             /* [*, 256] state before the step: rows in_row_spatial + s, in_row_temporal + e */
    long long in_row_spatial, in_row_temporal;
    long long out_row_spatial, out_row_temporal;   /* rows of this step in the arrays below */
    float *h_out;                  /* [*, 256]  h_t */
    float *ws;                     /* [*, 1024] r | z | n | W_hn hm + b_hn */
    void *hm_hi, *hm_lo;           /* bf16 [*, 256] split masked previous state m_t h_{t-1} (operand of dW_hh) */
    void *e_hi, *e_lo;             /* bf16 [*, 72]  split encoded input, then a constant 1 and seven 0: B operand of
                                      G^T [e | 1] = [dW_ih | column sums of G (bias gradients)] */
} CnEdgeSeqStep;
int cn_dsrnn_edge_sequence_step(CnDsrnn *m, int n_envs, int human_num, const CnEdgeSeqStep *io, void *stream);

/* Gate gradients of one step of a masked GRU sequence over `rows` rows, hid % 4 == 0 (elementwise, HBM-bound):
 *   g = grad_h + (d_inout_is_live ? m_next[row] * d : 0);  writes G = [dpre_n | dpre_r | dpre_z | dpre_n * r] as bf16 hi/lo
 *   pairs ([rows, 4 hid]: columns [0, 3 hid) are the gradient of gi in gate order n|r|z, columns [hid, 4 hid) the gradient of gh
 *   in gate order r|z|n) and d = g * z (fp32, in place), to which the caller adds G[:, hid:] W_hh with cn_gemm_bf16x3.
 *   hm = m_cur[row] * h_prev[row] is the masked state the step started from (h_prev == NULL: zero state). */
int cn_gru_gates_backward_pairs(const float *grad_h, float *d, int d_live, const float *m_next, const float *ws, const float *h_prev,
                                const float *m_cur, void *g_hi, void *g_lo, int rows, int hid, void *stream);

/* EdgeAttention of the update over a batch of T*n samples (srnn_model.py:256-339), key projection folded into the query:
 *   alpha = softmax_i((o_i . qt + cst) * scale), c = sum_i alpha_i o_i;  o [batch, human_num, 256], qt [batch, 256] = W_s^T q,
 *   cst [batch] = q . b_s (may be NULL), scale = human_num / sqrt(attention_size).  The backward returns d_o, d_qt and
 *   d_cst (may be NULL) from dc.  fp32, 16-byte aligned, human_num <= 32; HBM-bound (one pass over o forward, one backward). */
int cn_attention_train_forward(const float *o, const float *qt, const float *cst, float *c, float *alpha, float scale,
                               int batch, int human_num, void *stream);
int cn_attention_train_backward(const float *o, const float *qt, const float *alpha, const float *dc, float *d_o, float *d_qt,
                                float *d_cst, float scale, int batch, int human_num, void *stream);

/* Gradient of the edge encoder e = ReLU(W_enc x + b), x [rows, 2] (srnn_model.py:201-215): from de = dL/de [rows, 64] (fp32) and
 * the sign of e (bf16 image with row stride ld_e):  dw[64, 2] += sum_rows [e > 0] de x^T,  db[64] += sum_rows [e > 0] de.
 * dw / db must hold the initial value (zeros).  One HBM-bound pass over de.  cn_encoder_grad combines its block sums with
 * atomics (the order of the additions varies from run to run); cn_encoder_grad_ordered writes them to `workspace`
 * (cn_encoder_grad_ordered_workspace_bytes(rows) bytes, 16-byte aligned, owned by the caller) and adds them to dw / db in a
 * fixed order: the same inputs give the same bits.  A NULL, misaligned or too small workspace is refused. */
int cn_encoder_grad(const float *de, const void *e_hi, int ld_e, const float *x, float *dw, float *db, long long rows, void *stream);
size_t cn_encoder_grad_ordered_workspace_bytes(long long rows);
int cn_encoder_grad_ordered(const float *de, const void *e_hi, int ld_e, const float *x, float *dw, float *db, long long rows,
                            void *workspace, size_t workspace_bytes, void *stream);

/* Generic split-bf16 3-pass tensor-core GEMM (tcgen05, TMA-fed, fp32 accumulation in TMEM):
 *   C[m, n] (=, +=, or += for split-K)  (A_hi + A_lo)(B_hi + B_lo) minus the lo*lo term  (+ bias[n], activation).
 * Split-K partial products are added to C atomically by cn_gemm_bf16x3 (the order of the additions varies from run to run)
 * and in slice order by cn_gemm_bf16x3_ordered (below).
 * An operand is K-major (row-major [m|n, k] array) or MN-major (row-major [k, m|n] array); lo == NULL drops that operand's
 * correction pass.  Up to CN_GEMM_MAX_PROBLEMS independent problems per launch (grouped GEMM). */
#define CN_GEMM_MAX_PROBLEMS 4
typedef struct CnGemmOperand {
    const void *hi, *lo;   /* bfloat16, 16-byte aligned; ld % 8 == 0 */
    long long ld;          /* elements between consecutive rows of the array */
    int mn_major;          /* 0: array is [m|n, k] ; 1: array is [k, m|n] */
    int reserved;
} CnGemmOperand;
typedef struct CnGemm {
    CnGemmOperand a, b;
    float *c;              /* [m, ldc] */
    long long ldc;
    const float *bias;     /* [n] or NULL */
    int m, n, k;
    int act;               /* 0 none, 1 ReLU, 2 tanh */
    int accumulate;        /* split_k == 1 only: C += product instead of C = product */
    int split_k;           /* 1: no split.  >1 or 0 (= chosen by the library): k is cut into slices whose partial products are added
                              to C -- C must hold the initial value (zeros); no bias / activation */
} CnGemm;
int cn_gemm_bf16x3(const CnGemm *problems, int n_problems, void *stream);
/* Bit-reproducible form of cn_gemm_bf16x3: each k-slice stores its partial product into its own slice of `workspace` (owned by
 * the caller, 32-byte aligned), then C = C_in + P_0 + P_1 + ... + P_{S-1} is summed in slice order.  The slice count S of a
 * problem is a function of its own (m, n, k, split_k) only: split_k > 1 is taken as given (capped at one slice per 64-deep
 * k-block), split_k = 0 evaluates the library's automatic choice for the problem alone on a 148-SM budget.  So a problem
 * gives the same bits launched alone or grouped, on any device.  Problems with S = 1 are stored / accumulated directly.
 * cn_gemm_bf16x3_ordered_workspace_bytes returns the bytes the launch needs (sum over the problems with S > 1 of
 * S * m * n8 * 4, n8 = n rounded up to 8; pure host code) and, when `slices` is not NULL, each problem's S.  A launch whose
 * workspace is NULL, misaligned or smaller than that is refused (nothing is launched); no workspace is needed when it is 0. */
int cn_gemm_bf16x3_ordered_workspace_bytes(const CnGemm *problems, int n_problems, size_t *bytes, int *slices);
int cn_gemm_bf16x3_ordered(const CnGemm *problems, int n_problems, void *workspace, size_t workspace_bytes, void *stream);
/* Optional device timing of every cn_gemm_bf16x3 launch of this process (bench.py's roofline): CUDA events on the launching
 * stream; cn_gemm_time_ms synchronises them and returns the accumulated milliseconds, launch count and algorithmic FLOPs
 * (2 m n k per problem) since the last call, and resets them. */
int cn_gemm_enable_timing(int enable);
int cn_gemm_time_ms(float *ms, int *launches, double *flops);

#ifdef __cplusplus
}
#endif
#endif /* CROWDNAV_B200_H */
