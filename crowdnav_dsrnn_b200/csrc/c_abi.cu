// c_abi.cu -- extern "C" entry points of libcrowdnav_b200.so (include/crowdnav_b200.h).
// Host-side only: argument validation, handle bookkeeping, kernel launches.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <new>
#include "env_common.cuh"
#include "dsrnn.cuh"

static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CN_CUDA(call)                                                                   \
    do {                                                                                \
        cudaError_t err__ = (call);                                                     \
        if (err__ != cudaSuccess) return fail(CN_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(err__)); \
    } while (0)

// every entry point that owns a handle runs on the handle's device and leaves the caller's current device as it found it
struct DeviceGuard {
    int prev = -1;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int device)
    {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != device) err = cudaSetDevice(device);
        else prev = -1;                                  // nothing to restore
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define CN_ON_DEVICE(dev)                                                               \
    DeviceGuard guard__(dev);                                                           \
    if (guard__.err != cudaSuccess) return fail(CN_ERR_CUDA, "cudaSetDevice(%d): %s", (int)(dev), cudaGetErrorString(guard__.err))

extern "C" int cn_launch_crowd_step(const EnvParams *P, const CnStepOut *out, const float *action, int auto_reset, cudaStream_t stream);
extern "C" int cn_crowd_step_launches(const EnvParams *P);
extern "C" int cn_launch_crowd_reset(const EnvParams *P, const CnObsOut *obs, const uint8_t *mask, int mode, cudaStream_t stream);
enum { CN_RESET_LIVE = 0, CN_RESET_SPARE = 1, CN_RESET_SYNC = 2, CN_RESET_SPARE_LIST = 3 };   // crowd_reset.cu
extern "C" int cn_launch_crowd_observe(const EnvParams *P, const CnObsOut *obs, cudaStream_t stream);
extern "C" int cn_launch_state_convert(const EnvParams *P, const CnStateView *v, int dir, cudaStream_t stream);

#include <vector>
// pairs of events recorded around a kernel on the caller's stream; drained by *_time_ms()
struct EventTimer {
    bool enabled = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending, pool;
    void begin(cudaStream_t s) {
        if (!enabled) return;
        std::pair<cudaEvent_t, cudaEvent_t> p;
        if (!pool.empty()) { p = pool.back(); pool.pop_back(); }
        else { cudaEventCreate(&p.first); cudaEventCreate(&p.second); }
        cudaEventRecord(p.first, s);
        pending.push_back(p);
    }
    void end(cudaStream_t s) { if (enabled && !pending.empty()) cudaEventRecord(pending.back().second, s); }
    float drain(int *count) {
        float total = 0.f;
        for (auto &p : pending) {
            cudaEventSynchronize(p.second);
            float ms = 0.f;
            cudaEventElapsedTime(&ms, p.first, p.second);
            total += ms;
            pool.push_back(p);
        }
        if (count) *count = (int)pending.size();
        pending.clear();
        return total;
    }
    ~EventTimer() {
        for (auto &p : pending) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); }
        for (auto &p : pool) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); }
    }
};

struct CnEnv {
    EnvParams p;
    int device;
    int last_launches;
    EventTimer timer;
    // spare episodes are generated on an internal stream that forks from / joins the caller's stream with events
    cudaStream_t side = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_spare = nullptr;
    bool refill_pending = false;
};

// the caller's stream waits for the spare refill that is still in flight (if any)
static int join_refill(CnEnv *env, cudaStream_t s)
{
    if (env->refill_pending) {
        CN_CUDA(cudaStreamWaitEvent(s, env->ev_spare, 0));
        env->refill_pending = false;
    }
    return CN_OK;
}

// generate the next episode of every env flagged in need_spare, concurrently with whatever the caller enqueues next
static int fork_refill(CnEnv *env, cudaStream_t s, int mode = CN_RESET_SPARE_LIST)
{
    CN_CUDA(cudaEventRecord(env->ev_fork, s));
    CN_CUDA(cudaStreamWaitEvent(env->side, env->ev_fork, 0));
    CN_CUDA((cudaError_t)cn_launch_crowd_reset(&env->p, nullptr, nullptr, mode, env->side));
    CN_CUDA(cudaEventRecord(env->ev_spare, env->side));
    env->refill_pending = true;
    return CN_OK;
}

extern "C" const char *cn_last_error(void) { return g_err; }
extern "C" int cn_abi_version(void) { return CN_ABI_VERSION; }

static int check_config(const CnConfig *cfg)
{
    if (!cfg) return fail(CN_ERR_ARG, "cfg is NULL");
    if (cfg->abi_version != CN_ABI_VERSION) return fail(CN_ERR_ARG, "CnConfig.abi_version %d != %d", cfg->abi_version, CN_ABI_VERSION);
    if (cfg->human_num < 1 || cfg->human_num + (cfg->robot_visible ? 1 : 0) > CN_MAX_HUMANS)
        return fail(CN_ERR_ARG, "human_num %d out of range 1..%d", cfg->human_num, CN_MAX_HUMANS - (cfg->robot_visible ? 1 : 0));
    if (cfg->kinematics != CN_HOLONOMIC && cfg->kinematics != CN_UNICYCLE) return fail(CN_ERR_ARG, "unknown kinematics %d", cfg->kinematics);
    if (cfg->n_scenarios < 1 || cfg->n_scenarios > CN_MAX_SCENARIOS) return fail(CN_ERR_ARG, "n_scenarios %d out of range", cfg->n_scenarios);
    for (int i = 0; i < cfg->n_scenarios; ++i)
        if (cfg->scenarios[i] < 0 || cfg->scenarios[i] > CN_SCN_SIDE_PREF_CROSSING) return fail(CN_ERR_ARG, "unknown scenario id %d", cfg->scenarios[i]);
    if (!(cfg->time_step > 0.0) || cfg->timeout_step < 0) return fail(CN_ERR_ARG, "bad time_step/timeout_step");
    if (cfg->max_spawn_tries < 1 || cfg->max_goal_tries < 1 || cfg->max_robot_tries < 1) return fail(CN_ERR_ARG, "max_*_tries must be >= 1");
    if (cfg->case_size == 0) return fail(CN_ERR_ARG, "case_size must be > 0");
    if (cfg->social_metrics && cfg->n_scenarios != 4) return fail(CN_ERR_ARG, "social_metrics needs exactly 4 scenarios (crowd_sim_dict.py:116)");
    return CN_OK;
}

extern "C" size_t cn_env_state_bytes(const CnConfig *cfg, int n_envs)
{
    if (check_config(cfg) != CN_OK || n_envs < 1) return 0;
    return cn_carve(nullptr, nullptr, n_envs, cfg->human_num);
}

extern "C" int cn_env_create(const CnConfig *cfg, int n_envs, int device, void *state_dev, size_t state_bytes, CnEnv **out)
{
    if (!out) return fail(CN_ERR_ARG, "out is NULL");
    *out = nullptr;
    int rc = check_config(cfg);
    if (rc != CN_OK) return rc;
    if (n_envs < 1) return fail(CN_ERR_ARG, "n_envs must be >= 1");
    const size_t need = cn_carve(nullptr, nullptr, n_envs, cfg->human_num);
    if (!state_dev || state_bytes < need) return fail(CN_ERR_ARG, "state buffer too small: %zu < %zu", state_bytes, need);
    if (((uintptr_t)state_dev & 255) != 0) return fail(CN_ERR_ARG, "state buffer must be 256-byte aligned");
    int count = 0;
    CN_CUDA(cudaGetDeviceCount(&count));
    if (device < 0 || device >= count) return fail(CN_ERR_ARG, "device %d not present (%d devices)", device, count);
    cudaDeviceProp prop;
    CN_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(CN_ERR_UNSUPPORTED, "libcrowdnav_b200 is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
    CnEnv *env = new (std::nothrow) CnEnv();
    if (!env) return fail(CN_ERR_STATE, "out of host memory");
    env->p.cfg = *cfg;
    env->p.n_envs = n_envs;
    env->device = device;
    env->last_launches = 0;
    cn_carve(&env->p.a, state_dev, n_envs, cfg->human_num);
    DeviceGuard guard(device);
    if (guard.err != cudaSuccess) {
        delete env;
        return fail(CN_ERR_CUDA, "cudaSetDevice(%d): %s", device, cudaGetErrorString(guard.err));
    }
    if (cudaStreamCreateWithFlags(&env->side, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&env->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&env->ev_spare, cudaEventDisableTiming) != cudaSuccess) {
        cn_env_destroy(env);
        return fail(CN_ERR_CUDA, "could not create the spare-episode stream / events");
    }
    // spare bookkeeping starts empty whatever the caller's buffer holds: no valid spares, nothing flagged
    const size_t n = (size_t)n_envs;
    if (cudaMemset(env->p.a.sp_meta, 0, n * sizeof(int4)) != cudaSuccess || cudaMemset(env->p.a.need_spare, 0, n) != cudaSuccess ||
        cudaMemset(env->p.a.need_sync, 0, n) != cudaSuccess || cudaMemset(env->p.a.sync_count, 0, 4 * sizeof(int)) != cudaSuccess) {
        cn_env_destroy(env);
        return fail(CN_ERR_CUDA, "could not clear the spare-episode flags");
    }
    *out = env;
    return CN_OK;
}

extern "C" int cn_env_destroy(CnEnv *env)
{
    if (!env) return CN_OK;
    if (env->side) { cudaStreamSynchronize(env->side); cudaStreamDestroy(env->side); }
    if (env->ev_fork) cudaEventDestroy(env->ev_fork);
    if (env->ev_spare) cudaEventDestroy(env->ev_spare);
    delete env;
    return CN_OK;
}

extern "C" int cn_env_refill(CnEnv *env, void *stream)
{
    if (!env) return fail(CN_ERR_ARG, "env is NULL");
    CN_ON_DEVICE(env->device);
    int rc = join_refill(env, (cudaStream_t)stream);      // never two refills in flight
    if (rc != CN_OK) return rc;
    return fork_refill(env, (cudaStream_t)stream);
}

extern "C" int cn_env_join(CnEnv *env, void *stream)
{
    if (!env) return fail(CN_ERR_ARG, "env is NULL");
    CN_ON_DEVICE(env->device);
    return join_refill(env, (cudaStream_t)stream);
}

static int check_obs(const CnObsOut *obs)
{
    if (!obs || !obs->robot_node || !obs->temporal_edges || !obs->spatial_edges)
        return fail(CN_ERR_ARG, "CnObsOut needs robot_node, temporal_edges and spatial_edges");
    if (((uintptr_t)obs->spatial_edges & 7) != 0) return fail(CN_ERR_ARG, "spatial_edges must be 8-byte aligned");
    return CN_OK;
}

extern "C" int cn_env_reset(CnEnv *env, const uint8_t *mask_dev, const CnObsOut *obs, void *stream)
{
    if (!env) return fail(CN_ERR_ARG, "env is NULL");
    int rc = check_obs(obs);
    if (rc != CN_OK) return rc;
    CN_ON_DEVICE(env->device);
    rc = join_refill(env, (cudaStream_t)stream);
    if (rc != CN_OK) return rc;
    CN_CUDA((cudaError_t)cn_launch_crowd_reset(&env->p, obs, mask_dev, CN_RESET_LIVE, (cudaStream_t)stream));
    rc = fork_refill(env, (cudaStream_t)stream, CN_RESET_SPARE);       // the next episodes of the envs that were just reset
    if (rc != CN_OK) return rc;
    env->last_launches = 2;
    return CN_OK;
}

extern "C" int cn_env_step(CnEnv *env, const float *action_dev, const CnStepOut *out, int auto_reset, void *stream)
{
    if (!env) return fail(CN_ERR_ARG, "env is NULL");
    if (!action_dev || !out) return fail(CN_ERR_ARG, "action/out is NULL");
    int rc = check_obs(&out->obs);
    if (rc != CN_OK) return rc;
    if (!out->reward || !out->done || !out->event) return fail(CN_ERR_ARG, "CnStepOut needs reward, done and event");
    CN_ON_DEVICE(env->device);
#ifdef CN_DEBUG_SWITCHES
    {   // development builds only (make NET_FLAGS=-DCN_DEBUG_SWITCHES): 1 = no auto-reset at all, 2 = no spare refill
        static const int dbg = getenv("CN_DEBUG_RESET") ? atoi(getenv("CN_DEBUG_RESET")) : 0;
        if (dbg == 1) auto_reset = 0;
        if (dbg == 2 && auto_reset) auto_reset = 3;
    }
#endif
    rc = join_refill(env, (cudaStream_t)stream);        // the step kernel reads (and consumes) the spares
    if (rc != CN_OK) return rc;
    env->timer.begin((cudaStream_t)stream);
    CN_CUDA((cudaError_t)cn_launch_crowd_step(&env->p, out, action_dev, auto_reset ? 1 : 0, (cudaStream_t)stream));
    env->timer.end((cudaStream_t)stream);
    const int step_launches = cn_crowd_step_launches(&env->p);
    env->last_launches = step_launches;
    if (auto_reset) {
        // finished episodes were replaced by their spares inside the step kernel; the fall-back handles the envs whose
        // spare was missing (normally none: it exits at once), the refill runs beside the caller's next kernels
        CN_CUDA((cudaError_t)cn_launch_crowd_reset(&env->p, &out->obs, nullptr, CN_RESET_SYNC, (cudaStream_t)stream));
        env->last_launches = step_launches + 1;
        if (auto_reset == 1) {                         // 2: the caller (or the forward, cn_dsrnn_set_refill_env) starts the refill
            rc = fork_refill(env, (cudaStream_t)stream);
            if (rc != CN_OK) return rc;
            env->last_launches = step_launches + 2;
        }
    }
    return CN_OK;
}

extern "C" int cn_env_observe(CnEnv *env, const CnObsOut *obs, void *stream)
{
    if (!env) return fail(CN_ERR_ARG, "env is NULL");
    int rc = check_obs(obs);
    if (rc != CN_OK) return rc;
    CN_ON_DEVICE(env->device);
    CN_CUDA((cudaError_t)cn_launch_crowd_observe(&env->p, obs, (cudaStream_t)stream));
    env->last_launches = 1;
    return CN_OK;
}

extern "C" int cn_launch_robot_act(const EnvParams *P, int policy, float *action, cudaStream_t stream);

extern "C" int cn_env_robot_act(CnEnv *env, int32_t policy, float *action_dev, void *stream)
{
    if (!env) return fail(CN_ERR_ARG, "env is NULL");
    if (env->p.cfg.kinematics != CN_HOLONOMIC)
        return fail(CN_ERR_ARG, "cn_env_robot_act: ORCA and social force output velocities; a unicycle robot cannot take them");
    if (policy != CN_POLICY_ORCA && policy != CN_POLICY_SOCIAL_FORCE)
        return fail(CN_ERR_ARG, "cn_env_robot_act: unknown policy %d (CN_POLICY_ORCA or CN_POLICY_SOCIAL_FORCE)", (int)policy);
    if (!action_dev) return fail(CN_ERR_ARG, "cn_env_robot_act: action_dev is NULL");
    if (((uintptr_t)action_dev & 7) != 0) return fail(CN_ERR_ARG, "cn_env_robot_act: action_dev must be 8-byte aligned");
    CN_ON_DEVICE(env->device);
    int rc = join_refill(env, (cudaStream_t)stream);
    if (rc != CN_OK) return rc;
    CN_CUDA((cudaError_t)cn_launch_robot_act(&env->p, policy, action_dev, (cudaStream_t)stream));
    env->last_launches = 1;
    return CN_OK;
}

extern "C" int cn_launch_render(const EnvParams *P, const int32_t *ids, int k, const uint32_t *vis, int size, uint8_t *rgb,
                                cudaStream_t stream);

extern "C" int cn_env_render(CnEnv *env, const int32_t *env_ids_dev, int k, const uint32_t *visible_mask_dev, int size,
                             uint8_t *rgb_dev, void *stream)
{
    if (!env) return fail(CN_ERR_ARG, "env is NULL");
    if (size < CN_RENDER_MIN_SIZE || size > CN_RENDER_MAX_SIZE || size % CN_RENDER_SIZE_MULTIPLE != 0)
        return fail(CN_ERR_ARG, "cn_env_render: size %d must be a multiple of %d in %d..%d", size, CN_RENDER_SIZE_MULTIPLE,
                    CN_RENDER_MIN_SIZE, CN_RENDER_MAX_SIZE);
    if (k < 0) return fail(CN_ERR_ARG, "cn_env_render: k %d < 0", k);
    if (k == 0) {                                       // nothing to draw, nothing launched
        env->last_launches = 0;
        return CN_OK;
    }
    if (!rgb_dev) return fail(CN_ERR_ARG, "cn_env_render: rgb_dev is NULL");
    if (((uintptr_t)rgb_dev & 15) != 0) return fail(CN_ERR_ARG, "cn_env_render: rgb_dev must be 16-byte aligned");
    if (env_ids_dev == nullptr && k > env->p.n_envs)
        return fail(CN_ERR_ARG, "cn_env_render: k %d > %d envs without an id list", k, env->p.n_envs);
    CN_ON_DEVICE(env->device);
    // no join_refill: the render reads only the running episodes' arrays, which the refill never writes (render.cu)
    CN_CUDA((cudaError_t)cn_launch_render(&env->p, env_ids_dev, k, visible_mask_dev, size, rgb_dev, (cudaStream_t)stream));
    env->last_launches = 1;
    return CN_OK;
}

static int convert(CnEnv *env, const CnStateView *view, int dir, void *stream)
{
    if (!env || !view) return fail(CN_ERR_ARG, "env/view is NULL");
    CN_ON_DEVICE(env->device);
    if (join_refill(env, (cudaStream_t)stream) != CN_OK) return CN_ERR_CUDA;      // the refill reads the counters
    CN_CUDA((cudaError_t)cn_launch_state_convert(&env->p, view, dir, (cudaStream_t)stream));
    env->last_launches = 1;
    return CN_OK;
}

extern "C" int cn_env_set_state(CnEnv *env, const CnStateView *view, void *stream) { return convert(env, view, 0, stream); }
extern "C" int cn_env_get_state(CnEnv *env, const CnStateView *view, void *stream) { return convert(env, view, 1, stream); }
extern "C" int cn_env_last_launches(const CnEnv *env) { return env ? env->last_launches : 0; }
extern "C" int cn_env_enable_timing(CnEnv *env, int enable)
{
    if (!env) return fail(CN_ERR_ARG, "env is NULL");
    env->timer.drain(nullptr);
    env->timer.enabled = enable != 0;
    return CN_OK;
}
extern "C" int cn_env_time_ms(CnEnv *env, float *step_kernel_ms, int *n_steps)
{
    if (!env || !step_kernel_ms) return fail(CN_ERR_ARG, "env/out is NULL");
    *step_kernel_ms = env->timer.drain(n_steps);
    return CN_OK;
}

// ------------------------------------------------------------------------------------------------ DS-RNN
extern "C" int cn_dsrnn_create(const CnDsrnnWeights *w, int device, void *stream, CnDsrnn **out)
{
    if (!out) return fail(CN_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (!w) return fail(CN_ERR_ARG, "weights is NULL");
    const void *const *ptrs = reinterpret_cast<const void *const *>(w);
    for (size_t i = 0; i < sizeof(CnDsrnnWeights) / sizeof(void *); ++i)
        if (!ptrs[i]) return fail(CN_ERR_ARG, "CnDsrnnWeights member %zu is NULL", i);
    int count = 0;
    CN_CUDA(cudaGetDeviceCount(&count));
    if (device < 0 || device >= count) return fail(CN_ERR_ARG, "device %d not present (%d devices)", device, count);
    cudaDeviceProp prop;
    CN_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(CN_ERR_UNSUPPORTED, "libcrowdnav_b200 is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
    CN_ON_DEVICE(device);
    CnDsrnn *m = nullptr;
    const char *msg = dsrnn_create(w, device, (cudaStream_t)stream, &m);
    if (msg) return fail(CN_ERR_CUDA, "dsrnn_create: %s", msg);
    *out = m;
    return CN_OK;
}

extern "C" int cn_dsrnn_destroy(CnDsrnn *m)
{
    if (m) dsrnn_destroy(m);
    return CN_OK;
}

extern "C" int cn_dsrnn_update_weights(CnDsrnn *m, const CnDsrnnWeights *w, void *stream)
{
    if (!m || !w) return fail(CN_ERR_ARG, "model/weights is NULL");
    CN_ON_DEVICE(dsrnn_device(m));
    const char *msg = dsrnn_update_weights(m, w, (cudaStream_t)stream);
    if (msg) return fail(CN_ERR_CUDA, "dsrnn_update_weights: %s", msg);
    return CN_OK;
}

extern "C" size_t cn_dsrnn_workspace_bytes(int n_envs, int human_num)
{
    if (n_envs < 1 || human_num < 1 || human_num > CN_MAX_HUMANS) return 0;
    return dsrnn_workspace_bytes(n_envs, human_num);
}

extern "C" int cn_dsrnn_forward(CnDsrnn *m, int n_envs, int human_num, const CnDsrnnIO *io, int precision,
                                void *workspace_dev, size_t workspace_bytes, void *stream)
{
    if (!m || !io) return fail(CN_ERR_ARG, "model/io is NULL");
    if (n_envs < 1 || human_num < 1 || human_num > CN_MAX_HUMANS) return fail(CN_ERR_ARG, "bad n_envs/human_num");
    if (!io->robot_node || !io->temporal_edges || !io->spatial_edges || !io->h_node_in || !io->h_edge_in || !io->masks ||
        !io->h_node_out || !io->h_edge_out || !io->value || !io->action_mean)
        return fail(CN_ERR_ARG, "CnDsrnnIO has a NULL required member");
    if (precision < CN_PREC_FP32 || precision > CN_PREC_FP16)
        return fail(CN_ERR_ARG, "unknown precision %d", precision);
    const size_t need = dsrnn_workspace_bytes(n_envs, human_num);
    if (!workspace_dev || workspace_bytes < need) return fail(CN_ERR_ARG, "workspace too small: %zu < %zu", workspace_bytes, need);
    CN_ON_DEVICE(dsrnn_device(m));
    const char *msg = dsrnn_forward(m, n_envs, human_num, io, precision, workspace_dev, (cudaStream_t)stream);
    if (msg) return fail(CN_ERR_CUDA, "dsrnn_forward: %s", msg);
    return CN_OK;
}

extern "C" int cn_dsrnn_last_launches(const CnDsrnn *m) { return m ? dsrnn_last_launches(m) : 0; }
extern "C" int cn_dsrnn_set_refill_env(CnDsrnn *m, CnEnv *env)
{
    if (!m) return fail(CN_ERR_ARG, "model is NULL");
    dsrnn_set_refill_env(m, env);
    return CN_OK;
}

extern "C" int cn_dsrnn_set_edge_event(CnDsrnn *m, void *event)
{
    if (!m) return fail(CN_ERR_ARG, "model is NULL");
    dsrnn_set_edge_event(m, event);
    return CN_OK;
}

extern "C" int cn_dsrnn_set_edge_image(CnDsrnn *m, void *in_hi, void *in_lo, void *out_hi, void *out_lo)
{
    if (!m) return fail(CN_ERR_ARG, "model is NULL");
    if ((in_hi == nullptr) != (in_lo == nullptr) || (out_hi == nullptr) != (out_lo == nullptr))
        return fail(CN_ERR_ARG, "the hi and lo halves of an image come in pairs");
    dsrnn_set_edge_image(m, in_hi, in_lo, out_hi, out_lo);
    return CN_OK;
}

extern "C" int cn_dsrnn_enable_timing(CnDsrnn *m, int enable)
{
    if (!m) return fail(CN_ERR_ARG, "model is NULL");
    dsrnn_enable_timing(m, enable);
    return CN_OK;
}
extern "C" int cn_dsrnn_time_ms(CnDsrnn *m, float *edge_stage_ms, int *n_forwards)
{
    if (!m || !edge_stage_ms) return fail(CN_ERR_ARG, "model/out is NULL");
    *edge_stage_ms = dsrnn_time_ms(m, n_forwards);
    return CN_OK;
}

// ---------------------------------------------------------------------------------------------- training path (dsrnn_train.cu)
extern "C" int cn_launch_gru_gates_forward(const float *gi, const float *gh, const float *hm, const float *b_ih, const float *b_hh,
                                           const float *m_next, float *h_out, float *hm_next, float *ws, void *hm_next_hi,
                                           void *hm_next_lo, int R, int hid, cudaStream_t stream);
extern "C" int cn_launch_gru_gates_backward(const float *grad_h, const float *d_next, const float *m_next, const float *ws,
                                            const float *hm, float *dgi, float *dgh, float *dhm, void *const *pairs, int R, int hid,
                                            cudaStream_t stream);

extern "C" int cn_gru_gates_forward(const float *gi, const float *gh, const float *hm, const float *b_ih, const float *b_hh,
                                    const float *m_next, float *h_out, float *hm_next, float *ws, void *hm_next_hi, void *hm_next_lo,
                                    int rows, int hid, void *stream)
{
    if (!gi || !gh || !hm || !b_ih || !b_hh || !h_out || !ws) return fail(CN_ERR_ARG, "cn_gru_gates_forward: NULL pointer");
    const int rc = cn_launch_gru_gates_forward(gi, gh, hm, b_ih, b_hh, m_next, h_out, hm_next, ws, hm_next_hi, hm_next_lo, rows, hid,
                                               (cudaStream_t)stream);
    if (rc == -1) return fail(CN_ERR_ARG, "cn_gru_gates_forward: rows %d / hid %d / alignment / hm_next without m_next / half a bf16 pair", rows, hid);
    if (rc != 0) return fail(CN_ERR_CUDA, "gru_gates_forward_kernel: %s", cudaGetErrorString((cudaError_t)rc));
    return CN_OK;
}

extern "C" int cn_gru_gates_backward(const float *grad_h, const float *d_next, const float *m_next, const float *ws, const float *hm,
                                     float *dgi, float *dgh, float *dhm, void *dgi_hi, void *dgi_lo, void *dgh_hi, void *dgh_lo,
                                     int rows, int hid, void *stream)
{
    if (!grad_h || !ws || !hm || !dgi || !dgh || !dhm) return fail(CN_ERR_ARG, "cn_gru_gates_backward: NULL pointer");
    void *pairs[4] = {dgi_hi, dgi_lo, dgh_hi, dgh_lo};
    const bool any = dgi_hi || dgi_lo || dgh_hi || dgh_lo;
    const int rc = cn_launch_gru_gates_backward(grad_h, d_next, m_next, ws, hm, dgi, dgh, dhm, any ? pairs : nullptr, rows, hid,
                                                (cudaStream_t)stream);
    if (rc == -1) return fail(CN_ERR_ARG, "cn_gru_gates_backward: rows %d / hid %d / alignment / d_next without m_next / incomplete bf16 pairs", rows, hid);
    if (rc != 0) return fail(CN_ERR_CUDA, "gru_gates_backward_kernel: %s", cudaGetErrorString((cudaError_t)rc));
    return CN_OK;
}

extern "C" int cn_launch_split_bf16(const float *a, void *hi, void *lo, size_t n, cudaStream_t stream);
extern "C" int cn_split_bf16(const float *a, void *hi, void *lo, size_t n, void *stream)
{
    if (!a || !hi || !lo) return fail(CN_ERR_ARG, "cn_split_bf16: NULL pointer");
    const int rc = cn_launch_split_bf16(a, hi, lo, n, (cudaStream_t)stream);
    if (rc == -1) return fail(CN_ERR_ARG, "cn_split_bf16: n %zu must be a positive multiple of 4, a 16-byte and hi / lo 8-byte aligned", n);
    if (rc != 0) return fail(CN_ERR_CUDA, "split_bf16_kernel: %s", cudaGetErrorString((cudaError_t)rc));
    return CN_OK;
}

// ---------------------------------------------------------------------------------------------- native PPO-update path
extern "C" int cn_launch_gru_gates_backward_pairs(const float *grad_h, float *d, int d_live, const float *m_next, const float *ws,
                                                  const float *h_prev, const float *m_cur, void *g_hi, void *g_lo, int R, int hid,
                                                  cudaStream_t stream);
const char *gemm_bf16x3_launch(const CnGemm *problems, int n_problems, cudaStream_t stream, int *items_out, bool ordered,
                               void *workspace, size_t workspace_bytes);
const char *gemm_bf16x3_ordered_workspace(const CnGemm *problems, int n_problems, size_t *bytes, int *slices);

extern "C" int cn_gru_gates_backward_pairs(const float *grad_h, float *d, int d_live, const float *m_next, const float *ws,
                                           const float *h_prev, const float *m_cur, void *g_hi, void *g_lo, int rows, int hid, void *stream)
{
    if (!grad_h || !d || !ws || !g_hi || !g_lo) return fail(CN_ERR_ARG, "cn_gru_gates_backward_pairs: NULL pointer");
    const int rc = cn_launch_gru_gates_backward_pairs(grad_h, d, d_live, m_next, ws, h_prev, m_cur, g_hi, g_lo, rows, hid, (cudaStream_t)stream);
    if (rc == -1) return fail(CN_ERR_ARG, "cn_gru_gates_backward_pairs: rows %d / hid %d / alignment / live d without m_next / h_prev without m_cur", rows, hid);
    if (rc != 0) return fail(CN_ERR_CUDA, "gru_gates_backward_pairs_kernel: %s", cudaGetErrorString((cudaError_t)rc));
    return CN_OK;
}

extern "C" int cn_gemm_bf16x3(const CnGemm *problems, int n_problems, void *stream)
{
    if (!problems) return fail(CN_ERR_ARG, "cn_gemm_bf16x3: problems is NULL");
    const char *msg = gemm_bf16x3_launch(problems, n_problems, (cudaStream_t)stream, nullptr, false, nullptr, 0);
    if (msg) return fail(CN_ERR_ARG, "cn_gemm_bf16x3: %s", msg);
    return CN_OK;
}

extern "C" int cn_gemm_bf16x3_ordered_workspace_bytes(const CnGemm *problems, int n_problems, size_t *bytes, int *slices)
{
    if (!problems || !bytes) return fail(CN_ERR_ARG, "cn_gemm_bf16x3_ordered_workspace_bytes: NULL pointer");
    const char *msg = gemm_bf16x3_ordered_workspace(problems, n_problems, bytes, slices);
    if (msg) return fail(CN_ERR_ARG, "cn_gemm_bf16x3_ordered_workspace_bytes: %s", msg);
    return CN_OK;
}

extern "C" int cn_gemm_bf16x3_ordered(const CnGemm *problems, int n_problems, void *workspace, size_t workspace_bytes, void *stream)
{
    if (!problems) return fail(CN_ERR_ARG, "cn_gemm_bf16x3_ordered: problems is NULL");
    const char *msg = gemm_bf16x3_launch(problems, n_problems, (cudaStream_t)stream, nullptr, true, workspace, workspace_bytes);
    if (msg) return fail(CN_ERR_ARG, "cn_gemm_bf16x3_ordered: %s", msg);
    return CN_OK;
}

extern "C" int cn_dsrnn_edge_sequence_step(CnDsrnn *m, int n_envs, int human_num, const CnEdgeSeqStep *io, void *stream)
{
    if (!m || !io) return fail(CN_ERR_ARG, "model/io is NULL");
    if (n_envs < 1 || human_num < 1 || human_num > CN_MAX_HUMANS) return fail(CN_ERR_ARG, "bad n_envs/human_num");
    if (!io->temporal_edges || !io->spatial_edges || !io->masks || !io->h_in || !io->h_out || !io->ws || !io->hm_hi || !io->hm_lo ||
        !io->e_hi || !io->e_lo) return fail(CN_ERR_ARG, "CnEdgeSeqStep has a NULL member");
    CN_ON_DEVICE(dsrnn_device(m));
    const char *msg = dsrnn_edge_sequence_step(m, n_envs, human_num, io, (cudaStream_t)stream);
    if (msg) return fail(CN_ERR_CUDA, "dsrnn_edge_sequence_step: %s", msg);
    return CN_OK;
}

extern "C" int cn_launch_attention_train_forward(const float *o, const float *qt, const float *cst, float *c, float *alpha, float scale,
                                                 int B, int H, cudaStream_t stream);
extern "C" int cn_launch_attention_train_backward(const float *o, const float *qt, const float *alpha, const float *dc, float *d_o,
                                                  float *d_qt, float *d_cst, float scale, int B, int H, cudaStream_t stream);

extern "C" int cn_attention_train_forward(const float *o, const float *qt, const float *cst, float *c, float *alpha, float scale,
                                          int batch, int human_num, void *stream)
{
    if (!o || !qt || !c || !alpha) return fail(CN_ERR_ARG, "cn_attention_train_forward: NULL pointer");
    const int rc = cn_launch_attention_train_forward(o, qt, cst, c, alpha, scale, batch, human_num, (cudaStream_t)stream);
    if (rc == -1) return fail(CN_ERR_ARG, "cn_attention_train_forward: batch %d / human_num %d (1..32) / 16-byte alignment", batch, human_num);
    if (rc != 0) return fail(CN_ERR_CUDA, "attention_train_forward_kernel: %s", cudaGetErrorString((cudaError_t)rc));
    return CN_OK;
}

extern "C" int cn_attention_train_backward(const float *o, const float *qt, const float *alpha, const float *dc, float *d_o, float *d_qt,
                                           float *d_cst, float scale, int batch, int human_num, void *stream)
{
    if (!o || !qt || !alpha || !dc || !d_o || !d_qt) return fail(CN_ERR_ARG, "cn_attention_train_backward: NULL pointer");
    const int rc = cn_launch_attention_train_backward(o, qt, alpha, dc, d_o, d_qt, d_cst, scale, batch, human_num, (cudaStream_t)stream);
    if (rc == -1) return fail(CN_ERR_ARG, "cn_attention_train_backward: batch %d / human_num %d (1..32) / 16-byte alignment", batch, human_num);
    if (rc != 0) return fail(CN_ERR_CUDA, "attention_train_backward_kernel: %s", cudaGetErrorString((cudaError_t)rc));
    return CN_OK;
}

void gemm_bf16x3_enable_timing(int enable);
float gemm_bf16x3_time_ms(int *launches, double *flops);
extern "C" int cn_gemm_enable_timing(int enable) { gemm_bf16x3_enable_timing(enable); return CN_OK; }
extern "C" int cn_gemm_time_ms(float *ms, int *launches, double *flops)
{
    if (!ms) return fail(CN_ERR_ARG, "cn_gemm_time_ms: ms is NULL");
    *ms = gemm_bf16x3_time_ms(launches, flops);
    return CN_OK;
}

extern "C" int cn_launch_encoder_grad(const float *de, const void *e_hi, int ld_e, const float *x, float *dw, float *db, long long rows,
                                      cudaStream_t stream);
extern "C" int cn_encoder_grad(const float *de, const void *e_hi, int ld_e, const float *x, float *dw, float *db, long long rows, void *stream)
{
    if (!de || !e_hi || !x || !dw || !db) return fail(CN_ERR_ARG, "cn_encoder_grad: NULL pointer");
    const int rc = cn_launch_encoder_grad(de, e_hi, ld_e, x, dw, db, rows, (cudaStream_t)stream);
    if (rc == -1) return fail(CN_ERR_ARG, "cn_encoder_grad: rows %lld / ld_e %d (>= 64) / alignment", rows, ld_e);
    if (rc != 0) return fail(CN_ERR_CUDA, "encoder_grad_kernel: %s", cudaGetErrorString((cudaError_t)rc));
    return CN_OK;
}

extern "C" size_t cn_launch_encoder_grad_ordered_bytes(long long rows);
extern "C" int cn_launch_encoder_grad_ordered(const float *de, const void *e_hi, int ld_e, const float *x, float *dw, float *db, long long rows,
                                              void *workspace, size_t workspace_bytes, cudaStream_t stream);
extern "C" size_t cn_encoder_grad_ordered_workspace_bytes(long long rows) { return cn_launch_encoder_grad_ordered_bytes(rows); }
extern "C" int cn_encoder_grad_ordered(const float *de, const void *e_hi, int ld_e, const float *x, float *dw, float *db, long long rows,
                                       void *workspace, size_t workspace_bytes, void *stream)
{
    if (!de || !e_hi || !x || !dw || !db) return fail(CN_ERR_ARG, "cn_encoder_grad_ordered: NULL pointer");
    const int rc = cn_launch_encoder_grad_ordered(de, e_hi, ld_e, x, dw, db, rows, workspace, workspace_bytes, (cudaStream_t)stream);
    if (rc == -1) return fail(CN_ERR_ARG, "cn_encoder_grad_ordered: rows %lld / ld_e %d (>= 64) / alignment", rows, ld_e);
    if (rc == -2)
        return fail(CN_ERR_ARG, "cn_encoder_grad_ordered: workspace NULL, not 16-byte aligned or smaller than %zu bytes (%zu given)",
                    cn_launch_encoder_grad_ordered_bytes(rows), workspace_bytes);
    if (rc != 0) return fail(CN_ERR_CUDA, "encoder_grad_kernel (ordered): %s", cudaGetErrorString((cudaError_t)rc));
    return CN_OK;
}
