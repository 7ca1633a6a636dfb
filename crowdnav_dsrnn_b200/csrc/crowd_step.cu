// crowd_step.cu -- K1: the fused crowd-step kernel (sm_100a).  Compile with -fmad=false.
//
// One launch does, for every env, what CrowdSimDict.step does
// (crowd_sim/envs/crowd_sim_dict.py:205-271):
//   phase A  every human's ORCA solve (crowd_nav/policy/orca.py:64-139 -> RVO2
//            computeNeighbors / computeNewVelocity / linearProgram1-3), one G-lane
//            group per human: lane l owns neighbour l, builds its half-plane, the
//            group ranks the neighbours by (distSq, index) with shuffles, and the
//            incremental LP runs with ballots (first violated constraint) and
//            shuffle reductions (feasible interval on the violated line);
//   phase B  one warp per env, lane i owns human i: clip_action (srnn.py:18-48),
//            unicycle accumulation, calc_reward on the PRE-step state
//            (crowd_sim.py:907-1094), integration (agent.py:172-212), FOV mask +
//            belief update + observation writes (crowd_sim_dict.py:72-103,
//            crowd_sim.py:429-455, 820-865) and goal re-sampling
//            (crowd_sim.py:724-811) from the counter-based RNG.
// The CTA stages its E consecutive envs' humans in shared memory with coalesced
// float4 loads; nothing is re-read from HBM.  ORCA arithmetic is fp32 without
// FMA contraction (bit-identical to a stock x86-64 build of RVO2 and to
// oracle/orca_core.h); everything the reference does in Python floats is fp64.
#include <cstdlib>
#include "env_common.cuh"

#define ORCA_EPS 0.00001f
#ifndef STEP_THREADS
#define STEP_THREADS 256
#endif
#ifndef STEP_MIN_BLOCKS
#define STEP_MIN_BLOCKS 4
#endif

template <int G> struct GroupOps {
    static constexpr unsigned kLow = (G == 32) ? 0xffffffffu : ((1u << G) - 1u);
    unsigned gmask;  // lanes of this group inside the warp
    int gbase;       // first lane of the group
    int gl;          // lane index inside the group
    __device__ __forceinline__ float shfl(float v, int src) const { return __shfl_sync(gmask, v, src, G); }
    __device__ __forceinline__ int shfl_i(int v, int src) const { return __shfl_sync(gmask, v, src, G); }
    __device__ __forceinline__ unsigned ballot(bool p) const { return (__ballot_sync(gmask, p) >> gbase) & kLow; }
    // group-relative mask of the lanes holding the same value
    __device__ __forceinline__ unsigned match(int v) const { return (__match_any_sync(gmask, v) >> gbase) & kLow; }
    // min/max over the group in ONE instruction each: sm_100a reduces floats directly (redux.sync.{min,max}.f32 -> CREDUX.F32).
    // Exact: a reduction only selects one of its inputs, and the LP never feeds NaNs here.
    __device__ __forceinline__ float rmax(float v) const { float r; asm volatile("redux.sync.max.f32 %0, %1, %2;" : "=f"(r) : "f"(v), "r"(gmask)); return r; }
    __device__ __forceinline__ float rmin(float v) const { float r; asm volatile("redux.sync.min.f32 %0, %1, %2;" : "=f"(r) : "f"(v), "r"(gmask)); return r; }
};

struct Line { float px, py, dx, dy; };

__device__ __forceinline__ float det2(float ax, float ay, float bx, float by) { return ax * by - ay * bx; }

// linearProgram1: optimise on line k subject to the valid lines of lanes < k and the speed disc
// (`s_lines`: the same lines in shared memory, slot = lane: line k is one broadcast LDS.128 instead of four shuffles)
template <int G>
__device__ __forceinline__ bool lp1_group(const GroupOps<G> &g, const Line &ln, bool valid, int k, float radius,
                                          float optx, float opty, bool dir_opt, float &rx, float &ry, const float4 *s_lines)
{
    const float4 lk = s_lines[k];
    const float kpx = lk.x, kpy = lk.y, kdx = lk.z, kdy = lk.w;
    const float dp = kpx * kdx + kpy * kdy;
    const float disc = dp * dp + radius * radius - (kpx * kpx + kpy * kpy);
    if (disc < 0.0f) return false;
    const float sq = sqrtf(disc);
    float t_left = -dp - sq, t_right = -dp + sq;
    bool fail = false;
    float tl = -INFINITY, tr = INFINITY;
    if (valid && g.gl < k) {
        const float den = det2(kdx, kdy, ln.dx, ln.dy);
        const float num = det2(ln.dx, ln.dy, kpx - ln.px, kpy - ln.py);
        if (fabsf(den) <= ORCA_EPS) fail = num < 0.0f;
        else {
            const float t = num / den;
            if (den >= 0.0f) tr = t; else tl = t;
        }
    }
    const bool any_fail = g.ballot(fail) != 0u;
    tl = g.rmax(tl);
    tr = g.rmin(tr);
    if (t_left < tl) t_left = tl;
    if (tr < t_right) t_right = tr;
    if (any_fail || t_left > t_right) return false;
    float t;
    if (dir_opt) t = (optx * kdx + opty * kdy > 0.0f) ? t_right : t_left;
    else {
        t = kdx * (optx - kpx) + kdy * (opty - kpy);
        if (t < t_left) t = t_left; else if (t > t_right) t = t_right;
    }
    rx = kpx + t * kdx; ry = kpy + t * kdy;
    return true;
}

// linearProgram2 over the lanes' lines in lane order; returns the failing index or -1 when all lines hold
template <int G>
__device__ __forceinline__ int lp2_group(const GroupOps<G> &g, const Line &ln, bool valid, float radius,
                                         float optx, float opty, bool dir_opt, float &rx, float &ry, const float4 *s_lines)
{
    if (dir_opt) { rx = radius * optx; ry = radius * opty; }
    else if (optx * optx + opty * opty > radius * radius) {
        const float inv = 1.0f / sqrtf(optx * optx + opty * opty);
        rx = radius * (optx * inv); ry = radius * (opty * inv);
    } else { rx = optx; ry = opty; }
    int next = 0;
    while (true) {
        const bool viol = valid && g.gl >= next && det2(ln.dx, ln.dy, ln.px - rx, ln.py - ry) > 0.0f;
        const unsigned b = g.ballot(viol);
        if (b == 0u) return -1;
        const int k = __ffs(b) - 1;
        const float tx = rx, ty = ry;
        if (!lp1_group<G>(g, ln, valid, k, radius, optx, opty, dir_opt, rx, ry, s_lines)) { rx = tx; ry = ty; return k; }
        next = k + 1;
    }
}

// linearProgram3 (no obstacle lines): minimise the maximum penetration from line `begin` on
// (`s_lines`: the lanes' lines in shared memory; `s_proj`: scratch of the same size for the projected lines)
template <int G>
__device__ __forceinline__ void lp3_group(const GroupOps<G> &g, const Line &ln, int n, int begin, float radius,
                                          float &rx, float &ry, const float4 *s_lines, float4 *s_proj)
{
    float distance = 0.0f;
    // RVO2 walks the lines from `begin` and re-solves at every line that is penetrated by more than `distance`; between two
    // such lines neither the velocity nor `distance` changes, so every lane tests its own line and a ballot names the next one
    for (int i = begin; i < n; ++i) {
        const unsigned pen = g.ballot(g.gl >= i && g.gl < n && det2(ln.dx, ln.dy, ln.px - rx, ln.py - ry) > distance);
        if (pen == 0u) break;
        i = __ffs(pen) - 1;
        const float4 li = s_lines[i];
        const float kpx = li.x, kpy = li.y, kdx = li.z, kdy = li.w;
        {
            Line pl; pl.px = pl.py = pl.dx = pl.dy = 0.0f;
            bool pvalid = false;
            if (g.gl < i) {
                const float d = det2(kdx, kdy, ln.dx, ln.dy);
                if (fabsf(d) <= ORCA_EPS) {
                    if (!(kdx * ln.dx + kdy * ln.dy > 0.0f)) {
                        pl.px = 0.5f * (kpx + ln.px); pl.py = 0.5f * (kpy + ln.py); pvalid = true;
                    }
                } else {
                    const float t = det2(ln.dx, ln.dy, kpx - ln.px, kpy - ln.py) / d;
                    pl.px = kpx + t * kdx; pl.py = kpy + t * kdy; pvalid = true;
                }
                if (pvalid) {
                    const float ex = ln.dx - kdx, ey = ln.dy - kdy;
                    const float inv = 1.0f / sqrtf(ex * ex + ey * ey);
                    pl.dx = ex * inv; pl.dy = ey * inv;
                }
            }
            __syncwarp(g.gmask);                  // the previous round's readers are done with s_proj
            s_proj[g.gl] = make_float4(pl.px, pl.py, pl.dx, pl.dy);
            __syncwarp(g.gmask);
            const float tx = rx, ty = ry;
            if (lp2_group<G>(g, pl, pvalid, radius, -kdy, kdx, true, rx, ry, s_proj) >= 0) { rx = tx; ry = ty; }
            distance = det2(kdx, kdy, kpx - rx, kpy - ry);
        }
    }
}

// preferred velocity (orca.py:118-122), Python floats -> narrowed at the rvo2 boundary.  One fp64 sqrt and two fp64
// divisions per human: computed by ONE thread per human while the CTA stages its envs, not by every lane of the solve.
__device__ __forceinline__ float2 preferred_velocity(float4 pv, float4 gr)
{
    const double gdx = (double)gr.x - (double)pv.x, gdy = (double)gr.y - (double)pv.y;
    const double gsp = norm2d(gdx, gdy);
    return make_float2((float)(gsp > 1.0 ? gdx / gsp : gdx), (float)(gsp > 1.0 ? gdy / gsp : gdy));
}

// Who solves, and where its neighbours come from: human i of the env staged in shared memory (the step kernel), or the
// robot with the env's belief rows last_human_states as its neighbours (robot_act_kernel, robot.policy = orca /
// social_force).  Every branch on it is a compile-time constant, so each form compiles to its own straight code.
enum { AGENT_HUMAN = 0, AGENT_ROBOT_ORCA = 1, AGENT_ROBOT_SF = 2 };

// One agent's action by one G-lane group: the ORCA solve, or (kOpt builds and the social-force robot only) the
// social-force step.  kAgent == AGENT_HUMAN: s_pv/s_gr/s_th hold this env's humans (pre-step), i is the solver.  A robot
// agent is rob_pv / P.a.rob_gr[e] and lane k reads belief row k of env e (i, s_pv, s_gr, s_th, rob_radius and rob_theta
// are not used).  kOpt compiles the optional behaviours of SURVEY 8(f) N4 in (humans.policy = social_force,
// random_policy_changing, random_unobservability); the default kernel has none of them.
template <int G, bool kOpt, int kAgent = AGENT_HUMAN>
__device__ __forceinline__ float2 orca_group(const CnConfig &cfg, const GroupOps<G> &g, int i, int H,
                                             const float4 *s_pv, const float4 *s_gr, const float *s_th, float2 pref,
                                             float4 rob_pv, float rob_radius, float rob_theta, float4 *s_scratch,
                                             const EnvParams &P, int e)
{
    constexpr bool kRobot = kAgent != AGENT_HUMAN;
    const float4 me = kRobot ? rob_pv : s_pv[i];
    const float4 me_g = kRobot ? P.a.rob_gr[e] : s_gr[i];
    const float radius = (float)((double)me_g.z + 0.01 + (double)cfg.orca_safety_space);
    const float max_speed = me_g.w;
    const float prefx = pref.x, prefy = pref.y;

    const int M = kRobot ? H : H - 1 + (cfg.robot_visible ? 1 : 0);
    const bool have = g.gl < M;
    float ox = 0.f, oy = 0.f, ovx = 0.f, ovy = 0.f, orad = 0.f;
    double raw_r = 0.0;
    int4 ctr = make_int4(0, 0, 0, 0);
    if (kOpt) ctr = P.a.ctr[e];
    if (kRobot && have) {
        const size_t hi = (size_t)e * H + g.gl;
        const float4 b = P.a.hum_bel[hi];
        ox = b.x; oy = b.y; ovx = b.z; ovy = b.w; raw_r = (double)P.a.hum_br[hi];
        orad = (float)(raw_r + 0.01 + (double)cfg.orca_safety_space);
    }
    if (!kRobot && have) {
        const bool limited = cfg.human_fov < 2.0 * CN_PI;
        const double my_th = (limited && cfg.kinematics != CN_HOLONOMIC) ? (double)s_th[i] : 0.0;
        bool vis = true;
        // humans.random_unobservability (crowd_sim.py:1121-1153): human 0 misses each neighbour with unobservable_chance,
        // one draw per (step, neighbour slot)
        bool blind = false;
        if (kOpt && cfg.random_unobservability && i == 0)
            blind = u01(philox4x32(step_key(cfg, ctr.y, e), (uint32_t)g.gl, 0u, (uint32_t)ctr.x, RNG_UNOBS).x) <= cfg.unobservable_chance;
        if (g.gl < H - 1) {
            const int j = g.gl + (g.gl >= i ? 1 : 0);
            const float4 o = s_pv[j];
            ox = o.x; oy = o.y; ovx = o.z; ovy = o.w; raw_r = (double)s_gr[j].z;
            if (limited) vis = detect_visible_d(cfg.kinematics, me.x, me.y, me.z, me.w, my_th, ox, oy, cfg.human_fov);
            if (kOpt && blind) vis = false;
            if (!vis) raw_r = cfg.human_radius;
        } else {
            ox = rob_pv.x; oy = rob_pv.y; ovx = rob_pv.z; ovy = rob_pv.w; raw_r = (double)rob_radius;
            if (limited) vis = detect_visible_d(cfg.kinematics, me.x, me.y, me.z, me.w, my_th, ox, oy, cfg.human_fov);
            if (kOpt && blind) vis = false;
            if (!vis) raw_r = cfg.robot_radius;
        }
        if (!vis) { ox = 7.0f; oy = 7.0f; ovx = 0.0f; ovy = 0.0f; }   // dummy_human, crowd_sim.py:161-163
        orad = (float)(raw_r + 0.01 + (double)cfg.orca_safety_space);
    }
    if (kAgent == AGENT_ROBOT_SF || (kOpt && human_policy_of(cfg, ctr.z, e, i) == CN_POLICY_SOCIAL_FORCE)) {
        // SOCIAL_FORCE.predict (crowd_nav/policy/social_force.py:11-63), Python floats -> fp64.  Lane k owns the push of
        // neighbour slot k; the sum runs in slot order like the reference's loop.
        double tx = 0.0, ty = 0.0;
        if (have) {
            const double ddx = (double)me.x - (double)ox, ddy = (double)me.y - (double)oy;
            const double dist = sqrt(ddx * ddx + ddy * ddy);
            const double f = cfg.sf_A * exp(((double)me_g.z + raw_r - dist) / cfg.sf_B);
            tx = f * (ddx / dist); ty = f * (ddy / dist);
        }
        double ivx = 0.0, ivy = 0.0;
        for (int k = 0; k < M; ++k) {
            const double ax = __hiloint2double(g.shfl_i(__double2hiint(tx), k), g.shfl_i(__double2loint(tx), k));
            const double ay = __hiloint2double(g.shfl_i(__double2hiint(ty), k), g.shfl_i(__double2loint(ty), k));
            ivx += ax; ivy += ay;
        }
        const double gdx = (double)me_g.x - (double)me.x, gdy = (double)me_g.y - (double)me.y;
        const double gdist = sqrt(gdx * gdx + gdy * gdy);
        const double vp = (double)me_g.w;
        const double cdx = cfg.sf_KI * ((gdx / gdist) * vp - (double)me.z), cdy = cfg.sf_KI * ((gdy / gdist) * vp - (double)me.w);
        const double nvx = (double)me.z + (cdx + ivx) * cfg.time_step, nvy = (double)me.w + (cdy + ivy) * cfg.time_step;
        const double nrm = sqrt(nvx * nvx + nvy * nvy);
        if (nrm > vp) return make_float2((float)(nvx / nrm * vp), (float)(nvy / nrm * vp));
        return make_float2((float)nvx, (float)nvy);
    }
    (void)rob_theta;

    // computeNeighbors: everyone strictly inside neighborDist, ascending (distSq, index)
    const float ddx = me.x - ox, ddy = me.y - oy;
    const float dist_sq = ddx * ddx + ddy * ddy;
    const bool in = have && dist_sq < cfg.orca_neighbor_dist * cfg.orca_neighbor_dist;
    const unsigned in_bits = g.ballot(in);
    const int n = __popc(in_bits);
    // rank = number of in-range neighbours that sort before this one.  dist_sq >= +0, so its bit pattern orders like the
    // float; out-of-range slots get the largest key and never count.  Ties (equal distSq, lower index first) come from one
    // MATCH instruction instead of a second comparison per candidate.
    const int key = in ? __float_as_int(dist_sq) : 0x7fffffff;
    // the keys go through the group's scratch: every lane reads them back four at a time (broadcast LDS.128) instead of one
    // shuffle per candidate
    int rank = 0;
    {
        int *s_keys = reinterpret_cast<int *>(s_scratch);
        s_keys[g.gl] = key;                                     // slots >= M hold the out-of-range key and never count
        __syncwarp(g.gmask);
        for (int k4 = 0; k4 < (M + 3) >> 2; ++k4) {
            const int4 kk = reinterpret_cast<const int4 *>(s_keys)[k4];
            rank += (kk.x < key ? 1 : 0) + (kk.y < key ? 1 : 0) + (kk.z < key ? 1 : 0) + (kk.w < key ? 1 : 0);
        }
        __syncwarp(g.gmask);                                    // the scratch is reused for the ranked half-planes below
    }
    rank += __popc(g.match(key) & in_bits & ((1u << g.gl) - 1u));

    // computeNewVelocity: this lane's half-plane
    Line ln; ln.px = ln.py = ln.dx = ln.dy = 0.0f;
    if (in) {
        const float rpx = ox - me.x, rpy = oy - me.y;
        const float rvx = me.z - ovx, rvy = me.w - ovy;
        const float dsq = rpx * rpx + rpy * rpy;
        const float R = radius + orad;
        const float R2 = R * R;
        float ux, uy;
        if (dsq > R2) {
            const float inv_tau = 1.0f / cfg.orca_time_horizon;
            const float wx = rvx - inv_tau * rpx, wy = rvy - inv_tau * rpy;
            const float wl2 = wx * wx + wy * wy;
            const float dp1 = wx * rpx + wy * rpy;
            if (dp1 < 0.0f && dp1 * dp1 > R2 * wl2) {
                const float wl = sqrtf(wl2);
                const float inv = 1.0f / wl;
                const float uwx = wx * inv, uwy = wy * inv;
                ln.dx = uwy; ln.dy = -uwx;
                const float sc = R * inv_tau - wl;
                ux = sc * uwx; uy = sc * uwy;
            } else {
                const float leg = sqrtf(dsq - R2);
                const float inv = 1.0f / dsq;
                if (det2(rpx, rpy, wx, wy) > 0.0f) {
                    ln.dx = (rpx * leg - rpy * R) * inv; ln.dy = (rpx * R + rpy * leg) * inv;
                } else {
                    ln.dx = -((rpx * leg + rpy * R) * inv); ln.dy = -((-rpx * R + rpy * leg) * inv);
                }
                const float dp2 = rvx * ln.dx + rvy * ln.dy;
                ux = dp2 * ln.dx - rvx; uy = dp2 * ln.dy - rvy;
            }
        } else {
            const float inv_dt = 1.0f / (float)cfg.time_step;
            const float wx = rvx - inv_dt * rpx, wy = rvy - inv_dt * rpy;
            const float wl = sqrtf(wx * wx + wy * wy);
            const float inv = 1.0f / wl;
            const float uwx = wx * inv, uwy = wy * inv;
            ln.dx = uwy; ln.dy = -uwx;
            const float sc = R * inv_dt - wl;
            ux = sc * uwx; uy = sc * uwy;
        }
        ln.px = me.z + 0.5f * ux; ln.py = me.w + 0.5f * uy;
        s_scratch[rank] = make_float4(ln.px, ln.py, ln.dx, ln.dy);
    }
    __syncwarp(g.gmask);
    const bool valid = g.gl < n;
    if (valid) { const float4 t = s_scratch[g.gl]; ln.px = t.x; ln.py = t.y; ln.dx = t.z; ln.dy = t.w; }
    __syncwarp(g.gmask);

    float rx, ry;
    const int fail = lp2_group<G>(g, ln, valid, max_speed, prefx, prefy, false, rx, ry, s_scratch);
    if (fail >= 0) lp3_group<G>(g, ln, n, fail, max_speed, rx, ry, s_scratch, s_scratch + STEP_THREADS);
    return make_float2(rx, ry);
}

// ---------------------------------------------------------------------------------------------- phase A, sequential form
// One THREAD per human: the RVO2 solve exactly as the library runs it (computeNeighbors -> computeNewVelocity ->
// linearProgram2 [-> linearProgram3]), the thread's half-planes kept in shared memory in rank order, slot-major
// (`line a of thread t` = lines[a * stride + t]: conflict-free when the warp is converged).  Used for crowds of more
// than 16 neighbours, where the incremental LP is a long dependent chain and a 32-lane group mostly runs it with one
// useful lane: 32 humans share every issued instruction instead of one.  Same arithmetic, same order -> same bits as
// the group form and oracle/orca_core.h.
struct SmemLines {
    const float4 *p; int stride;
    __device__ __forceinline__ Line operator()(int a) const { const float4 t = p[a * stride]; return Line{t.x, t.y, t.z, t.w}; }
};

template <class LA>
__device__ __forceinline__ bool lp1_seq(const LA &L, int k, float radius, float optx, float opty, bool dir_opt, float &rx, float &ry)
{
    const Line lk = L(k);
    const float dp = lk.px * lk.dx + lk.py * lk.dy;
    const float disc = dp * dp + radius * radius - (lk.px * lk.px + lk.py * lk.py);
    if (disc < 0.0f) return false;
    const float sq = sqrtf(disc);
    float t_left = -dp - sq, t_right = -dp + sq;
    // no early exit inside the loop: t_left only grows and t_right only shrinks, so testing once at the end decides the
    // same way as RVO2's per-line test, and the iterations stay independent (four divisions in flight per thread)
    bool fail = false;
#pragma unroll 4
    for (int j = 0; j < k; ++j) {
        const Line lj = L(j);
        const float den = det2(lk.dx, lk.dy, lj.dx, lj.dy);
        const float num = det2(lj.dx, lj.dy, lk.px - lj.px, lk.py - lj.py);
        if (fabsf(den) <= ORCA_EPS) fail |= num < 0.0f;
        else {
            const float t = num / den;
            if (den >= 0.0f) { if (t < t_right) t_right = t; }
            else             { if (t_left < t) t_left = t; }
        }
    }
    if (fail || t_left > t_right) return false;
    float t;
    if (dir_opt) t = (optx * lk.dx + opty * lk.dy > 0.0f) ? t_right : t_left;
    else {
        t = lk.dx * (optx - lk.px) + lk.dy * (opty - lk.py);
        if (t < t_left) t = t_left; else if (t > t_right) t = t_right;
    }
    rx = lk.px + t * lk.dx; ry = lk.py + t * lk.dy;
    return true;
}

// returns the index of the first line that cannot be satisfied, or n
template <class LA>
__device__ __forceinline__ int lp2_seq(const LA &L, int n, float radius, float optx, float opty, bool dir_opt, float &rx, float &ry)
{
    if (dir_opt) { rx = radius * optx; ry = radius * opty; }
    else if (optx * optx + opty * opty > radius * radius) {
        const float inv = 1.0f / sqrtf(optx * optx + opty * opty);
        rx = radius * (optx * inv); ry = radius * (opty * inv);
    } else { rx = optx; ry = opty; }
    for (int i = 0; i < n; ++i) {
        const Line li = L(i);
        if (det2(li.dx, li.dy, li.px - rx, li.py - ry) > 0.0f) {
            const float tx = rx, ty = ry;
            if (!lp1_seq(L, i, radius, optx, opty, dir_opt, rx, ry)) { rx = tx; ry = ty; return i; }
        }
    }
    return n;
}

// neighbour slot k of human i: the other humans in index order, then the robot (orca.py:99-115); invisible ones are
// replaced by the dummy agent (crowd_sim.py:161-163, 1119-1153)
struct Neighbour { float x, y, vx, vy, rad; };
__device__ __forceinline__ Neighbour fetch_neighbour(const CnConfig &cfg, int i, int k, int H, float4 me, double my_th, bool limited,
                                                     const float4 *s_pv, const float4 *s_gr, float4 rob_pv, float rob_radius)
{
    Neighbour o;
    double raw_r, dummy_r;
    if (k < H - 1) {
        const int j = k + (k >= i ? 1 : 0);
        const float4 p = s_pv[j];
        o.x = p.x; o.y = p.y; o.vx = p.z; o.vy = p.w; raw_r = (double)s_gr[j].z; dummy_r = cfg.human_radius;
    } else {
        o.x = rob_pv.x; o.y = rob_pv.y; o.vx = rob_pv.z; o.vy = rob_pv.w; raw_r = (double)rob_radius; dummy_r = cfg.robot_radius;
    }
    if (limited && !detect_visible_d(cfg.kinematics, me.x, me.y, me.z, me.w, my_th, o.x, o.y, cfg.human_fov)) {
        raw_r = dummy_r; o.x = 7.0f; o.y = 7.0f; o.vx = 0.0f; o.vy = 0.0f;
    }
    o.rad = (float)(raw_r + 0.01 + (double)cfg.orca_safety_space);
    return o;
}

// computeNewVelocity's half-plane against one neighbour (RVO2 Agent.cpp, restated in oracle/orca_core.h)
__device__ __forceinline__ float4 orca_half_plane(const CnConfig &cfg, float4 me, float radius, const Neighbour &o)
{
    Line ln;
    const float rpx = o.x - me.x, rpy = o.y - me.y;
    const float rvx = me.z - o.vx, rvy = me.w - o.vy;
    const float dsq = rpx * rpx + rpy * rpy;
    const float R = radius + o.rad;
    const float R2 = R * R;
    float ux, uy;
    if (dsq > R2) {
        const float inv_tau = 1.0f / cfg.orca_time_horizon;
        const float wx = rvx - inv_tau * rpx, wy = rvy - inv_tau * rpy;
        const float wl2 = wx * wx + wy * wy;
        const float dp1 = wx * rpx + wy * rpy;
        if (dp1 < 0.0f && dp1 * dp1 > R2 * wl2) {
            const float wl = sqrtf(wl2);
            const float inv = 1.0f / wl;
            const float uwx = wx * inv, uwy = wy * inv;
            ln.dx = uwy; ln.dy = -uwx;
            const float sc = R * inv_tau - wl;
            ux = sc * uwx; uy = sc * uwy;
        } else {
            const float leg = sqrtf(dsq - R2);
            const float inv = 1.0f / dsq;
            if (det2(rpx, rpy, wx, wy) > 0.0f) {
                ln.dx = (rpx * leg - rpy * R) * inv; ln.dy = (rpx * R + rpy * leg) * inv;
            } else {
                ln.dx = -((rpx * leg + rpy * R) * inv); ln.dy = -((-rpx * R + rpy * leg) * inv);
            }
            const float dp2 = rvx * ln.dx + rvy * ln.dy;
            ux = dp2 * ln.dx - rvx; uy = dp2 * ln.dy - rvy;
        }
    } else {
        const float inv_dt = 1.0f / (float)cfg.time_step;
        const float wx = rvx - inv_dt * rpx, wy = rvy - inv_dt * rpy;
        const float wl = sqrtf(wx * wx + wy * wy);
        const float inv = 1.0f / wl;
        const float uwx = wx * inv, uwy = wy * inv;
        ln.dx = uwy; ln.dy = -uwx;
        const float sc = R * inv_dt - wl;
        ux = sc * uwx; uy = sc * uwy;
    }
    return make_float4(me.z + 0.5f * ux, me.w + 0.5f * uy, ln.dx, ln.dy);
}

// One human's ORCA solve by one thread up to linearProgram2.  lines / keys: this thread's column of the slot-major shared
// arrays.  fail < n_lines: the LP is infeasible from line `fail` on and the caller hands the human to linearProgram3.
__device__ __forceinline__ float2 orca_thread(const CnConfig &cfg, int i, int H, const float4 *s_pv, const float4 *s_gr,
                                              const float *s_th, float2 pref, float4 rob_pv, float rob_radius,
                                              float4 *lines, int *keys, int stride, int &n_lines, int &fail)
{
    const float4 me = s_pv[i];
    const float4 me_g = s_gr[i];
    const float radius = (float)((double)me_g.z + 0.01 + (double)cfg.orca_safety_space);
    const float max_speed = me_g.w;
    const int M = H - 1 + (cfg.robot_visible ? 1 : 0);
    const bool limited = cfg.human_fov < 2.0 * CN_PI;
    const double my_th = (limited && cfg.kinematics != CN_HOLONOMIC) ? (double)s_th[i] : 0.0;
    const float range_sq = cfg.orca_neighbor_dist * cfg.orca_neighbor_dist;

    // computeNeighbors: everyone strictly inside neighborDist; the sort key is the bit pattern of distSq (>= +0)
    int n = 0;
    for (int k = 0; k < M; ++k) {
        const Neighbour o = fetch_neighbour(cfg, i, k, H, me, my_th, limited, s_pv, s_gr, rob_pv, rob_radius);
        const float ddx = me.x - o.x, ddy = me.y - o.y;
        const float dist_sq = ddx * ddx + ddy * ddy;
        const bool in = dist_sq < range_sq;
        keys[k * stride] = in ? __float_as_int(dist_sq) : 0x7fffffff;
        n += in ? 1 : 0;
    }
    // rank = number of in-range neighbours that sort before this one in (distSq, index) order = RVO2's stable insertion
    for (int k = 0; k < M; ++k) {
        const int key = keys[k * stride];
        if (key == 0x7fffffff) continue;
        int rank = 0;
        for (int j = 0; j < k; ++j) rank += (keys[j * stride] <= key) ? 1 : 0;
        for (int j = k + 1; j < M; ++j) rank += (keys[j * stride] < key) ? 1 : 0;
        const Neighbour o = fetch_neighbour(cfg, i, k, H, me, my_th, limited, s_pv, s_gr, rob_pv, rob_radius);
        lines[rank * stride] = orca_half_plane(cfg, me, radius, o);
    }

    float rx, ry;
    const SmemLines L{lines, stride};
    fail = lp2_seq(L, n, max_speed, pref.x, pref.y, false, rx, ry);
    n_lines = n;
    return make_float2(rx, ry);
}

// ---------------------------------------------------------------------------------------------- phase B helpers
__device__ __forceinline__ void velocity_rect_d(double px, double py, double vx, double vy, double radius, double q[4][2])
{
    const double w = 2.0 * radius * 1.0;
    const double L = 3.0 * sqrt(vx * vx + vy * vy);
    const double heading = atan2(vy, vx);
    const double dth = heading - CN_PI / 2.0;
    const double xos = px + radius * cos(heading);
    const double yos = py + radius * sin(heading);
    double c = cos(dth), s = sin(dth);
    if (fabs(c) < 2.5e-16) c = 0.0;
    if (fabs(s) < 2.5e-16) s = 0.0;
    const double bx[4] = {w / 2, w / 2, -w / 2, -w / 2};
    const double by[4] = {-L / 2, L / 2, L / 2, -L / 2};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const double x = bx[k] + 0.0, y = by[k] + L / 2;
        const double xr = c * x + (-s) * y + 0.0;
        const double yr = s * x + c * y + 0.0;
        q[k][0] = xr + xos; q[k][1] = yr + yos;
    }
}

__device__ __forceinline__ bool rects_intersect_d(const double a[4][2], const double b[4][2])
{
#pragma unroll
    for (int which = 0; which < 2; ++which) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const double p0x = which ? b[k][0] : a[k][0], p0y = which ? b[k][1] : a[k][1];
            const double p1x = which ? b[(k + 1) & 3][0] : a[(k + 1) & 3][0];
            const double p1y = which ? b[(k + 1) & 3][1] : a[(k + 1) & 3][1];
            const double ax = -(p1y - p0y), ay = p1x - p0x;
            double a0 = INFINITY, a1 = -INFINITY, b0 = INFINITY, b1 = -INFINITY;
#pragma unroll
            for (int m = 0; m < 4; ++m) {
                const double va = a[m][0] * ax + a[m][1] * ay;
                const double vb = b[m][0] * ax + b[m][1] * ay;
                a0 = va < a0 ? va : a0; a1 = va > a1 ? va : a1;
                b0 = vb < b0 ? vb : b0; b1 = vb > b1 ? vb : b1;
            }
            if (a1 < b0 || b1 < a0) return false;
        }
    }
    return true;
}

__device__ __forceinline__ bool inside_world_d(double px, double py, double r, double t)
{
    const double wx[5] = {-t, t, t, -t, -t};
    const double wy[5] = {-t, -t, t, t, -t};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const double ax = wx[k], ay = wy[k];
        const double dx = wx[k + 1] - ax, dy = wy[k + 1] - ay;
        const double l2 = dx * dx + dy * dy;
        double tt = ((px - ax) * dx + (py - ay) * dy) / l2;
        tt = tt < 0.0 ? 0.0 : (tt > 1.0 ? 1.0 : tt);
        const double cx = ax + tt * dx, cy = ay + tt * dy;
        const double d2 = (px - cx) * (px - cx) + (py - cy) * (py - cy);
        if (d2 <= r * r) return false;
    }
    return true;
}

// ---- exact-by-construction pre-filters of the env tail.  The reference evaluates these predicates through long fp64 chains
// (atan2 / cos / sin / acos, crowd_sim.py:820-847, helper.py:199-231); a cheap fp32 evaluation of the same GEOMETRY decides them
// whenever the result is clear of the decision boundary by a margin far larger than its own error, and only the (rare) cases
// inside the margin run the exact chain -- so every flag is the one the exact chain gives.
struct QuickRect { float cx, cy, dx, dy, half_len, r; bool ok; };

// VelocityRectangle of an agent as centre, unit direction, half length and half width (helper.py:199-231: width 2 r, length
// 3 |v|, starting at the agent's front point p + r d; heading atan2(vy, vx), i.e. d = (1, 0) for v = (+0, +0))
__device__ __forceinline__ QuickRect quick_rect(float px, float py, float vx, float vy, float r)
{
    QuickRect q;
    q.r = r; q.ok = true; q.dx = 1.0f; q.dy = 0.0f; q.half_len = 0.0f;
    const float l2 = vx * vx + vy * vy;
    if (vx == 0.0f && vy == 0.0f) q.ok = !(signbit(vx) || signbit(vy));     // atan2 of a signed zero may be +-pi: exact path
    else if (!(l2 > 1e-20f) || !(l2 < 1e20f)) q.ok = false;
    else { const float inv = rsqrtf(l2); q.dx = vx * inv; q.dy = vy * inv; q.half_len = 1.5f * l2 * inv; }
    q.cx = px + (r + q.half_len) * q.dx;
    q.cy = py + (r + q.half_len) * q.dy;
    return q;
}

// +1: the two rectangles surely intersect, -1: surely disjoint, 0: within 1e-3 of touching (or degenerate input): run the exact
// test.  Separating-axis test on the four unit edge directions; coordinates are a few metres, fp32 error < 1e-5.
__device__ __forceinline__ int quick_rects_intersect(const QuickRect &a, const QuickRect &b)
{
    if (!(a.ok && b.ok)) return 0;
    const float m = 1e-3f;
    const float ex = b.cx - a.cx, ey = b.cy - a.cy;
    const float dd = fabsf(a.dx * b.dx + a.dy * b.dy), dn = fabsf(a.dx * b.dy - a.dy * b.dx);     // |d_a.d_b| = |n_a.n_b|, |d_a.n_b| = |n_a.d_b|
    const float g0 = fabsf(ex * a.dx + ey * a.dy) - (a.half_len + b.half_len * dd + b.r * dn);    // axis d_a
    const float g1 = fabsf(ey * a.dx - ex * a.dy) - (a.r + b.half_len * dn + b.r * dd);           // axis n_a
    const float g2 = fabsf(ex * b.dx + ey * b.dy) - (b.half_len + a.half_len * dd + a.r * dn);    // axis d_b
    const float g3 = fabsf(ey * b.dx - ex * b.dy) - (b.r + a.half_len * dn + a.r * dd);           // axis n_b
    const float gmax = fmaxf(fmaxf(g0, g1), fmaxf(g2, g3));
    if (gmax > m) return -1;
    if (gmax < -m) return 1;
    return 0;
}

// detect_visible (crowd_sim.py:820-847) of point 2 from agent 1 whose unit heading (hx, hy) is known to ~1e-6:
// +1 visible, -1 not visible, 0 undecided (within 1e-4 of the FOV boundary in cosine space, or a degenerate heading)
__device__ __forceinline__ int quick_visible(float hx, float hy, bool heading_ok, float p1x, float p1y, float p2x, float p2y, float cos_half_fov)
{
    const float dx = p2x - p1x, dy = p2y - p1y;
    if (dx == 0.0f && dy == 0.0f) return -1;                 // coincident: the reference's nan <= fov / 2 is False
    const float l2 = dx * dx + dy * dy;
    if (!heading_ok || !(l2 > 1e-20f)) return 0;
    const float c = (hx * dx + hy * dy) * rsqrtf(l2);
    if (c > cos_half_fov + 1e-4f) return 1;
    if (c < cos_half_fov - 1e-4f) return -1;
    return 0;
}

// does goal (gx,gy) of human i come within min_dist of any other agent's position or goal (crowd_sim.py:750-759)
// (kOpt builds, group environment: check_collision_group instead, crowd_sim.py:747-748, 792-793)
template <bool kOpt>
__device__ __forceinline__ bool goal_collides(const CnConfig &cfg, int H, int i, double gx, double gy, const float4 *s_pv,
                                              const float4 *s_gr, float4 rob_pv, float4 rob_gr, const float4 *grp)
{
    if (kOpt && cfg.group_human) return collides_with_groups(grp, gx, gy, (double)s_gr[i].z, 2 * 0.5, s_pv, s_gr, H, true);
    const double ri = (double)s_gr[i].z, dd = cfg.discomfort_dist;
    {
        const double md = ri + (double)rob_gr.z + dd;
        if (norm2d_lt(gx - (double)rob_pv.x, gy - (double)rob_pv.y, md) ||
            norm2d_lt(gx - (double)rob_gr.x, gy - (double)rob_gr.y, md)) return true;
    }
    // fp32 pass over the other humans (positions and goals are stored as floats): a squared distance outside a 1e-4 band around
    // the threshold decides the fp64 rule for certain (fp32 error of the squared distance < 1e-5 relative there); the exact rule
    // only runs for a candidate that lands inside some band without a certain hit
    const float gxf = (float)gx, gyf = (float)gy, rdf = (float)(ri + dd);
    bool hit = false, band = false;
    for (int k = 0; k < H; ++k) {
        if (k == i) continue;
        const float4 p = s_pv[k], q = s_gr[k];
        const float md = rdf + q.z, md2 = md * md, lo = md2 * (1.0f - 1e-4f), hi = md2 * (1.0f + 1e-4f);
        const float ax = gxf - p.x, ay = gyf - p.y, bx = gxf - q.x, by = gyf - q.y;
        const float sa = ax * ax + ay * ay, sb = bx * bx + by * by;
        hit |= (md > 0.0f) & ((sa < lo) | (sb < lo));
        band |= !(md > 1e-3f) | ((sa >= lo) & (sa <= hi)) | ((sb >= lo) & (sb <= hi));
    }
    if (hit) return true;
    if (!band) return false;
    for (int k = 0; k < H; ++k) {
        if (k == i) continue;
        const float4 p = s_pv[k], q = s_gr[k];
        const double md = ri + (double)q.z + dd;
        if (norm2d_lt(gx - (double)p.x, gy - (double)p.y, md) || norm2d_lt(gx - (double)q.x, gy - (double)q.y, md)) return true;
    }
    return false;
}

// Episode over: replace the env's state by its spare episode (= what crowd_reset_kernel would produce from these
// counters, crowd_reset.cu) and write the reset observation; a missing or stale spare is left to the synchronous
// fall-back launched after this kernel.  One warp per env.
__device__ __noinline__ void swap_in_spare(const EnvParams &P, const CnStepOut &out, int e, int lane, int4 ctr)
{
    const CnConfig &cfg = P.cfg;
    const int H = cfg.human_num;
    const int4 meta = P.a.sp_meta[e];
    __syncwarp();          // lane 0's goal writes in env_tail are ordered before the other lanes' writes below
    if (meta.x == 1 && meta.y == ctr.z && meta.z == ctr.y) {
        if (lane < H) {
            const size_t hi = (size_t)e * H + lane;
            P.a.hum_pv[hi] = P.a.sp_pv[hi];
            P.a.hum_gr[hi] = P.a.sp_gr[hi];
            P.a.hum_th[hi] = P.a.sp_th[hi];
        }
        if (cfg.group_human && lane < CN_MAX_GROUPS) P.a.grp[(size_t)e * CN_MAX_GROUPS + lane] = P.a.sp_grp[(size_t)e * CN_MAX_GROUPS + lane];
        const float4 npv = P.a.sp_rob_pv[e], ngr = P.a.sp_rob_gr[e];
        const float nth = P.a.sp_theta[e];
        ctr.x = 0;
        ctr.z = (int)(uint32_t)(((uint64_t)(uint32_t)ctr.z + (uint64_t)cfg.nenv) % cfg.case_size);
        ctr.w = meta.w;
        ctr.y += 1;
        __syncwarp();
        write_reset_obs(P, out.obs, e, lane, H, npv, ngr, nth, true);
        if (lane == 0) {
            float4 nx;
            nx.x = nth;
            nx.y = 0.0f;
            nx.z = (float)(-fabs(norm2d((double)npv.x - (double)ngr.x, (double)npv.y - (double)ngr.y)));
            nx.w = 0.0f;
            P.a.rob_pv[e] = npv;
            P.a.rob_gr[e] = ngr;
            P.a.rob_x[e] = nx;
            P.a.ctr[e] = ctr;
            P.a.sp_meta[e] = make_int4(0, 0, 0, 0);
            // (the list holds n_envs entries: if nobody ran the refill for many steps the surplus is dropped and those envs
            //  simply take the synchronous fall-back at their next reset)
            const int slot = atomicAdd(&P.a.sync_count[2], 1);
            if (slot < P.n_envs) P.a.refill_list[slot] = e;
        }
    } else if (lane == 0) {
        P.a.need_sync[e] = 1;
        atomicAdd(&P.a.sync_count[0], 1);
    }
}

// one warp finishes one env: reward/done/info, integration, observation, goal updates
template <bool kOpt>
__device__ __forceinline__ void env_tail(const EnvParams &P, const CnStepOut &out, const float *__restrict__ action, int e,
                                         int lane, float4 *s_pv, float4 *s_gr, const float2 *s_nv, int auto_reset)
{
    const CnConfig &cfg = P.cfg;
    const int H = cfg.human_num;
    const unsigned FULL = 0xffffffffu;
    const double dt = cfg.time_step;
    float4 rpv = P.a.rob_pv[e];
    float4 rgr = P.a.rob_gr[e];
    float4 rx = P.a.rob_x[e];          // theta, desired_v, potential, episode_return
    float2 racc = P.a.rob_acc[e];
    int4 ctr = P.a.ctr[e];

    // ---- clip_action in float32 (srnn.py:18-48)
    float a0 = action[2 * (size_t)e], a1 = action[2 * (size_t)e + 1];
    double act_v = 0.0, act_r = 0.0, avx, avy;
    if (cfg.kinematics == CN_HOLONOMIC) {
        const float nrm = sqrtf(a0 * a0 + a1 * a1);
        if (nrm > rgr.w) { a0 = a0 / nrm * rgr.w; a1 = a1 / nrm * rgr.w; }
        avx = a0; avy = a1;
    } else {
        a0 = fminf(fmaxf(a0, -0.1f), 0.1f);
        a1 = fminf(fmaxf(a1, -0.1f), 0.1f);
        double dv = (double)rx.y + (double)a0;
        const double vp = rgr.w;
        dv = dv < -vp ? -vp : (dv > vp ? vp : dv);
        rx.y = (float)dv;
        act_v = (double)rx.y; act_r = (double)a1;
        avx = act_v * cos((double)rx.x + act_r);     // patch P1 velocity for SM4/SM5
        avy = act_v * sin((double)rx.x + act_r);
    }

    // ---- calc_reward on the pre-step state; lane i <-> human i
    const bool act = lane < H;
    const float4 hpv = act ? s_pv[lane] : make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 hgr = act ? s_gr[lane] : make_float4(0.f, 0.f, 0.f, 0.f);
    const double hdx = (double)hpv.x - (double)rpv.x, hdy = (double)hpv.y - (double)rpv.y;
    const double closest = sqrt(hdx * hdx + hdy * hdy) - (double)hgr.z - (double)rgr.z;
    const unsigned cbits = __ballot_sync(FULL, act && closest < 0.0);
    const int first_coll = cbits ? (__ffs(cbits) - 1) : H;
    const bool collision = cbits != 0u;
    const bool counted = act && lane < first_coll;
    double dmin = counted ? closest : (double)INFINITY;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double other = shfl_d(FULL, dmin, lane ^ o);
        dmin = other < dmin ? other : dmin;
    }
    // SM2 (crowd_sim.py:962-967): do the velocity rectangles of the robot and of human `lane` intersect
    bool rects_hit = false;
    if (counted) {
        const int quick = quick_rects_intersect(quick_rect(rpv.x, rpv.y, rpv.z, rpv.w, rgr.z), quick_rect(hpv.x, hpv.y, hpv.z, hpv.w, hgr.z));
        if (quick != 0) rects_hit = quick > 0;
        else {
            double rvr[4][2], hvr[4][2];
            velocity_rect_d(rpv.x, rpv.y, rpv.z, rpv.w, rgr.z, rvr);
            velocity_rect_d(hpv.x, hpv.y, hpv.z, hpv.w, hgr.z, hvr);
            rects_hit = rects_intersect_d(rvr, hvr);
        }
    }
    const int vec_viol = __popc(__ballot_sync(FULL, rects_hit));
    const bool h_reached = norm2d_lt((double)hpv.x - (double)hgr.x, (double)hpv.y - (double)hgr.y, (double)hgr.z);
    int agg_nav = __popc(__ballot_sync(FULL, counted && !h_reached));
    const double dgoal = norm2d((double)rpv.x - (double)rgr.x, (double)rpv.y - (double)rgr.y);
    const bool reaching_goal = dgoal < (double)rgr.z;
    if (!reaching_goal) agg_nav += 1;

    // ---- robot end pose (agent.py:172-212)
    double npx, npy, nth = rx.x, nvx, nvy;
    if (cfg.kinematics == CN_HOLONOMIC) {
        npx = (double)rpv.x + avx * dt; npy = (double)rpv.y + avy * dt; nvx = avx; nvy = avy;
    } else {
        double Rr;
        if (fabs(act_r) < 0.0001) Rr = 0.0;
        else { const double w = act_r / dt; Rr = act_v / w; }
        const double th = rx.x;
        npx = (double)rpv.x - Rr * sin(th) + Rr * sin(th + act_r);
        npy = (double)rpv.y + Rr * cos(th) - Rr * cos(th + act_r);
        nth = fmod(th + act_r, 2.0 * CN_PI);
        if (nth < 0.0) nth += 2.0 * CN_PI;
        nvx = act_v * cos(nth); nvy = act_v * sin(nth);
    }

    // ---- step_info (crowd_sim.py:973-1030)
    float side_left = 0.f, side_right = 0.f, separation = 0.f;
    if (cfg.side_preference) {
        const float4 h0 = s_pv[0];
        const float4 g0 = s_gr[0];
        if (npy <= (double)h0.y + (double)g0.z && npy >= (double)h0.y - (double)g0.z) {
            if (npx < (double)h0.x) side_left = 1.f; else side_right = 1.f;
        }
        separation = (float)norm2d((double)h0.x - (double)rpv.x, (double)h0.y - (double)rpv.y);
    }
    const double ax = avx - (double)rpv.z, ay = avy - (double)rpv.w;
    const double dax = ax - (double)racc.x, day = ay - (double)racc.y;
    const float jerk = (float)(dax * dax + day * day);
    racc.x = (float)ax; racc.y = (float)ay;
    // check_inside_world (helper.py:42-55): clear of every wall by more than 1e-6 -> inside without the segment distances
    bool inside = true;
    {
        const double half = cfg.square_width / 2.0;
        const double reach = fmax(fabs((double)rpv.x), fabs((double)rpv.y)) + (double)rgr.z;
        if (!(reach < half - 1e-6)) inside = inside_world_d(rpv.x, rpv.y, rgr.z, half);
    }
    const float speed_viol = (sqrt(avx * avx + avy * avy) > cfg.max_walking_speed) ? 1.f : 0.f;

    // ---- reward / done / event (crowd_sim.py:1032-1092)
    double reward;
    int done, event;
    const int s = ctr.x;
    if (s >= cfg.timeout_step) { reward = 0.0; done = 1; event = CN_EV_TIMEOUT; }
    else if (collision || !inside) { reward = cfg.collision_penalty; done = 1; event = CN_EV_COLLISION; }
    else if (reaching_goal) {
        reward = cfg.success_reward;
        if (cfg.time_factor) reward *= (cfg.time_limit - (double)s * dt) / cfg.time_limit;
        done = 1; event = CN_EV_REACH_GOAL;
    } else if (dmin < cfg.discomfort_dist) {
        reward = (dmin - cfg.discomfort_dist) * cfg.discomfort_penalty_factor; done = 0; event = CN_EV_DANGER;
    } else {
        reward = 0.0;
        if (cfg.potential_based) {
            reward = cfg.potential_factor * (-fabs(dgoal) - (double)rx.z);
            rx.z = (float)(-fabs(dgoal));
        } else if (cfg.exponential) {
            reward = cfg.exp_factor * (1.0 - pow(dgoal / cfg.exp_denom, 0.4));
        }
        done = 0; event = CN_EV_NOTHING;
    }
    if (cfg.kinematics == CN_UNICYCLE) {
        const double r_spin = -2.0 * act_r * act_r;
        const double r_back = (act_v < 0.0) ? -2.0 * fabs(act_v) : 0.0;
        reward = reward + r_spin + r_back;
    }

    // ---- apply the actions; the state holds float32
    rpv = make_float4((float)npx, (float)npy, (float)nvx, (float)nvy);
    rx.x = (float)nth;
    float4 npv = hpv;
    if (act) {
        const float2 nv = s_nv[lane];
        npv = make_float4((float)((double)hpv.x + (double)nv.x * dt), (float)((double)hpv.y + (double)nv.y * dt), nv.x, nv.y);
        s_pv[lane] = npv;
        P.a.hum_pv[(size_t)e * H + lane] = npv;
    }
    ctr.x = s + 1;
    __syncwarp();

    // ---- generate_ob: FOV mask, belief, observation (crowd_sim_dict.py:72-103)
    bool vis = false;
    // the robot's unit heading for the quick FOV test: v / |v| (holonomic: atan2(vy, vx)) or (cos, sin) of theta, in fp32
    float fov_hx = 1.0f, fov_hy = 0.0f, fov_cos = 0.0f;
    bool fov_ok = false;
    if (cfg.robot_fov < 2.0 * CN_PI) {
        fov_cos = cosf((float)(cfg.robot_fov / 2.0));
        if (cfg.kinematics == CN_HOLONOMIC) {
            const float l2 = rpv.z * rpv.z + rpv.w * rpv.w;
            if (rpv.z == 0.0f && rpv.w == 0.0f) fov_ok = !(signbit(rpv.z) || signbit(rpv.w));
            else if (l2 > 1e-20f && l2 < 1e20f) { const float inv = rsqrtf(l2); fov_hx = rpv.z * inv; fov_hy = rpv.w * inv; fov_ok = true; }
        } else {
            sincosf(rx.x, &fov_hy, &fov_hx);
            fov_ok = fabsf(rx.x) < 1e4f;
        }
    }
    if (act) {
        if (cfg.robot_fov >= 2.0 * CN_PI) vis = !((double)npv.x - (double)rpv.x == 0.0 && (double)npv.y - (double)rpv.y == 0.0);
        else {
            const int quick = quick_visible(fov_hx, fov_hy, fov_ok, rpv.x, rpv.y, npv.x, npv.y, fov_cos);
            vis = quick != 0 ? quick > 0
                             : detect_visible_d(cfg.kinematics, rpv.x, rpv.y, rpv.z, rpv.w, rx.x, npv.x, npv.y, cfg.robot_fov);
        }
        const size_t hi = (size_t)e * H + lane;
        float4 bel;
        if (vis) { bel = npv; P.a.hum_br[hi] = hgr.z; }
        else {
            bel = P.a.hum_bel[hi];
            bel.x = (float)((double)bel.x + (double)bel.z * dt);
            bel.y = (float)((double)bel.y + (double)bel.w * dt);
        }
        P.a.hum_bel[hi] = bel;
        reinterpret_cast<float2 *>(out.obs.spatial_edges)[hi] =
            make_float2((float)((double)bel.x - (double)rpv.x), (float)((double)bel.y - (double)rpv.y));
    }
    const unsigned vis_bits = __ballot_sync(FULL, vis);
    if (lane < 7) {
        const float v = lane == 0 ? rpv.x : lane == 1 ? rpv.y : lane == 2 ? rgr.z : lane == 3 ? rgr.x
                      : lane == 4 ? rgr.y : lane == 5 ? rgr.w : rx.x;
        out.obs.robot_node[(size_t)e * 7 + lane] = v;
    } else if (lane < 9) {
        out.obs.temporal_edges[(size_t)e * 2 + (lane - 7)] = lane == 7 ? rpv.z : rpv.w;
    }

    // ---- goal re-sampling (crowd_sim_dict.py:261-269; crowd_sim.py:724-811), bounded tries, lane t <-> try t
    unsigned changed = 0u;
    const float4 *grp = P.a.grp + (size_t)e * CN_MAX_GROUPS;      // group environment only (kOpt builds)
    const uint32_t su = (uint32_t)ctr.x;
    const uint64_t key = step_key(cfg, ctr.y, e);
    if (cfg.random_goal_changing && su < 32u * CN_STEP_TABLE_WORDS && ((cfg.goal_change_steps[su >> 5] >> (su & 31)) & 1u)) {
        for (int i = 0; i < H; ++i) {
            const float4 gi = s_gr[i];
            if (gi.w == 0.0f) continue;
            const uint4 dec = philox4x32(key, RNG_DECISION, (uint32_t)i, su, RNG_GOAL_RANDOM);
            if (!(u01(dec.x) <= cfg.goal_change_chance)) continue;
            for (int t0 = 0; t0 < cfg.max_goal_tries; t0 += 32) {
                const int t = t0 + lane;
                const uint4 x = philox4x32(key, (uint32_t)t, (uint32_t)i, su, RNG_GOAL_RANDOM);
                const double angle = u01(x.x) * CN_PI * 2.0;
                const double vp = (double)gi.w;
                const double gx = cfg.circle_radius * cos(angle) + (u01(x.y) - 0.5) * vp;
                const double gy = cfg.circle_radius * sin(angle) + (u01(x.z) - 0.5) * vp;
                const bool ok = t < cfg.max_goal_tries && !goal_collides<kOpt>(cfg, H, i, gx, gy, s_pv, s_gr, rpv, rgr, grp);
                const unsigned okb = __ballot_sync(FULL, ok);
                if (okb) {
                    const int src = __ffs(okb) - 1;
                    const float ngx = (float)shfl_d(FULL, gx, src), ngy = (float)shfl_d(FULL, gy, src);
                    if (lane == 0) {
                        s_gr[i] = make_float4(ngx, ngy, gi.z, gi.w);
                        P.a.hum_gr[(size_t)e * H + i] = make_float4(ngx, ngy, gi.z, gi.w);
                    }
                    changed |= 1u << i;
                    break;
                }
            }
            __syncwarp();
        }
    }
    if (cfg.end_goal_changing) {
        // lane i tests human i (a new goal of an earlier human does not enter a later human's own reached-goal test),
        // the warp then walks the few humans that did reach their goal in index order
        bool reached = false;
        if (lane < H) {
            const float4 pl = s_pv[lane], gl = s_gr[lane];
            reached = norm2d_lt((double)gl.x - (double)pl.x, (double)gl.y - (double)pl.y, (double)gl.z);
        }
        for (unsigned todo = __ballot_sync(FULL, reached); todo; todo &= todo - 1u) {
            const int i = __ffs(todo) - 1;
            float4 gi = s_gr[i];
            const uint4 dec = philox4x32(key, RNG_DECISION, (uint32_t)i, su, RNG_GOAL_END);
            if (!(u01(dec.x) <= cfg.end_goal_change_chance)) continue;
            if (kOpt && (cfg.random_radii | cfg.random_v_pref)) {
                // humans.random_radii / random_v_pref (crowd_sim.py:779-786): the human that gets a new end goal also gets
                // radius / v_pref += uniform(-0.1, 0.1); the goal search below already uses the new values
                if (cfg.random_radii) gi.z = (float)((double)gi.z + (-0.1 + 0.2 * u01(dec.y)));
                if (cfg.random_v_pref) gi.w = (float)((double)gi.w + (-0.1 + 0.2 * u01(dec.z)));
                __syncwarp();
                if (lane == 0) { s_gr[i] = gi; P.a.hum_gr[(size_t)e * H + i] = gi; }
                __syncwarp();
            }
            for (int t0 = 0; t0 < cfg.max_goal_tries; t0 += 32) {
                const int t = t0 + lane;
                const uint4 xa = philox4x32(key, (uint32_t)(2 * t), (uint32_t)i, su, RNG_GOAL_END);
                const uint4 xb = philox4x32(key, (uint32_t)(2 * t + 1), (uint32_t)i, su, RNG_GOAL_END);
                const double u6[6] = {u01(xa.x), u01(xa.y), u01(xa.z), u01(xa.w), u01(xb.x), u01(xb.y)};
                const SpawnCand c = agent_attributes(cfg, ctr.w, (double)gi.z, (double)gi.w, (double)rgr.z, u6);
                const bool ok = t < cfg.max_goal_tries && !goal_collides<kOpt>(cfg, H, i, c.gx, c.gy, s_pv, s_gr, rpv, rgr, grp);
                const unsigned okb = __ballot_sync(FULL, ok);
                if (okb) {
                    const int src = __ffs(okb) - 1;
                    const float ngx = (float)shfl_d(FULL, c.gx, src), ngy = (float)shfl_d(FULL, c.gy, src);
                    if (lane == 0) {
                        s_gr[i] = make_float4(ngx, ngy, gi.z, gi.w);
                        P.a.hum_gr[(size_t)e * H + i] = make_float4(ngx, ngy, gi.z, gi.w);
                    }
                    changed |= 1u << i;
                    break;
                }
            }
            __syncwarp();
        }
    }

    // ---- per-env scalars
    rx.w = (float)((double)rx.w + reward);
    if (lane == 0) {
        P.a.rob_pv[e] = rpv;
        P.a.rob_x[e] = rx;
        P.a.rob_acc[e] = racc;
        P.a.ctr[e] = ctr;
        out.reward[e] = (float)reward;
        out.done[e] = (uint8_t)done;
        if (out.not_done) out.not_done[e] = done ? 0.0f : 1.0f;
        out.event[e] = event;
        if (out.scenario) out.scenario[e] = ctr.w;
        if (out.episode_return) out.episode_return[e] = rx.w;
        if (out.episode_length) out.episode_length[e] = ctr.x;
        if (out.obs.visible_mask) out.obs.visible_mask[e] = vis_bits;
        if (out.goal_changed) out.goal_changed[e] = changed;
    }
    if (out.info && lane < CN_INFO_DIM) {
        float v = 0.f;
        switch (lane) {
        case CN_INFO_DMIN: v = (float)dmin; break;
        case CN_INFO_AGGREGATE_NAV_TIME: v = (float)agg_nav; break;
        case CN_INFO_PATH_VIOLATION: v = (float)vec_viol; break;
        case CN_INFO_PERSONAL_VIOLATION: v = (dmin < cfg.min_personal_space) ? 1.f : 0.f; break;
        case CN_INFO_JERK_COST: v = jerk; break;
        case CN_INFO_DIST_TO_GOAL: v = (float)dgoal; break;
        case CN_INFO_SPEED_VIOLATION: v = speed_viol; break;
        case CN_INFO_SIDE_LEFT: v = side_left; break;
        case CN_INFO_SIDE_RIGHT: v = side_right; break;
        case CN_INFO_SEPARATION: v = separation; break;
        default: break;
        }
        out.info[(size_t)e * CN_INFO_DIM + lane] = v;
    }

    // ---- episode over: swap the pre-generated spare episode in (out of line: it runs for ~3 % of the envs per step and
    // must not cost the common path registers)
    if (done && auto_reset) swap_in_spare(P, out, e, lane, ctr);
}

// ---------------------------------------------------------------------------------------------- the kernel
// grid: ceil(N / E) CTAs of 256 threads, each owning E consecutive envs.
// dynamic smem: E*H*(float4 pv + float4 gr + float2 nv + float th) + 2 x 256 float4 line scratch
// kPhase 0: the whole step in one launch (the default).  kPhase 1 / 2: the same code as TWO launches -- 1 = staging + phase A
// (the new velocities go to hum_nv), 2 = staging (+ hum_nv) + phase B -- behind CN_STEP_SPLIT=1: no faster, but it isolates the
// ORCA solves (issue-bound: 83 % of the issue slots) from the env tail (instruction-fetch and latency bound) in a profile.
#ifndef STEP_TAIL_THREADS
#define STEP_TAIL_THREADS 256       // CTA of the env-tail kernel (kPhase 2): one warp per env
#endif
template <int G, bool kOpt, int kPhase>
__global__ void __launch_bounds__(kPhase == 2 ? STEP_TAIL_THREADS : STEP_THREADS, kPhase == 2 ? (1024 / STEP_TAIL_THREADS) : STEP_MIN_BLOCKS)
crowd_step_kernel(const __grid_constant__ EnvParams P, const __grid_constant__ CnStepOut out,
                  const float *__restrict__ action, int E, int auto_reset)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const CnConfig &cfg = P.cfg;
    const int H = cfg.human_num;
    const int e0 = blockIdx.x * E;
    const int ne = min(E, P.n_envs - e0);
    const int EH = E * H;
    float4 *s_pv = reinterpret_cast<float4 *>(smem_raw);
    float4 *s_gr = s_pv + EH;
    float4 *s_scr = s_gr + EH;
    float2 *s_nv = reinterpret_cast<float2 *>(s_scr + 2 * STEP_THREADS);     // scratch: ranked lines + projected lines of every group
    float *s_th = reinterpret_cast<float *>(s_nv + EH);
    __shared__ float4 s_rob_pv[64];
    __shared__ float2 s_rob_rt[64];   // radius, theta

    // stage: coalesced float4 loads of ne*H consecutive humans
    const size_t base = (size_t)e0 * H;
    const bool need_th = cfg.human_fov < 2.0 * CN_PI && cfg.kinematics != CN_HOLONOMIC;
    const int nthreads = kPhase == 2 ? STEP_TAIL_THREADS : STEP_THREADS;
    for (int k = threadIdx.x; k < ne * H; k += nthreads) {
        const float4 pv = P.a.hum_pv[base + k], gr = P.a.hum_gr[base + k];
        s_pv[k] = pv;
        s_gr[k] = gr;
        if (kPhase == 2) s_nv[k] = P.a.hum_nv[base + k];
        else s_nv[k] = preferred_velocity(pv, gr);      // phase A replaces it with the new velocity of the same human
        if (kPhase != 2 && need_th) s_th[k] = P.a.hum_th[base + k];
    }
    if (kPhase != 2 && cfg.robot_visible) {
        for (int k = threadIdx.x; k < ne; k += STEP_THREADS) {
            s_rob_pv[k] = P.a.rob_pv[e0 + k];
            s_rob_rt[k] = make_float2(P.a.rob_gr[e0 + k].z, P.a.rob_x[e0 + k].x);
        }
    }
    __syncthreads();

    // phase A: ORCA, one G-lane group per (env, human) task
    if (kPhase != 2) {
        GroupOps<G> g;
        const int lane = threadIdx.x & 31;
        g.gl = lane % G;
        g.gbase = lane - g.gl;
        g.gmask = (G == 32) ? 0xffffffffu : (GroupOps<G>::kLow << g.gbase);
        const int group = threadIdx.x / G;
        constexpr int kGroups = STEP_THREADS / G;
        float4 *scratch = s_scr + group * G;
        // (el, i) = divmod(task, H) kept incrementally: one division per thread instead of one per task
        const int step_el = kGroups / H, step_i = kGroups - step_el * H;
        int el = group / H, i = group - el * H;
        for (int task = group; task < ne * H; task += kGroups, el += step_el, i += step_i) {
            if (i >= H) { i -= H; ++el; }
            const float4 rob = cfg.robot_visible ? s_rob_pv[el] : make_float4(0.f, 0.f, 0.f, 0.f);
            const float2 rrt = cfg.robot_visible ? s_rob_rt[el] : make_float2(0.f, 0.f);
            const float2 nv = orca_group<G, kOpt>(cfg, g, i, H, s_pv + el * H, s_gr + el * H, s_th + el * H, s_nv[task], rob, rrt.x, rrt.y,
                                                  scratch, P, e0 + el);
            if (g.gl == 0) s_nv[task] = nv;
        }
    }
    if (kPhase != 2) __syncthreads();
    if (kPhase == 1) {
        for (int k = threadIdx.x; k < ne * H; k += STEP_THREADS) P.a.hum_nv[base + k] = s_nv[k];
        return;
    }

    // phase B: one warp per env
    {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        for (int el = warp; el < ne; el += nthreads / 32)
            env_tail<kOpt>(P, out, action, e0 + el, lane, s_pv + el * H, s_gr + el * H, s_nv + el * H, auto_reset);
    }
}

// The sequential form of phase A (thread per human) around the same staging and phase B.
// dynamic smem: E*H*(float4 pv + float4 gr + float2 nv + float th) + S * M * (float4 line + int key), S = solver threads
#ifndef STEP_SEQ_MIN_BLOCKS
#define STEP_SEQ_MIN_BLOCKS 2
#endif
__global__ void __launch_bounds__(STEP_THREADS, STEP_SEQ_MIN_BLOCKS)
crowd_step_seq_kernel(const __grid_constant__ EnvParams P, const __grid_constant__ CnStepOut out,
                      const float *__restrict__ action, int E, int S, int auto_reset)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const CnConfig &cfg = P.cfg;
    const int H = cfg.human_num;
    const int M = H - 1 + (cfg.robot_visible ? 1 : 0);
    const int e0 = blockIdx.x * E;
    const int ne = min(E, P.n_envs - e0);
    const int EH = E * H;
    float4 *s_pv = reinterpret_cast<float4 *>(smem_raw);
    float4 *s_gr = s_pv + EH;
    float4 *s_lines = s_gr + EH;
    float2 *s_nv = reinterpret_cast<float2 *>(s_lines + S * M);
    int *s_keys = reinterpret_cast<int *>(s_nv + EH);
    float *s_th = reinterpret_cast<float *>(s_keys + S * M);
    __shared__ float4 s_rob_pv[64];
    __shared__ float2 s_rob_rt[64];   // radius, theta
    __shared__ int s_fail[STEP_THREADS];   // queue of humans for linearProgram3: thread | n << 8 | first failed line << 16
    __shared__ float4 s_lp3[STEP_THREADS / 32][2][32];
    __shared__ int s_ctl[3];

    const size_t base = (size_t)e0 * H;
    const bool need_th = cfg.human_fov < 2.0 * CN_PI && cfg.kinematics != CN_HOLONOMIC;
    for (int k = threadIdx.x; k < ne * H; k += STEP_THREADS) {
        const float4 pv = P.a.hum_pv[base + k], gr = P.a.hum_gr[base + k];
        s_pv[k] = pv;
        s_gr[k] = gr;
        s_nv[k] = preferred_velocity(pv, gr);
        if (need_th) s_th[k] = P.a.hum_th[base + k];
    }
    if (cfg.robot_visible) {
        for (int k = threadIdx.x; k < ne; k += STEP_THREADS) {
            s_rob_pv[k] = P.a.rob_pv[e0 + k];
            s_rob_rt[k] = make_float2(P.a.rob_gr[e0 + k].z, P.a.rob_x[e0 + k].x);
        }
    }
    __syncthreads();

    // phase A: thread t < S solves human task0 + t up to linearProgram2.  Humans whose LP is infeasible (common in dense
    // crowds: ~1 in 8 at H = 20) are finished with the lane-parallel linearProgram3 by whole warps -- run by their own
    // thread they would hold the CTA at the barrier for tens of microseconds.  The two run CONCURRENTLY: solver threads
    // push (thread, n, fail) records into a shared-memory queue, and every warp that has no solver thread left (the
    // spare warps from the start, the solver warps as they finish) pops records until the queue is closed and drained.
    const int lane = threadIdx.x & 31;
    volatile int *vctl = s_ctl;
    volatile int *vfail = s_fail;
    for (int task0 = 0; task0 < ne * H; task0 += S) {
        const int todo = min(S, ne * H - task0);
        const int solver_warps = (todo + 31) >> 5;
        s_fail[threadIdx.x] = -1;
        if (threadIdx.x < 3) s_ctl[threadIdx.x] = 0;       // records pushed | records popped | solver warps finished
        __syncthreads();
        if (threadIdx.x < todo) {
            const int task = task0 + threadIdx.x;
            const int el = task / H, i = task - el * H;
            const float4 rob = cfg.robot_visible ? s_rob_pv[el] : make_float4(0.f, 0.f, 0.f, 0.f);
            const float rr = cfg.robot_visible ? s_rob_rt[el].x : 0.f;
            int n, fail;
            s_nv[task] = orca_thread(cfg, i, H, s_pv + el * H, s_gr + el * H, s_th + el * H, s_nv[task], rob, rr,
                                     s_lines + threadIdx.x, s_keys + threadIdx.x, S, n, fail);
            if (fail < n) {
                const int slot = atomicAdd(&s_ctl[0], 1);
                __threadfence_block();                       // lines and the LP2 result before the record
                vfail[slot] = (int)threadIdx.x | (n << 8) | (fail << 16);
            }
        }
        __syncwarp();
        if ((threadIdx.x >> 5) < solver_warps && lane == 0) { __threadfence_block(); atomicAdd(&s_ctl[2], 1); }
        GroupOps<32> g;
        g.gl = lane; g.gbase = 0; g.gmask = 0xffffffffu;
        for (;;) {
            int rec = -1;
            if (lane == 0) {
                const int slot = atomicAdd(&s_ctl[1], 1);
                for (;;) {
                    if (slot < STEP_THREADS) rec = vfail[slot];
                    if (rec >= 0) break;
                    if (vctl[2] >= solver_warps && slot >= vctl[0]) { rec = -2; break; }     // closed and drained
                    __nanosleep(40);
                }
            }
            rec = __shfl_sync(0xffffffffu, rec, 0);
            if (rec < 0) break;
            const int owner = rec & 0xff, n = (rec >> 8) & 0xff, fail = rec >> 16, t = task0 + owner;
            Line ln; ln.px = ln.py = ln.dx = ln.dy = 0.0f;
            float4 (*lp3)[32] = s_lp3[threadIdx.x >> 5];      // this warp's contiguous copy of the lines + projected-line scratch
            __syncwarp();
            if (g.gl < n) { const float4 v = s_lines[g.gl * S + owner]; ln.px = v.x; ln.py = v.y; ln.dx = v.z; ln.dy = v.w; lp3[0][g.gl] = v; }
            __syncwarp();
            float2 r = s_nv[t];
            lp3_group<32>(g, ln, n, fail, s_gr[t].w, r.x, r.y, lp3[0], lp3[1]);
            if (g.gl == 0) s_nv[t] = r;
        }
        __syncthreads();
    }

    // phase B: one warp per env
    for (int el = threadIdx.x >> 5; el < ne; el += STEP_THREADS / 32)
        env_tail<false>(P, out, action, e0 + el, lane, s_pv + el * H, s_gr + el * H, s_nv + el * H, auto_reset);
}

static inline int pick_group(int M)
{
    return M <= 4 ? 4 : (M <= 8 ? 8 : (M <= 16 ? 16 : 32));
}

static bool step_has_options(const CnConfig &c)
{
    return c.human_policy != CN_POLICY_ORCA || c.random_policy_changing || c.random_unobservability || c.random_radii ||
           c.random_v_pref || c.group_human;
}

// launches of one crowd step: 1, or 2 (ORCA kernel + env-tail kernel) with CN_STEP_SPLIT=1 -- a development switch: the two
// forms take the same time (0.433 vs 0.438 ms at 16384 envs x 20 humans) and give the same bits (tests/test_gpu_crowd_step.py
// runs both); the split form is what shows each phase on its own in a profile (profiles/r2_ncu_final_kernels.txt).
extern "C" int cn_crowd_step_launches(const EnvParams *P)
{
    if (step_has_options(P->cfg)) return 1;
    if (const char *dbg = getenv("CN_STEP_SEQ")) if (atoi(dbg) != 0) return 1;
    if (const char *dbg = getenv("CN_STEP_SPLIT")) return atoi(dbg) != 0 ? 2 : 1;
    return 1;
}

// the instantiation of the group form the launcher runs first (the split form's ORCA launch has the same shared memory)
template <int G>
static const void *step_kernel_of(bool opt)
{
    return opt ? (const void *)crowd_step_kernel<G, true, 0> : (const void *)crowd_step_kernel<G, false, 0>;
}

// host launcher (called from c_abi.cu)
extern "C" int cn_launch_crowd_step(const EnvParams *P, const CnStepOut *out, const float *action, int auto_reset, cudaStream_t stream)
{
    const int H = P->cfg.human_num;
    const int M = H - 1 + (P->cfg.robot_visible ? 1 : 0);
    const int G = pick_group(M < 1 ? 1 : M);
    static int num_sms = 0;
    if (num_sms == 0) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev); }
    // CN_STEP_SEQ=1: the thread-per-human form of phase A.  Same bits; measured at 16384 envs x 20 humans it executes 30 %
    // fewer instructions than the group form but is latency-bound at the ~15 solver warps per SM its 400 B of shared memory
    // per human allow, so it is no faster (0.49-0.53 vs 0.51 ms, profiles/README.md) and stays a development switch.
    // the optional human behaviours of SURVEY 8(f) N4 live in their own instantiation of the group form
    const bool opt = step_has_options(P->cfg);
    bool seq = false;
    if (const char *dbg = getenv("CN_STEP_SEQ")) seq = atoi(dbg) != 0 && M >= 1 && M <= 32 && !opt;
    if (seq) {
        int E = STEP_THREADS / H;           // one solve per thread
        E = E < 1 ? 1 : (E > 64 ? 64 : E);
        if (num_sms > 0 && P->n_envs < E * 2 * num_sms) { E = P->n_envs / (2 * num_sms); E = E < 1 ? 1 : E; }
        if (const char *dbg = getenv("CN_STEP_ENVS_PER_CTA")) { const int v = atoi(dbg); if (v >= 1 && v <= 64) E = v; }
        int S = (E * H + 31) & ~31;         // solver threads per pass = columns of the slot-major line / key arrays
        S = S > STEP_THREADS ? STEP_THREADS : S;
        const size_t smem = (size_t)E * H * (16 + 16 + 8 + 4) + (size_t)S * M * (16 + 4);
        static bool attr_set = false;
        if (!attr_set) {
            const cudaError_t rc = cudaFuncSetAttribute(crowd_step_seq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
            if (rc != cudaSuccess) return (int)rc;
            attr_set = true;
        }
        if (smem > 200 * 1024) return (int)cudaErrorInvalidValue;
        const int grid = (P->n_envs + E - 1) / E;
        crowd_step_seq_kernel<<<grid, STEP_THREADS, smem, stream>>>(*P, *out, action, E, S, auto_reset);
        return (int)cudaGetLastError();
    }
    // envs per CTA: ~2 rounds of ORCA groups per CTA, at most 64 (s_rob_* capacity), at least 8 (one tail warp each)
    int E = (2 * (STEP_THREADS / G) + H - 1) / H;
    E = E < 8 ? 8 : (E > 64 ? 64 : E);
    // small batches (BASELINE configs[0], [1]): a CTA is a latency chain of ~E*H/groups solves plus one tail per warp, and
    // there are not enough CTAs to fill the GPU anyway -- spread the envs over at least ~4 CTAs per SM
    if (num_sms > 0 && P->n_envs < E * 4 * num_sms) { E = P->n_envs / (4 * num_sms); E = E < 1 ? 1 : E; }
    if (const char *dbg = getenv("CN_STEP_ENVS_PER_CTA")) {          // tuning knob
        const int v = atoi(dbg);
        if (v >= 1 && v <= 64) E = v;
        // the kernel runs with the default 48 KB shared-memory limit (no cudaFuncSetAttribute: more would change the
        // occupancy of the default shapes), so a value whose E*H humans do not fit beside the kernel's static shared
        // memory is clamped to the largest that does (E = 43 at H = 20, 27 at H = 32; the default E always fits)
        const void *k = G == 4 ? step_kernel_of<4>(opt) : G == 8 ? step_kernel_of<8>(opt) : G == 16 ? step_kernel_of<16>(opt) : step_kernel_of<32>(opt);
        cudaFuncAttributes fa;
        const cudaError_t rc = cudaFuncGetAttributes(&fa, k);
        if (rc != cudaSuccess) return (int)rc;
        const int e_fit = (int)((48 * 1024 - fa.sharedSizeBytes - 2 * STEP_THREADS * 16) / (H * (16 + 16 + 8 + 4)));
        if (E > e_fit) E = e_fit;
    }
    const size_t smem = (size_t)E * H * (16 + 16 + 8 + 4) + 2 * STEP_THREADS * 16;
    const int grid = (P->n_envs + E - 1) / E;
    if (opt) {
        switch (G) {
        case 4: crowd_step_kernel<4, true, 0><<<grid, STEP_THREADS, smem, stream>>>(*P, *out, action, E, auto_reset); break;
        case 8: crowd_step_kernel<8, true, 0><<<grid, STEP_THREADS, smem, stream>>>(*P, *out, action, E, auto_reset); break;
        case 16: crowd_step_kernel<16, true, 0><<<grid, STEP_THREADS, smem, stream>>>(*P, *out, action, E, auto_reset); break;
        default: crowd_step_kernel<32, true, 0><<<grid, STEP_THREADS, smem, stream>>>(*P, *out, action, E, auto_reset); break;
        }
        return (int)cudaGetLastError();
    }
    if (cn_crowd_step_launches(P) == 2) {
        switch (G) {
        case 4: crowd_step_kernel<4, false, 1><<<grid, STEP_THREADS, smem, stream>>>(*P, *out, action, E, auto_reset); break;
        case 8: crowd_step_kernel<8, false, 1><<<grid, STEP_THREADS, smem, stream>>>(*P, *out, action, E, auto_reset); break;
        case 16: crowd_step_kernel<16, false, 1><<<grid, STEP_THREADS, smem, stream>>>(*P, *out, action, E, auto_reset); break;
        default: crowd_step_kernel<32, false, 1><<<grid, STEP_THREADS, smem, stream>>>(*P, *out, action, E, auto_reset); break;
        }
        const int E2 = STEP_TAIL_THREADS / 32;            // one warp per env
        const size_t smem2 = (size_t)E2 * H * (16 + 16 + 8 + 4) + 2 * STEP_THREADS * 16;
        crowd_step_kernel<32, false, 2><<<(P->n_envs + E2 - 1) / E2, STEP_TAIL_THREADS, smem2, stream>>>(*P, *out, action, E2, auto_reset);
        return (int)cudaGetLastError();
    }
    switch (G) {
    case 4: crowd_step_kernel<4, false, 0><<<grid, STEP_THREADS, smem, stream>>>(*P, *out, action, E, auto_reset); break;
    case 8: crowd_step_kernel<8, false, 0><<<grid, STEP_THREADS, smem, stream>>>(*P, *out, action, E, auto_reset); break;
    case 16: crowd_step_kernel<16, false, 0><<<grid, STEP_THREADS, smem, stream>>>(*P, *out, action, E, auto_reset); break;
    default: crowd_step_kernel<32, false, 0><<<grid, STEP_THREADS, smem, stream>>>(*P, *out, action, E, auto_reset); break;
    }
    return (int)cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------- K8: model-based robot
// The action of an ORCA or social-force robot (config robot.policy = orca / social_force): orca.py:64-139 or
// social_force.py:11-63 with the robot as agent 0 and the H rows of last_human_states (hum_bel / hum_br: what the DS-RNN
// observation is built from) as the others, in human index order.  One G-lane group per env, lane k owns belief row k;
// the solve is the humans' own (orca_group), so the arithmetic is the same fp32 / fp64.
// Reads only the running episode's arrays (never the spares the forked refill writes); writes float32 [N, 2].
template <int G, int kAgent>
__global__ void __launch_bounds__(STEP_THREADS)
robot_act_kernel(const __grid_constant__ EnvParams P, float2 *__restrict__ action)
{
    __shared__ __align__(16) float4 s_scr[2 * STEP_THREADS];     // per group: G ranked lines + G projected lines
    const CnConfig &cfg = P.cfg;
    const int H = cfg.human_num;
    GroupOps<G> g;
    const int lane = threadIdx.x & 31;
    g.gl = lane % G;
    g.gbase = lane - g.gl;
    g.gmask = (G == 32) ? 0xffffffffu : (GroupOps<G>::kLow << g.gbase);
    const int group = threadIdx.x / G;
    const int e = blockIdx.x * (STEP_THREADS / G) + group;
    if (e >= P.n_envs) return;                                  // whole groups only: no lane of a live group leaves
    const float4 me = P.a.rob_pv[e];
    const float2 pref = kAgent == AGENT_ROBOT_ORCA ? preferred_velocity(me, P.a.rob_gr[e]) : make_float2(0.f, 0.f);
    const float2 v = orca_group<G, false, kAgent>(cfg, g, 0, H, nullptr, nullptr, nullptr, pref, me, 0.f, 0.f, s_scr + group * G, P, e);
    if (g.gl == 0) action[e] = v;
}

// host launcher (called from c_abi.cu): one launch, no allocation, no synchronisation
extern "C" int cn_launch_robot_act(const EnvParams *P, int policy, float *action, cudaStream_t stream)
{
    const int H = P->cfg.human_num;
    const int G = pick_group(H);
    const int grid = (P->n_envs + STEP_THREADS / G - 1) / (STEP_THREADS / G);
    float2 *out = reinterpret_cast<float2 *>(action);
    if (policy == CN_POLICY_SOCIAL_FORCE) {
        switch (G) {
        case 4: robot_act_kernel<4, AGENT_ROBOT_SF><<<grid, STEP_THREADS, 0, stream>>>(*P, out); break;
        case 8: robot_act_kernel<8, AGENT_ROBOT_SF><<<grid, STEP_THREADS, 0, stream>>>(*P, out); break;
        case 16: robot_act_kernel<16, AGENT_ROBOT_SF><<<grid, STEP_THREADS, 0, stream>>>(*P, out); break;
        default: robot_act_kernel<32, AGENT_ROBOT_SF><<<grid, STEP_THREADS, 0, stream>>>(*P, out); break;
        }
    } else {
        switch (G) {
        case 4: robot_act_kernel<4, AGENT_ROBOT_ORCA><<<grid, STEP_THREADS, 0, stream>>>(*P, out); break;
        case 8: robot_act_kernel<8, AGENT_ROBOT_ORCA><<<grid, STEP_THREADS, 0, stream>>>(*P, out); break;
        case 16: robot_act_kernel<16, AGENT_ROBOT_ORCA><<<grid, STEP_THREADS, 0, stream>>>(*P, out); break;
        default: robot_act_kernel<32, AGENT_ROBOT_ORCA><<<grid, STEP_THREADS, 0, stream>>>(*P, out); break;
        }
    }
    return (int)cudaGetLastError();
}
