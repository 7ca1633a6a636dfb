// render.cu -- K7: rgb_array frames of any subset of envs, rasterised straight from the SoA state in HBM
// (CrowdSim.render, crowd_sim.py:1207-1461, without matplotlib).  sm_100a only.
//
// One CTA fills one band of RENDER_BAND consecutive pixels (row-major, so whole rows or part of one row) of one frame:
//   1. warp 0 stages the env's robot, goal and humans in shared memory and culls the discs against the band's bounding
//      box (lane i <-> human i, one ballot), so a pixel tests O(1) discs instead of H + 2;
//   2. every thread colours 4 consecutive pixels per pass and packs them into 3 32-bit words in shared memory;
//   3. the band, contiguous in the output, is stored with 16-byte coalesced stores.
// At large batches the kernel is bound by its HBM writes (3 S^2 bytes per frame).
//
// All geometry is fp32 in a fixed operation order and built with -fmad=false (ENV_SRC), so that the tests' numpy
// restatement (render_oracle.py) can repeat every predicate bit for bit:
//   pixel centre   x_j = ((float)j + 0.5f) * scale - half,  y_i = half - ((float)i + 0.5f) * scale
//                  scale = (float)(L / S), half = (float)(L * 0.5), L = sim.square_width (the world of check_inside_world)
//   disc           dx = x - cx, dy = y - cy:  dx * dx + dy * dy <= r * r
//   wedge / sector a = dx * fx + dy * fy, c = |dy * fx - dx * fy|:  cos(h) * c <= sin(h) * a   (angle to f <= h, h < pi)
//   heading f      unicycle (cos th, sin th) rounded from fp64; holonomic (vx, vy) / |(vx, vy)|, (1, 0) at zero speed
//                  (detect_visible's atan2(0, 0) = 0)
//
// Graph capture / concurrency: the kernel allocates nothing and never synchronises.  It reads only the running episode's
// arrays (rob_pv, rob_gr, rob_x, hum_pv, hum_gr), never the spare-episode arrays (sp_*) that the refill forked by
// cn_env_step / cn_env_reset writes on the library's side stream, so it may run on the caller's stream while a refill is
// still in flight: no join is needed and none is made.  The running arrays are only written on the caller's stream
// (step kernel, synchronous reset fall-back, set_state), which orders them against the render.
#include "env_common.cuh"

#define RENDER_THREADS 256
#define RENDER_PIX_PER_THREAD 8                                   // two passes of 4 consecutive pixels
#define RENDER_BAND (RENDER_THREADS * RENDER_PIX_PER_THREAD)      // 2048 pixels = 6144 bytes per CTA

struct RenderView {
    float scale, half;        // pixel size, L / 2
    float fov_c, fov_s;       // cos / sin of half the robot's FOV
    float head_c, head_s;     // cos / sin of CN_RENDER_HEADING_HALF
    int draw_fov;             // robot.FOV < 2
};

struct RenderEnv {
    float rx, ry, rr2, fx, fy, gx, gy;
    unsigned live;            // bit i: human i may touch the band
    int draw_goal, draw_robot;
    float4 hum[CN_MAX_HUMANS];   // cx, cy, r * r, inside FOV (1 / 0)
};

// does a disc (cx, cy, r) come within one pixel of the band's pixel centres?  Generous on purpose: it only culls
__device__ __forceinline__ bool disc_near(float cx, float cy, float r, float x_lo, float x_hi, float y_lo, float y_hi, float slack)
{
    const float s = r + slack + 1e-5f * (fabsf(cx) + fabsf(cy) + fabsf(r));
    return cx + s >= x_lo && cx - s <= x_hi && cy + s >= y_lo && cy - s <= y_hi;
}

__device__ __forceinline__ bool in_disc(float x, float y, float cx, float cy, float r2)
{
    const float dx = x - cx, dy = y - cy;
    return dx * dx + dy * dy <= r2;
}

// angle between (x, y) - (ox, oy) and the unit vector f is <= h (c_h = cos h, s_h = sin h, 0 < h < pi)
__device__ __forceinline__ bool in_wedge(float x, float y, float ox, float oy, float fx, float fy, float c_h, float s_h)
{
    const float dx = x - ox, dy = y - oy;
    const float a = dx * fx + dy * fy;
    const float c = fabsf(dy * fx - dx * fy);
    return c_h * c <= s_h * a;
}

__device__ __forceinline__ unsigned pixel_rgb(const RenderEnv &s, const RenderView &v, float x, float y)
{
    unsigned rgb = CN_RENDER_RGB_BACKGROUND;
    if (v.draw_fov && in_wedge(x, y, s.rx, s.ry, s.fx, s.fy, v.fov_c, v.fov_s)) rgb = CN_RENDER_RGB_FOV;
    if (s.draw_goal && in_disc(x, y, s.gx, s.gy, (float)CN_RENDER_GOAL_RADIUS * (float)CN_RENDER_GOAL_RADIUS)) rgb = CN_RENDER_RGB_GOAL;
    for (unsigned m = s.live; m; m &= m - 1) {                  // ascending index: later humans over earlier ones
        const float4 h = s.hum[__ffs(m) - 1];
        if (in_disc(x, y, h.x, h.y, h.z)) rgb = h.w != 0.0f ? CN_RENDER_RGB_HUMAN_IN : CN_RENDER_RGB_HUMAN_OUT;
    }
    if (s.draw_robot && in_disc(x, y, s.rx, s.ry, s.rr2))
        rgb = in_wedge(x, y, s.rx, s.ry, s.fx, s.fy, v.head_c, v.head_s) ? CN_RENDER_RGB_HEADING : CN_RENDER_RGB_ROBOT;
    return rgb;
}

__global__ void __launch_bounds__(RENDER_THREADS) render_kernel(const EnvParams P, const int32_t *__restrict__ ids, int k,
                                                               const uint32_t *__restrict__ vis, int S, const RenderView v,
                                                               uint8_t *__restrict__ rgb)
{
    __shared__ RenderEnv s;
    __shared__ __align__(16) uint32_t words[RENDER_BAND * 3 / 4];
    const int t = threadIdx.x, lane = t & 31;
    const int H = P.cfg.human_num;
    const long long npix_frame = (long long)S * S;
    const int base = blockIdx.x * RENDER_BAND;                  // first pixel of the band
    const int npix = (int)min((long long)RENDER_BAND, npix_frame - base);
    // bounding box of the band's pixel centres
    const int i0 = base / S, i1 = (base + npix - 1) / S;
    const int j0 = i0 == i1 ? base % S : 0, j1 = i0 == i1 ? (base + npix - 1) % S : S - 1;
    const float x_lo = ((float)j0 + 0.5f) * v.scale - v.half, x_hi = ((float)j1 + 0.5f) * v.scale - v.half;
    const float y_hi = v.half - ((float)i0 + 0.5f) * v.scale, y_lo = v.half - ((float)i1 + 0.5f) * v.scale;

    for (int f = blockIdx.y; f < k; f += gridDim.y) {
        const int e = ids ? ids[f] : f;
        const bool valid = e >= 0 && e < P.n_envs;             // never read the state of an id outside [0, N)
        if (valid && t < 32) {
            const size_t hi = (size_t)e * H + lane;
            bool near = false;
            if (lane < H) {
                const float4 pv = P.a.hum_pv[hi], gr = P.a.hum_gr[hi];
                const bool in_fov = vis ? ((vis[e] >> lane) & 1u) != 0u : true;
                s.hum[lane] = make_float4(pv.x, pv.y, gr.z * gr.z, in_fov ? 1.0f : 0.0f);
                near = disc_near(pv.x, pv.y, gr.z, x_lo, x_hi, y_lo, y_hi, v.scale);
            }
            const unsigned live = __ballot_sync(0xffffffffu, near);
            if (lane == 0) {
                const float4 pv = P.a.rob_pv[e], gr = P.a.rob_gr[e];
                float fx = 1.0f, fy = 0.0f;
                if (P.cfg.kinematics == CN_HOLONOMIC) {
                    const float n = sqrtf(pv.z * pv.z + pv.w * pv.w);
                    if (n > 0.0f) { fx = pv.z / n; fy = pv.w / n; }
                } else {
                    const double th = (double)P.a.rob_x[e].x;
                    fx = (float)cos(th); fy = (float)sin(th);
                }
                s.rx = pv.x; s.ry = pv.y; s.rr2 = gr.z * gr.z; s.fx = fx; s.fy = fy; s.gx = gr.x; s.gy = gr.y;
                s.live = live;
                s.draw_goal = disc_near(gr.x, gr.y, (float)CN_RENDER_GOAL_RADIUS, x_lo, x_hi, y_lo, y_hi, v.scale);
                s.draw_robot = disc_near(pv.x, pv.y, gr.z, x_lo, x_hi, y_lo, y_hi, v.scale);
            }
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < RENDER_PIX_PER_THREAD / 4; ++q) {
            const int p = q * RENDER_THREADS * 4 + t * 4;       // band-relative index of the first of 4 pixels
            if (p < npix) {
                unsigned c[4];
                if (!valid) {
                    c[0] = c[1] = c[2] = c[3] = CN_RENDER_RGB_INVALID;
                } else {
                    const int i = (base + p) / S, j = (base + p) % S;   // S % 4 == 0: the 4 pixels share a row
                    const float y = v.half - ((float)i + 0.5f) * v.scale;
#pragma unroll
                    for (int u = 0; u < 4; ++u) c[u] = pixel_rgb(s, v, ((float)(j + u) + 0.5f) * v.scale - v.half, y);
                }
                // bytes R0 G0 B0 R1 | G1 B1 R2 G2 | B2 R3 G3 B3 as little-endian words
#define R_(x) (((x) >> 16) & 0xFFu)
#define G_(x) (((x) >> 8) & 0xFFu)
#define B_(x) ((x) & 0xFFu)
                uint32_t *w = words + (p / 4) * 3;
                w[0] = R_(c[0]) | G_(c[0]) << 8 | B_(c[0]) << 16 | R_(c[1]) << 24;
                w[1] = G_(c[1]) | B_(c[1]) << 8 | R_(c[2]) << 16 | G_(c[2]) << 24;
                w[2] = B_(c[2]) | R_(c[3]) << 8 | G_(c[3]) << 16 | B_(c[3]) << 24;
#undef R_
#undef G_
#undef B_
            }
        }
        __syncthreads();
        // the band is contiguous in the output and 16-byte aligned (S^2 % 256 == 0 and RENDER_BAND % 256 == 0)
        uint4 *dst = reinterpret_cast<uint4 *>(rgb + ((size_t)f * (size_t)npix_frame + (size_t)base) * 3);
        const uint4 *src = reinterpret_cast<const uint4 *>(words);
        const int n16 = npix * 3 / 16;
        for (int x = t; x < n16; x += RENDER_THREADS) dst[x] = src[x];
        __syncthreads();                                        // `s` and `words` are reused by the next frame
    }
}

extern "C" int cn_launch_render(const EnvParams *P, const int32_t *ids, int k, const uint32_t *vis, int size, uint8_t *rgb,
                                cudaStream_t stream)
{
    if (k == 0) return 0;
    RenderView v;
    const double L = P->cfg.square_width;
    v.scale = (float)(L / (double)size);
    v.half = (float)(L * 0.5);
    v.draw_fov = P->cfg.robot_fov < 2.0 * CN_PI;
    v.fov_c = (float)cos(P->cfg.robot_fov / 2.0);
    v.fov_s = (float)sin(P->cfg.robot_fov / 2.0);
    v.head_c = (float)cos((double)CN_RENDER_HEADING_HALF);
    v.head_s = (float)sin((double)CN_RENDER_HEADING_HALF);
    const long long npix = (long long)size * size;
    const dim3 grid((unsigned)((npix + RENDER_BAND - 1) / RENDER_BAND), (unsigned)(k < 65535 ? k : 65535));
    render_kernel<<<grid, RENDER_THREADS, 0, stream>>>(*P, ids, k, vis, size, v, rgb);
    return (int)cudaGetLastError();
}
