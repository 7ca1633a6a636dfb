// dsrnn_train.cu -- gate math of the masked GRU sequences of the PPO update (SURVEY.md 8(f) row N1; the reference's
// training forward is srnn_model.py:53-104, one nn.GRU step per mask segment).  The recurrent GEMMs stay cuBLAS calls
// made by the host (model.py `_MaskedGruSequence`); these two kernels are everything between them, fused so that a
// step of the sequence is two launches in each direction (GEMM + gates) and nothing is copied:
//   forward : gates -> h_t straight into the [T, R, hid] output, the gate values the backward needs into the [T, R, 4 hid]
//             workspace, and the MASKED state of the next step (h_t * m_{t+1}, the next GEMM's operand);
//   backward: g = dL/dh_t + m_{t+1} * dL/d(masked state of step t+1) formed in registers, then the gate gradients
//             straight into the [T, R, 3 hid] buffers the single weight-gradient GEMMs read at the end.
// HBM-bound, one thread per four hidden units (float4 everywhere): 13 floats of traffic per hidden unit forward, 14 backward
// (52 / 56 B; measured 38 / 42 us for 20480 rows x 256 = 7.1 / 7.0 TB/s, profiles/r1_ncu_gate_kernels.txt).
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace {

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

struct F4 { float v[4]; };
__device__ __forceinline__ F4 ld4(const float *p) { const float4 t = *reinterpret_cast<const float4 *>(p); return F4{{t.x, t.y, t.z, t.w}}; }
__device__ __forceinline__ void st4(float *p, const F4 &a) { *reinterpret_cast<float4 *>(p) = make_float4(a.v[0], a.v[1], a.v[2], a.v[3]); }
// a = hi + lo with hi = bf16(a), lo = bf16(a - hi): the operand pair of a split-bf16 3-pass GEMM (error ~2^-16 relative)
__device__ __forceinline__ void st4_split(__nv_bfloat16 *hi, __nv_bfloat16 *lo, const F4 &a)
{
    __nv_bfloat16 h[4], l[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        h[k] = __float2bfloat16_rn(a.v[k]);
        l[k] = __float2bfloat16_rn(a.v[k] - __bfloat162float(h[k]));
    }
    *reinterpret_cast<uint2 *>(hi) = *reinterpret_cast<const uint2 *>(h);
    *reinterpret_cast<uint2 *>(lo) = *reinterpret_cast<const uint2 *>(l);
}

__global__ void __launch_bounds__(256)
gru_gates_forward_kernel(const float *__restrict__ gi, const float *__restrict__ gh, const float *__restrict__ hm,
                         const float *__restrict__ b_ih, const float *__restrict__ b_hh, const float *__restrict__ m_next,
                         float *__restrict__ h_out, float *__restrict__ hm_next, float *__restrict__ ws,
                         __nv_bfloat16 *__restrict__ hm_next_hi, __nv_bfloat16 *__restrict__ hm_next_lo, int R, int hid)
{
    const int q = hid >> 2;                                     // float4 columns per row
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)R * q) return;
    const int row = (int)(idx / q), c = (int)(idx - (size_t)row * q) << 2;
    const float *gir = gi + (size_t)row * 3 * hid, *ghr = gh + (size_t)row * 3 * hid;
    const F4 ir = ld4(gir + c), iz = ld4(gir + hid + c), in = ld4(gir + 2 * hid + c);
    const F4 hr = ld4(ghr + c), hz = ld4(ghr + hid + c), hnn = ld4(ghr + 2 * hid + c);
    const F4 bir = ld4(b_ih + c), biz = ld4(b_ih + hid + c), bin = ld4(b_ih + 2 * hid + c);
    const F4 bhr = ld4(b_hh + c), bhz = ld4(b_hh + hid + c), bhn = ld4(b_hh + 2 * hid + c);
    const F4 hp = ld4(hm + (size_t)row * hid + c);
    F4 r, z, n, hn, h;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        r.v[k] = sigmoidf_((ir.v[k] + bir.v[k]) + (hr.v[k] + bhr.v[k]));
        z.v[k] = sigmoidf_((iz.v[k] + biz.v[k]) + (hz.v[k] + bhz.v[k]));
        hn.v[k] = hnn.v[k] + bhn.v[k];
        n.v[k] = tanhf((in.v[k] + bin.v[k]) + r.v[k] * hn.v[k]);
        h.v[k] = n.v[k] + z.v[k] * (hp.v[k] - n.v[k]);
    }
    st4(h_out + (size_t)row * hid + c, h);
    float *w = ws + (size_t)row * 4 * hid;
    st4(w + c, r); st4(w + hid + c, z); st4(w + 2 * hid + c, n); st4(w + 3 * hid + c, hn);
    if (hm_next) {
        const float m = m_next[row];
        F4 o;
#pragma unroll
        for (int k = 0; k < 4; ++k) o.v[k] = h.v[k] * m;
        st4(hm_next + (size_t)row * hid + c, o);
        if (hm_next_hi) st4_split(hm_next_hi + (size_t)row * hid + c, hm_next_lo + (size_t)row * hid + c, o);
    }
}

__global__ void __launch_bounds__(256)
gru_gates_backward_kernel(const float *__restrict__ grad_h, const float *__restrict__ d_next, const float *__restrict__ m_next,
                          const float *__restrict__ ws, const float *__restrict__ hm, float *__restrict__ dgi,
                          float *__restrict__ dgh, float *__restrict__ dhm, __nv_bfloat16 *__restrict__ dgi_hi,
                          __nv_bfloat16 *__restrict__ dgi_lo, __nv_bfloat16 *__restrict__ dgh_hi, __nv_bfloat16 *__restrict__ dgh_lo,
                          int R, int hid)
{
    const int q = hid >> 2;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)R * q) return;
    const int row = (int)(idx / q), c = (int)(idx - (size_t)row * q) << 2;
    F4 g = ld4(grad_h + (size_t)row * hid + c);
    if (d_next) {
        const float m = m_next[row];
        const F4 d = ld4(d_next + (size_t)row * hid + c);
#pragma unroll
        for (int k = 0; k < 4; ++k) g.v[k] = g.v[k] + d.v[k] * m;
    }
    const float *w = ws + (size_t)row * 4 * hid;
    const F4 r = ld4(w + c), z = ld4(w + hid + c), n = ld4(w + 2 * hid + c), hn = ld4(w + 3 * hid + c);
    const F4 hp = ld4(hm + (size_t)row * hid + c);
    F4 pr, pz, pn, pnr, dh;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        pn.v[k] = g.v[k] * (1.0f - z.v[k]) * (1.0f - n.v[k] * n.v[k]);
        pr.v[k] = pn.v[k] * hn.v[k] * r.v[k] * (1.0f - r.v[k]);
        pz.v[k] = g.v[k] * (hp.v[k] - n.v[k]) * z.v[k] * (1.0f - z.v[k]);
        pnr.v[k] = pn.v[k] * r.v[k];
        dh.v[k] = g.v[k] * z.v[k];
    }
    float *a = dgi + (size_t)row * 3 * hid, *b = dgh + (size_t)row * 3 * hid;
    st4(a + c, pr); st4(a + hid + c, pz); st4(a + 2 * hid + c, pn);
    st4(b + c, pr); st4(b + hid + c, pz); st4(b + 2 * hid + c, pnr);
    st4(dhm + (size_t)row * hid + c, dh);
    if (dgi_hi) {                                               // the same gradients as bf16 pairs for the 3-pass GEMMs
        const size_t o = (size_t)row * 3 * hid + c;
        st4_split(dgi_hi + o, dgi_lo + o, pr); st4_split(dgi_hi + o + hid, dgi_lo + o + hid, pz);
        st4_split(dgi_hi + o + 2 * hid, dgi_lo + o + 2 * hid, pn);
        st4_split(dgh_hi + o, dgh_lo + o, pr); st4_split(dgh_hi + o + hid, dgh_lo + o + hid, pz);
        st4_split(dgh_hi + o + 2 * hid, dgh_lo + o + 2 * hid, pnr);
    }
}

// Gate gradients of one step, written as the split-bf16 operand G = [pn | pr | pz | pn*r] ([R, 4 hid]) of the tensor-core
// products that follow (cn_gemm_bf16x3): columns [0, 3 hid) are d(gi) in gate order n|r|z (-> dx, dW_ih), columns
// [hid, 4 hid) are d(gh) in gate order r|z|n (-> the recurrent product G[:, hid:] W_hh and dW_hh).  d = g * z in place.
// 9 floats read + 1 float and 8 bf16 written per hidden unit (56 B).
__global__ void __launch_bounds__(256)
gru_gates_backward_pairs_kernel(const float *__restrict__ grad_h, float *__restrict__ d, int d_live, const float *__restrict__ m_next,
                                const float *__restrict__ ws, const float *__restrict__ h_prev, const float *__restrict__ m_cur,
                                __nv_bfloat16 *__restrict__ g_hi, __nv_bfloat16 *__restrict__ g_lo, int R, int hid)
{
    const int q = hid >> 2;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)R * q) return;
    const int row = (int)(idx / q), c = (int)(idx - (size_t)row * q) << 2;
    F4 g = ld4(grad_h + (size_t)row * hid + c);
    float *drow = d + (size_t)row * hid + c;
    if (d_live) {
        const float m = m_next[row];
        const F4 dn = ld4(drow);
#pragma unroll
        for (int k = 0; k < 4; ++k) g.v[k] = g.v[k] + dn.v[k] * m;
    }
    const float *w = ws + (size_t)row * 4 * hid;
    const F4 r = ld4(w + c), z = ld4(w + hid + c), n = ld4(w + 2 * hid + c), hn = ld4(w + 3 * hid + c);
    F4 hp = F4{{0.f, 0.f, 0.f, 0.f}};
    if (h_prev) {
        const float mc = m_cur[row];
        hp = ld4(h_prev + (size_t)row * hid + c);
#pragma unroll
        for (int k = 0; k < 4; ++k) hp.v[k] *= mc;
    }
    F4 pr, pz, pn, pnr, dh;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        pn.v[k] = g.v[k] * (1.0f - z.v[k]) * (1.0f - n.v[k] * n.v[k]);
        pr.v[k] = pn.v[k] * hn.v[k] * r.v[k] * (1.0f - r.v[k]);
        pz.v[k] = g.v[k] * (hp.v[k] - n.v[k]) * z.v[k] * (1.0f - z.v[k]);
        pnr.v[k] = pn.v[k] * r.v[k];
        dh.v[k] = g.v[k] * z.v[k];
    }
    st4(drow, dh);
    const size_t o = (size_t)row * 4 * hid + c;
    st4_split(g_hi + o, g_lo + o, pn); st4_split(g_hi + o + hid, g_lo + o + hid, pr);
    st4_split(g_hi + o + 2 * hid, g_lo + o + 2 * hid, pz); st4_split(g_hi + o + 3 * hid, g_lo + o + 3 * hid, pnr);
}

__global__ void __launch_bounds__(256)
split_bf16_kernel(const float *__restrict__ a, __nv_bfloat16 *__restrict__ hi, __nv_bfloat16 *__restrict__ lo, size_t n4)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    st4_split(hi + 4 * i, lo + 4 * i, ld4(a + 4 * i));
}

// ------------------------------------------------------------------------------------------------ attention (training)
// EdgeAttention over a [B = T*n] batch (srnn_model.py:256-339) with the key projection folded into the query:
//   s_i = (o_i . qt + cst) * scale,  alpha = softmax_i(s),  c = sum_i alpha_i o_i          (qt = W_s^T q, cst = q . b_s)
// One warp per sample; lane l owns hidden units [4l, 4l+4) and [128 + 4l, 128 + 4l + 4) (two coalesced float4 per row).
// HBM-bound: the forward reads o once (H KB per sample) and writes c and alpha; the backward reads o (twice, the second
// time out of L1/L2), dc, qt, alpha and writes d_o (H KB) and d_qt.
__device__ __forceinline__ float warp_sum(float v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float dot8(const float4 &a0, const float4 &a1, const float4 &b0, const float4 &b1)
{
    return a0.x * b0.x + a0.y * b0.y + a0.z * b0.z + a0.w * b0.w + a1.x * b1.x + a1.y * b1.y + a1.z * b1.z + a1.w * b1.w;
}

__global__ void __launch_bounds__(128)
attention_train_forward_kernel(const float *__restrict__ o, const float *__restrict__ qt, const float *__restrict__ cst,
                               float *__restrict__ c, float *__restrict__ alpha, float scale, int B, int H)
{
    const int b = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= B) return;
    const float4 *q4 = reinterpret_cast<const float4 *>(qt + (size_t)b * 256);
    const float4 q0 = q4[lane], q1 = q4[32 + lane];
    const float k = cst ? cst[b] : 0.f;
    const float4 *orow = reinterpret_cast<const float4 *>(o + (size_t)b * H * 256);
    float my_s = -INFINITY;                  // lane i keeps s_i
    float run_max = -INFINITY, run_sum = 0.f;
    float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0;
    for (int i = 0; i < H; ++i) {
        const float4 v0 = orow[i * 64 + lane], v1 = orow[i * 64 + 32 + lane];
        const float s = (warp_sum(dot8(v0, v1, q0, q1)) + k) * scale;
        if (lane == i) my_s = s;
        const float m = fmaxf(run_max, s);
        const float f = __expf(run_max - m), w = __expf(s - m);      // online softmax: rescale what was accumulated so far
        run_sum = run_sum * f + w;
        a0.x = a0.x * f + w * v0.x; a0.y = a0.y * f + w * v0.y; a0.z = a0.z * f + w * v0.z; a0.w = a0.w * f + w * v0.w;
        a1.x = a1.x * f + w * v1.x; a1.y = a1.y * f + w * v1.y; a1.z = a1.z * f + w * v1.z; a1.w = a1.w * f + w * v1.w;
        run_max = m;
    }
    const float inv = 1.0f / run_sum;
    float4 *c4 = reinterpret_cast<float4 *>(c + (size_t)b * 256);
    c4[lane] = make_float4(a0.x * inv, a0.y * inv, a0.z * inv, a0.w * inv);
    c4[32 + lane] = make_float4(a1.x * inv, a1.y * inv, a1.z * inv, a1.w * inv);
    if (lane < H) alpha[(size_t)b * H + lane] = __expf(my_s - run_max) * inv;
}

__global__ void __launch_bounds__(128)
attention_train_backward_kernel(const float *__restrict__ o, const float *__restrict__ qt, const float *__restrict__ alpha,
                                const float *__restrict__ dc, float *__restrict__ d_o, float *__restrict__ d_qt,
                                float *__restrict__ d_cst, float scale, int B, int H)
{
    const int b = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= B) return;
    const float4 *q4 = reinterpret_cast<const float4 *>(qt + (size_t)b * 256), *g4 = reinterpret_cast<const float4 *>(dc + (size_t)b * 256);
    const float4 q0 = q4[lane], q1 = q4[32 + lane], g0 = g4[lane], g1 = g4[32 + lane];
    const float4 *orow = reinterpret_cast<const float4 *>(o + (size_t)b * H * 256);
    const float al = lane < H ? alpha[(size_t)b * H + lane] : 0.f;
    float da = 0.f;                          // lane i: o_i . dc
    for (int i = 0; i < H; ++i) {
        const float d = warp_sum(dot8(orow[i * 64 + lane], orow[i * 64 + 32 + lane], g0, g1));
        if (lane == i) da = d;
    }
    const float dot = warp_sum(al * da);
    const float ds = al * (da - dot) * scale;            // dL/d(o_i . qt + cst), lane i
    float4 t0 = make_float4(0.f, 0.f, 0.f, 0.f), t1 = t0;
    float4 *drow = reinterpret_cast<float4 *>(d_o + (size_t)b * H * 256);
    for (int i = 0; i < H; ++i) {
        const float a_i = __shfl_sync(0xffffffffu, al, i), s_i = __shfl_sync(0xffffffffu, ds, i);
        const float4 v0 = orow[i * 64 + lane], v1 = orow[i * 64 + 32 + lane];
        drow[i * 64 + lane] = make_float4(a_i * g0.x + s_i * q0.x, a_i * g0.y + s_i * q0.y, a_i * g0.z + s_i * q0.z, a_i * g0.w + s_i * q0.w);
        drow[i * 64 + 32 + lane] = make_float4(a_i * g1.x + s_i * q1.x, a_i * g1.y + s_i * q1.y, a_i * g1.z + s_i * q1.z, a_i * g1.w + s_i * q1.w);
        t0.x += s_i * v0.x; t0.y += s_i * v0.y; t0.z += s_i * v0.z; t0.w += s_i * v0.w;
        t1.x += s_i * v1.x; t1.y += s_i * v1.y; t1.z += s_i * v1.z; t1.w += s_i * v1.w;
    }
    float4 *dq4 = reinterpret_cast<float4 *>(d_qt + (size_t)b * 256);
    dq4[lane] = t0; dq4[32 + lane] = t1;
    if (d_cst) { const float tot = warp_sum(ds); if (lane == 0) d_cst[b] = tot; }
}

// ------------------------------------------------------------------------------------------------ edge-encoder gradient
// e = ReLU(W_enc x + b) with x [rows, 2] (HumanHumanEdgeRNN.encoder_linear, srnn_model.py:201-215).  Given de = dL/de
// [rows, 64] (fp32) and the sign of e (its bf16 hi image, row stride ld_e):  dW_enc[k, j] = sum_rows [e_k > 0] de_k x_j,
// db_enc[k] = sum_rows [e_k > 0] de_k.  One pass over de: HBM-bound.  Block = 4 rows x 64 columns per iteration; block sums are
// combined in shared memory and added to the outputs with 64 x 3 atomics per block.  The ordered instantiation writes the
// 64 x 3 block sums to part[block] instead, and encoder_grad_reduce_kernel adds them to dw / db in block order.
template <bool kOrdered>
__global__ void __launch_bounds__(256)
encoder_grad_kernel(const float *__restrict__ de, const __nv_bfloat16 *__restrict__ e_hi, int ld_e, const float *__restrict__ x,
                    float *__restrict__ dw, float *__restrict__ db, long long rows, float *__restrict__ part_out)
{
    __shared__ float part[4][64][3];
    const int col = threadIdx.x & 63, rsub = threadIdx.x >> 6;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f;
    for (long long row = (long long)blockIdx.x * 4 + rsub; row < rows; row += (long long)gridDim.x * 4) {
        const float v = de[row * 64 + col];
        const bool on = __bfloat162float(e_hi[row * ld_e + col]) > 0.0f;
        const float2 xv = *reinterpret_cast<const float2 *>(x + row * 2);
        if (on) { s0 += v * xv.x; s1 += v * xv.y; s2 += v; }
    }
    part[rsub][col][0] = s0; part[rsub][col][1] = s1; part[rsub][col][2] = s2;
    __syncthreads();
    if (threadIdx.x < 192) {
        const int c = threadIdx.x / 3, k = threadIdx.x - 3 * c;
        const float t = part[0][c][k] + part[1][c][k] + part[2][c][k] + part[3][c][k];
        if (kOrdered) part_out[(size_t)blockIdx.x * 192 + threadIdx.x] = t;
        else if (k < 2) atomicAdd(dw + c * 2 + k, t); else atomicAdd(db + c, t);
    }
}

// dw[c, k] (k < 2) / db[c] (k = 2) += part[0][c][k] + part[1][c][k] + ... in block order; one thread per output
__global__ void __launch_bounds__(192)
encoder_grad_reduce_kernel(const float *__restrict__ part, int blocks, float *__restrict__ dw, float *__restrict__ db)
{
    const int t = threadIdx.x, c = t / 3, k = t - 3 * c;
    float *out = k < 2 ? dw + c * 2 + k : db + c;
    float acc = *out;
#pragma unroll 16
    for (int b = 0; b < blocks; ++b) acc += part[(size_t)b * 192 + t];
    *out = acc;
}

// grid of encoder_grad_kernel: a function of `rows` only
inline long long encoder_grad_blocks(long long rows)
{
    const long long blocks = (rows + 3) / 4;
    return blocks < 148 * 8 ? blocks : 148 * 8;
}

inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline bool aligned8(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }

}  // namespace

// host launchers (called from c_abi.cu); return a cudaError_t as int, -1 for bad arguments
extern "C" int cn_launch_gru_gates_forward(const float *gi, const float *gh, const float *hm, const float *b_ih, const float *b_hh,
                                           const float *m_next, float *h_out, float *hm_next, float *ws, void *hm_next_hi,
                                           void *hm_next_lo, int R, int hid, cudaStream_t stream)
{
    if (R < 1 || hid < 4 || (hid & 3) || !aligned16(gi) || !aligned16(gh) || !aligned16(hm) || !aligned16(b_ih) || !aligned16(b_hh) ||
        !aligned16(h_out) || !aligned16(ws) || (hm_next && !aligned16(hm_next)) || (hm_next && !m_next) ||
        ((hm_next_hi != nullptr) != (hm_next_lo != nullptr)) || (hm_next_hi && (!hm_next || !aligned8(hm_next_hi) || !aligned8(hm_next_lo))))
        return -1;
    const size_t n = (size_t)R * (hid >> 2);
    gru_gates_forward_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(gi, gh, hm, b_ih, b_hh, m_next, h_out, hm_next, ws,
        static_cast<__nv_bfloat16 *>(hm_next_hi), static_cast<__nv_bfloat16 *>(hm_next_lo), R, hid);
    return (int)cudaGetLastError();
}

extern "C" int cn_launch_gru_gates_backward(const float *grad_h, const float *d_next, const float *m_next, const float *ws,
                                            const float *hm, float *dgi, float *dgh, float *dhm, void *const *pairs, int R, int hid,
                                            cudaStream_t stream)
{
    if (R < 1 || hid < 4 || (hid & 3) || !aligned16(grad_h) || (d_next && (!aligned16(d_next) || !m_next)) || !aligned16(ws) ||
        !aligned16(hm) || !aligned16(dgi) || !aligned16(dgh) || !aligned16(dhm)) return -1;
    __nv_bfloat16 *p[4] = {nullptr, nullptr, nullptr, nullptr};
    if (pairs) {
        for (int k = 0; k < 4; ++k) {
            if (!pairs[k] || !aligned8(pairs[k])) return -1;
            p[k] = static_cast<__nv_bfloat16 *>(pairs[k]);
        }
    }
    const size_t n = (size_t)R * (hid >> 2);
    gru_gates_backward_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(grad_h, d_next, m_next, ws, hm, dgi, dgh, dhm,
                                                                               p[0], p[1], p[2], p[3], R, hid);
    return (int)cudaGetLastError();
}

extern "C" int cn_launch_split_bf16(const float *a, void *hi, void *lo, size_t n, cudaStream_t stream)
{
    if (n == 0 || (n & 3) || !aligned16(a) || !aligned8(hi) || !aligned8(lo)) return -1;
    const size_t n4 = n >> 2;
    split_bf16_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, stream>>>(a, static_cast<__nv_bfloat16 *>(hi), static_cast<__nv_bfloat16 *>(lo), n4);
    return (int)cudaGetLastError();
}

extern "C" int cn_launch_gru_gates_backward_pairs(const float *grad_h, float *d, int d_live, const float *m_next, const float *ws,
                                                  const float *h_prev, const float *m_cur, void *g_hi, void *g_lo, int R, int hid,
                                                  cudaStream_t stream)
{
    if (R < 1 || hid < 4 || (hid & 3) || !aligned16(grad_h) || !aligned16(d) || !aligned16(ws) || (h_prev && (!aligned16(h_prev) || !m_cur)) ||
        (d_live && !m_next) || !aligned8(g_hi) || !aligned8(g_lo)) return -1;
    const size_t n = (size_t)R * (hid >> 2);
    gru_gates_backward_pairs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(grad_h, d, d_live, m_next, ws, h_prev, m_cur,
        static_cast<__nv_bfloat16 *>(g_hi), static_cast<__nv_bfloat16 *>(g_lo), R, hid);
    return (int)cudaGetLastError();
}

extern "C" int cn_launch_attention_train_forward(const float *o, const float *qt, const float *cst, float *c, float *alpha, float scale,
                                                 int B, int H, cudaStream_t stream)
{
    if (B < 1 || H < 1 || H > 32 || !aligned16(o) || !aligned16(qt) || !aligned16(c)) return -1;
    attention_train_forward_kernel<<<(B + 3) / 4, 128, 0, stream>>>(o, qt, cst, c, alpha, scale, B, H);
    return (int)cudaGetLastError();
}

extern "C" int cn_launch_attention_train_backward(const float *o, const float *qt, const float *alpha, const float *dc, float *d_o,
                                                  float *d_qt, float *d_cst, float scale, int B, int H, cudaStream_t stream)
{
    if (B < 1 || H < 1 || H > 32 || !aligned16(o) || !aligned16(qt) || !aligned16(dc) || !aligned16(d_o) || !aligned16(d_qt)) return -1;
    attention_train_backward_kernel<<<(B + 3) / 4, 128, 0, stream>>>(o, qt, alpha, dc, d_o, d_qt, d_cst, scale, B, H);
    return (int)cudaGetLastError();
}

extern "C" int cn_launch_encoder_grad(const float *de, const void *e_hi, int ld_e, const float *x, float *dw, float *db, long long rows,
                                      cudaStream_t stream)
{
    if (rows < 1 || ld_e < 64 || !aligned16(de) || !aligned8(x)) return -1;
    const long long blocks = encoder_grad_blocks(rows);
    encoder_grad_kernel<false><<<(unsigned)blocks, 256, 0, stream>>>(de, static_cast<const __nv_bfloat16 *>(e_hi), ld_e, x, dw, db, rows,
                                                                     nullptr);
    return (int)cudaGetLastError();
}

extern "C" size_t cn_launch_encoder_grad_ordered_bytes(long long rows)
{
    return rows < 1 ? 0 : (size_t)encoder_grad_blocks(rows) * 192 * sizeof(float);
}

// -1 bad arguments, -2 workspace NULL / misaligned / too small
extern "C" int cn_launch_encoder_grad_ordered(const float *de, const void *e_hi, int ld_e, const float *x, float *dw, float *db, long long rows,
                                              void *workspace, size_t workspace_bytes, cudaStream_t stream)
{
    if (rows < 1 || ld_e < 64 || !aligned16(de) || !aligned8(x)) return -1;
    if (!workspace || !aligned16(workspace) || workspace_bytes < cn_launch_encoder_grad_ordered_bytes(rows)) return -2;
    const long long blocks = encoder_grad_blocks(rows);
    float *part = static_cast<float *>(workspace);
    encoder_grad_kernel<true><<<(unsigned)blocks, 256, 0, stream>>>(de, static_cast<const __nv_bfloat16 *>(e_hi), ld_e, x, dw, db, rows, part);
    const cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return (int)err;
    encoder_grad_reduce_kernel<<<1, 192, 0, stream>>>(part, (int)blocks, dw, db);
    return (int)cudaGetLastError();
}
