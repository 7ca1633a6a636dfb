// gemm_bf16x3.cu -- the GEMM of the PPO update (SURVEY.md 8(f) row N1) on the 5th-gen tensor cores (tcgen05 / TMEM / TMA),
// sm_100a only.  Replaces every cuBLAS product of the reference's update (ppo.py:36-118 -> evaluate_actions,
// srnn_model.py:53-104 and its autograd transpose): forward linears, the recurrent products of the masked GRU sequences
// and their backward, and the weight-gradient reductions over the T*R row dimension.
//
//     C[M,N] (fp32)   =  | +=  | split-K: += partial products     (A_hi + A_lo)(B_hi + B_lo)   (+ bias[n], ReLU / tanh)
//
// Split-bf16 3-pass arithmetic (A_hi B_hi + A_lo B_hi + A_hi B_lo, fp32 accumulation in TMEM; operand error ~2^-16: the
// precision of the rollout kernels, CN_PREC_BF16X3).  Operands are bf16 (hi, lo) pairs in global memory, written by the
// kernels that produce them (cn_split_bf16, the gate kernels, the edge sequence kernel).  Each operand is either
//   K-major  : a row-major [MN, K] array (activations x weights^T: A = X [M,K], B = W [N,K]), or
//   MN-major : a row-major [K, MN] array -- what the backward products read without any transposition:
//              dX = dY W  (B = W [K=N_out, N=K_in] row-major), dW = dY^T X (A = dY [K=rows, M], B = X [K=rows, N]).
// Both forms are fetched by TMA (cp.async.bulk.tensor.2d, SWIZZLE_128B) straight into the canonical UMMA shared-memory
// layouts; the MMA instruction descriptor carries the a_major / b_major bits.
//
// One persistent CTA per SM walks work items (problem, k-slice, 128-row tile, n-tile).  320 threads:
//   warp 0      TMA producer: one elected lane streams 64-deep k-blocks of A (hi, lo) and B (hi, lo) through a ring of stages;
//   warp 1      owns TMEM (512 columns = two accumulator buffers of up to 256 columns) and issues tcgen05.mma
//               (M = 128, N = n-tile, K = 16; 12 per k-block for the three passes);
//   warps 2-9   epilogue: tcgen05.ld -> (bias, activation) -> 256-bit stores of each lane's row segment, read-modify-write
//               (accumulate) or red.global.add (split-K partial sums), overlapped with the MMAs of the next item through
//               the second TMEM buffer.
// Ordered split-K (cn_gemm_bf16x3_ordered, the `kOrdered` instantiation): a k-slice stores its partial tile into its own
// slice of a caller-provided workspace instead (every element written once, by one CTA: no atomics, no inter-CTA waits),
// and splitk_reduce_kernel then forms C = C_in + P_0 + ... + P_{S-1} in slice order.  The slice count is a function of the
// problem's own (m, n, k, split_k) only (ordered_slices), so a product gives the same bits alone or grouped, on any device.
// CTAs are launched as clusters of c = 1, 2 or 4 that walk c consecutive 128-row tiles of the same (k-slice, n-tile) in lock
// step: the B tile (weights: the same for every row tile, and the larger operand of the recurrent products) is fetched from
// L2 once per cluster -- every CTA loads 1/c of it and TMA-multicasts it into all c shared memories
// (cp.async.bulk.tensor ... .multicast::cluster); tcgen05.commit multicasts the "stage free" arrivals back.
// Up to kMaxProblems independent problems share one launch (grouped GEMM: the spatial / temporal edge GRUs have different
// weights; the weight gradients of both are one launch).
#include <cuda.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "tc_common.cuh"
#include "../../include/crowdnav_b200.h"

using namespace tc;

void gemm_bf16x3_enable_timing(int enable);
float gemm_bf16x3_time_ms(int *launches, double *flops);

namespace {

constexpr int kMaxProblems = CN_GEMM_MAX_PROBLEMS;
constexpr int kThreads = 320;              // TMA producer, MMA issuer, 8 epilogue warps
constexpr int kTileM = 128;
constexpr int kABytes = kTileM * 128;              // one 128 x 64 bf16 image (hi or lo) of A: 16 KB in either major
constexpr int kMaxStages = 6;
constexpr int kScratchBytes = 0;
constexpr int kSmemLimit = 232448 - 1024;          // dynamic shared memory of one sm_100 CTA minus the alignment slack

struct alignas(64) GemmProblem {
    CUtensorMap a_hi, a_lo, b_hi, b_lo;
    float *c;
    const float *bias;
    long long ldc;
    int m, n, k;
    int bn;                    // n-tile = MMA N (multiple of 16, <= 256)
    int m_tiles, n_tiles;
    int split_k, kb_per_split; // k-blocks (64 deep) per k-slice
    int a_mn, b_mn;            // operand majors (1 = MN-major)
    int a_lo_on, b_lo_on;      // passes A_lo*B_hi / A_hi*B_lo enabled
    int act, mode;             // mode 0 store, 1 read-modify-write add, 2 atomic add, 3 store into workspace slice ks (ordered)
    int m_groups;              // groups of c consecutive m-tiles (one per cluster and item)
    int b_slice_bytes;         // bytes of one CTA's slice of the B tile (K-major: bn/c rows; MN-major: 64/c k-rows of every atom)
    int item0, items;          // this problem's range of global work items (one item = one cluster-wide group of m-tiles)
    unsigned stage_tx;         // bytes one stage of this problem brings in
};

struct GemmArgs {
    GemmProblem p[kMaxProblems];
    int n_problems, total_items;
    int stages, stage_bytes, b_off_lo;   // ring geometry: A_hi @0, A_lo @16K, B_hi @32K, B_lo @32K + b_off_lo
    int cluster;                         // CTAs per cluster (1, 2, 4)
};

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void *tmap, int c0, int c1, uint32_t mbar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(tmap), "r"(mbar), "r"(c0), "r"(c1) : "memory");
}

__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const void *tmap, int c0, int c1, uint32_t mbar, uint16_t mask)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
                 ::"r"(dst), "l"(tmap), "r"(mbar), "r"(c0), "r"(c1), "h"(mask) : "memory");
}
// completion of all prior MMAs of this thread arrives on the barrier at this offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_mc(uint32_t bar, uint16_t mask)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(mask) : "memory");
}
__device__ __forceinline__ void umma_commit_mc_if(uint32_t lead, uint32_t bar, uint16_t mask)      // warp-uniform issue form
{
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t"
                 "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t}"
                 ::"r"(bar), "h"(mask), "r"(lead) : "memory");
}
__device__ __forceinline__ uint32_t cluster_nctarank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return r;
}

__device__ __forceinline__ void ld_global_v8(const float *p, float *v)
{
    asm volatile("ld.global.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7]) : "l"(p) : "memory");
}

struct Item { int p, ks, mt, nt; };

// item -> (problem, k-slice, m-tile of THIS CTA, n-tile); the c CTAs of a cluster get c consecutive m-tiles of the same
// (k-slice, n-tile), possibly past the last one (then the tile is all padding: zero operands, no stores)
__device__ __forceinline__ Item decode_item(const GemmArgs &a, int item, int rank)
{
    Item it;
    int p = 0;
    while (p + 1 < a.n_problems && item >= a.p[p + 1].item0) ++p;
    const GemmProblem &g = a.p[p];
    int r = item - g.item0;
    it.p = p;
    it.nt = r % g.n_tiles; r /= g.n_tiles;      // n-tiles of the same rows run on neighbouring clusters (A comes out of L2),
    it.mt = (r % g.m_groups) * a.cluster + rank; r /= g.m_groups;   // then the m-tiles of one k-slice (split-K: B comes out of L2)
    it.ks = r;
    return it;
}

template <bool kOrdered>
__global__ void __launch_bounds__(kThreads, 1) gemm_bf16x3_kernel(const __grid_constant__ GemmArgs a)
{
    extern __shared__ unsigned char smem_dyn[];
    unsigned char *smem = reinterpret_cast<unsigned char *>(((uintptr_t)smem_dyn + 1023) & ~(uintptr_t)1023);
    const uint32_t s_base = smem_u32(smem);
    const int ring_bytes = a.stages * a.stage_bytes;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + ring_bytes + kScratchBytes);
    uint32_t *s_tmem = reinterpret_cast<uint32_t *>(bars + 2 * kMaxStages + 4);
    const uint32_t bar0 = smem_u32(bars);
    // barrier map: [0, S) full | [S, 2S) empty | 2S, 2S+1 tmem_full | 2S+2, 2S+3 tmem_empty      (S = kMaxStages)
    auto bar_full = [&](int s) { return bar0 + 8u * (uint32_t)s; };
    auto bar_empty = [&](int s) { return bar0 + 8u * (uint32_t)(kMaxStages + s); };
    auto bar_tfull = [&](int b) { return bar0 + 8u * (uint32_t)(2 * kMaxStages + b); };
    auto bar_tempty = [&](int b) { return bar0 + 8u * (uint32_t)(2 * kMaxStages + 2 + b); };
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int csize = a.cluster;
    const int rank = csize > 1 ? (int)cluster_ctarank() : 0;
    const int cluster_id = blockIdx.x / csize, num_clusters = gridDim.x / csize;
    const uint16_t cmask = (uint16_t)((1u << csize) - 1u);

    if (threadIdx.x == 0) {
        // a stage is free when the MMAs of ALL CTAs of the cluster have read it (peers multicast into it)
        for (int s = 0; s < kMaxStages; ++s) { mbar_init(bar_full(s), 1); mbar_init(bar_empty(s), csize); }
        mbar_init(bar_tfull(0), 1); mbar_init(bar_tfull(1), 1);
        mbar_init(bar_tempty(0), 8); mbar_init(bar_tempty(1), 8);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    if (csize > 1) cluster_sync_all();          // barrier initialisation is visible to the peers before anything arrives on them
    tc_fence_after();
    const uint32_t tmem_base = *s_tmem;

    if (warp == 0) {
        // =============================================================== TMA producer
        if (lane == 0) {
            uint32_t stage = 0, parity = 1;           // a fresh barrier passes a wait on parity 1
            for (int item = cluster_id; item < a.total_items; item += num_clusters) {
                const Item it = decode_item(a, item, rank);
                const GemmProblem &g = a.p[it.p];
                const int kb0 = it.ks * g.kb_per_split;
                int kb1 = kb0 + g.kb_per_split;
                const int kb_total = (g.k + 63) >> 6;
                if (kb1 > kb_total) kb1 = kb_total;
                const int m0 = it.mt * kTileM, n0 = it.nt * g.bn;
                const int brow = g.b_mn ? rank * (64 / csize) : rank * (g.bn / csize);    // this CTA's slice of the B tile
                for (int kb = kb0; kb < kb1; ++kb) {
                    mbar_wait(bar_empty(stage), parity);
                    const uint32_t full = bar_full(stage);
                    mbar_expect_tx(full, g.stage_tx);
                    const uint32_t sa = s_base + stage * a.stage_bytes, sb = sa + 2 * kABytes;
                    const int k0 = kb << 6;
                    if (g.a_mn) {                      // [K, M] array: two 64-wide M atoms of 64 k-rows each
                        tma_load_2d(sa, &g.a_hi, m0, k0, full);
                        tma_load_2d(sa + 8192, &g.a_hi, m0 + 64, k0, full);
                        if (g.a_lo_on) { tma_load_2d(sa + kABytes, &g.a_lo, m0, k0, full); tma_load_2d(sa + kABytes + 8192, &g.a_lo, m0 + 64, k0, full); }
                    } else {                           // [M, K] array: one box of 128 rows x 64 k
                        tma_load_2d(sa, &g.a_hi, k0, m0, full);
                        if (g.a_lo_on) tma_load_2d(sa + kABytes, &g.a_lo, k0, m0, full);
                    }
                    if (csize == 1) {
                        if (g.b_mn) {
                            for (int j = 0; j * 64 < g.bn; ++j) {
                                tma_load_2d(sb + j * 8192, &g.b_hi, n0 + j * 64, k0, full);
                                if (g.b_lo_on) tma_load_2d(sb + a.b_off_lo + j * 8192, &g.b_lo, n0 + j * 64, k0, full);
                            }
                        } else {
                            tma_load_2d(sb, &g.b_hi, k0, n0, full);
                            if (g.b_lo_on) tma_load_2d(sb + a.b_off_lo, &g.b_lo, k0, n0, full);
                        }
                    } else if (g.b_mn) {           // 64/c k-rows of every 64-wide atom, multicast to the whole cluster
                        const uint32_t soff = (uint32_t)brow * 128u;
                        for (int j = 0; j * 64 < g.bn; ++j) {
                            tma_load_2d_mc(sb + j * 8192 + soff, &g.b_hi, n0 + j * 64, k0 + brow, full, cmask);
                            if (g.b_lo_on) tma_load_2d_mc(sb + a.b_off_lo + j * 8192 + soff, &g.b_lo, n0 + j * 64, k0 + brow, full, cmask);
                        }
                    } else {                       // bn/c rows of the [bn, 64] tile
                        const uint32_t soff = (uint32_t)brow * 128u;
                        tma_load_2d_mc(sb + soff, &g.b_hi, k0, n0 + brow, full, cmask);
                        if (g.b_lo_on) tma_load_2d_mc(sb + a.b_off_lo + soff, &g.b_lo, k0, n0 + brow, full, cmask);
                    }
                    if (++stage == (uint32_t)a.stages) { stage = 0; parity ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // =============================================================== MMA issuer: warp-uniform control flow, the elected lane issues
        // (elect_one_sync in tc_common.cuh: descriptors stay in uniform registers, no R2UR waterfall per UTCHMMA)
        {
            const uint32_t lead = elect_one_sync();
            constexpr uint32_t kDescHi = (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29);     // SBO = 1024 B, version 1, SWIZZLE_128B
            auto make_desc = [](uint32_t lo) { uint64_t d; asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(kDescHi)); return d; };
            uint32_t stage = 0, parity = 0, iter = 0;
            for (int item = cluster_id; item < a.total_items; item += num_clusters, ++iter) {
                const Item it = decode_item(a, item, rank);
                const GemmProblem &g = a.p[it.p];
                const int kb0 = it.ks * g.kb_per_split;
                int kb1 = kb0 + g.kb_per_split;
                const int kb_total = (g.k + 63) >> 6;
                if (kb1 > kb_total) kb1 = kb_total;
                const uint32_t buf = iter & 1u;
                mbar_wait(bar_tempty(buf), ((iter >> 1) & 1u) ^ 1u);
                tc_fence_after();
                const uint32_t d = tmem_base + buf * 256u;
                const uint32_t idesc = idesc_bf16(g.bn) | ((uint32_t)g.a_mn << 15) | ((uint32_t)g.b_mn << 16);
                // descriptor low words: (address >> 4) | LBO << 16.  K-major: LBO unused (1), a K = 16 step is 32 bytes along the
                // 128-byte row.  MN-major: LBO = 8192 B (the next 64-wide MN atom), a K = 16 step is 16 rows of 128 bytes.
                const uint32_t a_lbo = g.a_mn ? (8192u >> 4) << 16 : 1u << 16, b_lbo = g.b_mn ? (8192u >> 4) << 16 : 1u << 16;
                const uint32_t a_step = g.a_mn ? 2048u >> 4 : 32u >> 4, b_step = g.b_mn ? 2048u >> 4 : 32u >> 4;
                uint32_t first = 1;
                for (int kb = kb0; kb < kb1; ++kb) {
                    mbar_wait(bar_full(stage), parity);
                    tc_fence_after();
                    // (in a cluster the shared-window address carries the CTA rank in its upper bits: only the low 18 bits
                    // are the matrix start address, anything above would spill into the descriptor's LBO field)
                    const uint32_t sa = (s_base & 0x3FFFFu) + stage * a.stage_bytes, sb = sa + 2 * kABytes;
                    const uint32_t a_hi = (sa >> 4) | a_lbo, a_lo = ((sa + kABytes) >> 4) | a_lbo;
                    const uint32_t b_hi = (sb >> 4) | b_lbo, b_lo = ((sb + a.b_off_lo) >> 4) | b_lbo;
#pragma unroll
                    for (int k16 = 0; k16 < 4; ++k16) {
                        umma_bf16_if(lead, d, make_desc(a_hi + k16 * a_step), make_desc(b_hi + k16 * b_step), idesc, first ? 0u : 1u);
                        first = 0;
                    }
                    if (g.a_lo_on) {
#pragma unroll
                        for (int k16 = 0; k16 < 4; ++k16) umma_bf16_if(lead, d, make_desc(a_lo + k16 * a_step), make_desc(b_hi + k16 * b_step), idesc, 1u);
                    }
                    if (g.b_lo_on) {
#pragma unroll
                        for (int k16 = 0; k16 < 4; ++k16) umma_bf16_if(lead, d, make_desc(a_hi + k16 * a_step), make_desc(b_lo + k16 * b_step), idesc, 1u);
                    }
                    if (csize == 1) umma_commit_if(lead, bar_empty(stage));
                    else umma_commit_mc_if(lead, bar_empty(stage), cmask);       // frees the stage in every CTA of the cluster
                    if (++stage == (uint32_t)a.stages) { stage = 0; parity ^= 1u; }
                }
                umma_commit_if(lead, bar_tfull(buf));
            }
        }
    } else {
        // =============================================================== epilogue (warps 2-9)
        // tcgen05.ld gives every lane one row of the tile (TMEM lane quarter = warp % 4); the two warps of a quarter take the
        // even / odd 32-column chunks.  A thread therefore owns 128 contiguous bytes of a row of C per chunk: four 256-bit
        // stores (full 32-byte sectors), for the accumulating form four 256-bit loads issued together before them.
        const int q = warp & 3, half = (warp - 2) >> 2;
        uint32_t iter = 0;
        for (int item = cluster_id; item < a.total_items; item += num_clusters, ++iter) {
            const Item it = decode_item(a, item, rank);
            const GemmProblem &g = a.p[it.p];
            const uint32_t buf = iter & 1u;
            mbar_wait(bar_tfull(buf), (iter >> 1) & 1u);     // (also for padding tiles: keeps the phase bookkeeping in step)
            tc_fence_after();
            const uint32_t t0 = tmem_base + buf * 256u + ((uint32_t)(q * 32) << 16);
            const int m = it.mt * kTileM + q * 32 + lane;
            const int col0 = it.nt * g.bn;
            const int ncols = g.n - col0 < g.bn ? g.n - col0 : g.bn;       // valid columns of this n-tile
            const int mode = g.mode, act = g.act;
            if (it.mt * kTileM + q * 32 < g.m) {              // else padding rows (ragged last tile / last group): nothing to store
                const bool row_ok = m < g.m;
                // (mode 3: c is slice 0 of this problem's workspace, [m, ldc] per slice)
                float *crow = g.c + (kOrdered && mode == 3 ? (size_t)it.ks * g.m * g.ldc : 0) + (size_t)(row_ok ? m : 0) * g.ldc + col0;
                const bool fast = ((g.ldc & 7) == 0) && ((reinterpret_cast<uintptr_t>(g.c) & 31) == 0) && ((col0 & 7) == 0);
                for (int cb = half; cb * 32 < ncols; cb += 2) {
                    const int c0 = cb * 32;
                    const int nvalid = ncols - c0 < 32 ? ncols - c0 : 32;
                    float acc[32];
                    tmem_ld16(t0 + c0, acc);
                    if (c0 + 16 < g.bn) tmem_ld16(t0 + c0 + 16, acc + 16);
                    else {
#pragma unroll
                        for (int j = 16; j < 32; ++j) acc[j] = 0.f;
                    }
                    tmem_ld_wait();
                    if (!kOrdered && mode == 2) {             // split-K partial sums
                        if (row_ok) {
#pragma unroll
                            for (int j = 0; j < 32; ++j)
                                if (j < nvalid) atomicAdd(crow + c0 + j, acc[j]);
                        }
                        continue;
                    }
                    if (g.bias) {
                        const float bv = lane < nvalid ? __ldg(g.bias + col0 + c0 + lane) : 0.f;
#pragma unroll
                        for (int j = 0; j < 32; ++j) acc[j] += __shfl_sync(0xffffffffu, bv, j);
                    }
                    if (act == 1) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) acc[j] = fmaxf(acc[j], 0.f);
                    } else if (act == 2) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) acc[j] = tanhf(acc[j]);
                    }
                    if (!row_ok) continue;
                    float *y = crow + c0;
                    if (fast && nvalid == 32) {
                        if (mode == 1) {
                            float old[32];
#pragma unroll
                            for (int v = 0; v < 4; ++v) ld_global_v8(y + 8 * v, old + 8 * v);
#pragma unroll
                            for (int j = 0; j < 32; ++j) acc[j] += old[j];
                        }
#pragma unroll
                        for (int v = 0; v < 4; ++v) st_global_v8(y + 8 * v, acc + 8 * v);
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j)
                            if (j < nvalid) y[j] = mode == 1 ? y[j] + acc[j] : acc[j];
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_tempty(buf));
        }
    }

    tc_fence_before();
    __syncthreads();
    if (csize > 1) cluster_sync_all();          // peers may still multicast into this CTA's shared memory / arrive on its barriers
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    }
}

// Ordered split-K reduction: C = C_in + P_0 + P_1 + ... + P_{S-1}, summed left to right in fp32, for every split problem of
// one ordered launch.  P_s is [m, n_pad] (n_pad = n rounded up to 8) at p + s * m * n_pad.  One thread per 4 columns of a row:
// float4 loads of the partials (read once: evict-first), float4 read-modify-write of C where its layout allows it.
struct ReduceProblem {
    float *c;
    const float *p;
    long long ldc;
    long long unit0;           // first unit (4 columns of a row) of this problem in the launch
    int m, n, n_pad, slices, vec;
};
struct ReduceArgs {
    ReduceProblem p[kMaxProblems];
    int n_problems;
    long long total_units;
};

__global__ void __launch_bounds__(256) splitk_reduce_kernel(const __grid_constant__ ReduceArgs a)
{
    for (long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x; u < a.total_units; u += (long long)gridDim.x * blockDim.x) {
        int i = 0;
        while (i + 1 < a.n_problems && u >= a.p[i + 1].unit0) ++i;
        const ReduceProblem &g = a.p[i];
        const long long r = u - g.unit0;
        const int q4 = g.n_pad >> 2;
        const int row = (int)(r / q4), col = (int)(r - (long long)row * q4) << 2;
        const int nv = g.n - col < 4 ? g.n - col : 4;
        if (nv <= 0) continue;
        const size_t slice = (size_t)g.m * g.n_pad;
        const float *src = g.p + (size_t)row * g.n_pad + col;
        float *dst = g.c + (size_t)row * g.ldc + col;
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        const bool v4 = g.vec && nv == 4;
        if (v4) {
            const float4 t = *reinterpret_cast<const float4 *>(dst);
            acc[0] = t.x; acc[1] = t.y; acc[2] = t.z; acc[3] = t.w;
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) if (j < nv) acc[j] = dst[j];
        }
        for (int s = 0; s < g.slices; ++s) {
            const float4 t = __ldcs(reinterpret_cast<const float4 *>(src + s * slice));
            acc[0] += t.x; acc[1] += t.y; acc[2] += t.z; acc[3] += t.w;
        }
        if (v4) {
            *reinterpret_cast<float4 *>(dst) = make_float4(acc[0], acc[1], acc[2], acc[3]);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) if (j < nv) dst[j] = acc[j];
        }
    }
}

typedef CUresult (*EncodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiled encode_fn()
{
    static EncodeTiled fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess) fn = reinterpret_cast<EncodeTiled>(p);
    }
    return fn;
}

// tensor map of a row-major bf16 [rows, cols] array (ld elements between rows), box = box_rows x 64 columns, SWIZZLE_128B
bool make_map(CUtensorMap *map, const void *base, long long rows, long long cols, long long ld, int box_rows)
{
    EncodeTiled fn = encode_fn();
    if (!fn) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    const cuuint32_t box[2] = {64, (cuuint32_t)box_rows}, estr[2] = {1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace

// CTAs per cluster for this launch: 2 (4 only when forced) if every problem's B tile can be sliced c ways
// (K-major B: bn / c rows, a multiple of the 8-row swizzle atom) and little work is padding (m-tile groups are rounded up
// to c); CN_GEMM_CLUSTER=c overrides (development / A-B timing).
static int pick_cluster(const GemmArgs &args, int n_problems, int forced)
{
    for (int c = forced == 4 ? 4 : 2; c >= 2; c >>= 1) {     // measured: pairs help the weight gradients a little, fours never did
        if (forced && c != forced) continue;
        bool ok = true;
        long long tiles = 0, padded = 0;
        for (int i = 0; i < n_problems; ++i) {
            const GemmProblem &g = args.p[i];
            if (!g.b_mn && (g.bn % (8 * c)) != 0) ok = false;
            tiles += (long long)g.m_tiles * g.n_tiles;
            padded += (long long)((g.m_tiles + c - 1) / c) * c * g.n_tiles;
        }
        if (ok && (forced || padded * 8 <= tiles * 9)) return c;       // at most 12.5 % padding tiles
    }
    return 1;
}

// n-tile of a problem: n rounded up to 16 up to 256; wider problems get even n-tiles (e.g. 320 -> 2 x 160) instead of a
// full tile and a sliver
static int tile_n(int n)
{
    if (n <= 256) return (n + 15) & ~15;
    const int tiles = (n + 255) / 256;
    return (((n + tiles - 1) / tiles) + 15) & ~15;
}

// Slice count of a problem in ordered mode: a pure function of its own (m, n, k, split_k).  split_k = 0 evaluates the auto
// rule of gemm_bf16x3_launch below for the problem alone (share 1) with a fixed budget of 74 clusters of 2 (148 SMs, a
// B200), so that neither the device, the cluster choice nor the other problems of a launch change the summation order.
static constexpr int kOrderedClusters = 74, kOrderedCluster = 2;
static int ordered_slices(const CnGemm &q)
{
    const int kb_total = (q.k + 63) >> 6;
    int split = q.split_k;
    if (split == 0) {
        const int m_tiles = (q.m + kTileM - 1) / kTileM, bn = tile_n(q.n);
        const long long tiles = (long long)((m_tiles + kOrderedCluster - 1) / kOrderedCluster) * ((q.n + bn - 1) / bn);
        split = (int)(2.0 * kOrderedClusters / (double)tiles + 0.5);
        if (split < 1) split = 1;
    }
    if (split > kb_total) split = kb_total;
    const int per = (kb_total + split - 1) / split;
    return (kb_total + per - 1) / per;                          // no empty slices
}

static size_t ordered_slice_floats(const CnGemm &q) { return (size_t)q.m * (size_t)((q.n + 7) & ~7); }

// bytes of the partial-product workspace of an ordered launch (sum over its split problems of slices x m x n_pad x 4) and
// optionally each problem's slice count; pure host code.  Returns NULL on success or a static error string.
const char *gemm_bf16x3_ordered_workspace(const CnGemm *problems, int n_problems, size_t *bytes, int *slices)
{
    if (n_problems < 1 || n_problems > kMaxProblems) return "n_problems out of range";
    size_t total = 0;
    for (int i = 0; i < n_problems; ++i) {
        const CnGemm &q = problems[i];
        if (q.m < 1 || q.n < 1 || q.k < 1) return "m, n, k must be positive";
        if (q.split_k < 0) return "split_k must be >= 0";
        const int s = ordered_slices(q);
        if (slices) slices[i] = s;
        if (s > 1) total += (size_t)s * ordered_slice_floats(q) * sizeof(float);
    }
    *bytes = total;
    return nullptr;
}

// optional device timing of every launch (bench.py's roofline): CUDA events on the launching stream, drained by
// gemm_bf16x3_time_ms
#include <vector>
namespace {
struct GemmTimer {
    bool enabled = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending, pool;
    double flops = 0.0;
} g_timer;
}

void gemm_bf16x3_enable_timing(int enable)
{
    gemm_bf16x3_time_ms(nullptr, nullptr);
    g_timer.enabled = enable != 0;
}

float gemm_bf16x3_time_ms(int *launches, double *flops)
{
    float total = 0.f;
    for (auto &p : g_timer.pending) {
        cudaEventSynchronize(p.second);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, p.first, p.second);
        total += ms;
        g_timer.pool.push_back(p);
    }
    if (launches) *launches = (int)g_timer.pending.size();
    if (flops) *flops = g_timer.flops;
    g_timer.pending.clear();
    g_timer.flops = 0.0;
    return total;
}

// returns NULL on success or a static error string (called from c_abi.cu).  ordered: split problems take their slice count
// from ordered_slices and store their partial tiles into `workspace` (gemm_bf16x3_ordered_workspace bytes, 32-byte aligned),
// then splitk_reduce_kernel adds them to C in slice order.
const char *gemm_bf16x3_launch(const CnGemm *problems, int n_problems, cudaStream_t stream, int *items_out, bool ordered,
                               void *workspace, size_t workspace_bytes)
{
    static int num_sms = 0;
    static bool attr_set[2] = {false, false};
    static int forced_cluster = -1;
    if (n_problems < 1 || n_problems > kMaxProblems) return "n_problems out of range";
    if (num_sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    }
    if (forced_cluster < 0) {
        const char *env = getenv("CN_GEMM_CLUSTER");
        forced_cluster = env ? atoi(env) : 0;
        if (forced_cluster != 1 && forced_cluster != 2 && forced_cluster != 4) forced_cluster = 0;
    }
    if (ordered) {
        size_t need = 0;
        if (const char *msg = gemm_bf16x3_ordered_workspace(problems, n_problems, &need, nullptr)) return msg;
        if (need > 0 && !workspace) return "workspace is NULL";
        if (need > 0 && (reinterpret_cast<uintptr_t>(workspace) & 31)) return "workspace must be 32-byte aligned";
        if (workspace_bytes < need) return "workspace too small (see cn_gemm_bf16x3_ordered_workspace_bytes)";
    }
    if (!attr_set[ordered]) {
        if (cudaFuncSetAttribute(ordered ? gemm_bf16x3_kernel<true> : gemm_bf16x3_kernel<false>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit + 1024) != cudaSuccess)
            return "cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed";
        attr_set[ordered] = true;
    }
    static thread_local ReduceArgs red;
    red.n_problems = 0;
    red.total_units = 0;
    float *ws_next = static_cast<float *>(workspace);
    static thread_local GemmArgs args;
    int max_b_bytes = 0;
    long long total_kb_items = 0;
    for (int i = 0; i < n_problems; ++i) {
        const CnGemm &q = problems[i];
        GemmProblem &g = args.p[i];
        if (q.m < 1 || q.n < 1 || q.k < 1) return "m, n, k must be positive";
        if (!q.a.hi || !q.b.hi || !q.c) return "operand hi pointers and c are required";
        if ((q.a.ld & 7) || (q.b.ld & 7)) return "operand leading dimensions must be multiples of 8 elements";
        if ((reinterpret_cast<uintptr_t>(q.a.hi) | reinterpret_cast<uintptr_t>(q.a.lo) | reinterpret_cast<uintptr_t>(q.b.hi) |
             reinterpret_cast<uintptr_t>(q.b.lo)) & 15) return "operand pointers must be 16-byte aligned";
        if (q.act < 0 || q.act > 2) return "unknown activation";
        const int bn = tile_n(q.n);
        g.bn = bn;
        g.m = q.m; g.n = q.n; g.k = q.k;
        g.m_tiles = (q.m + kTileM - 1) / kTileM;
        g.n_tiles = (q.n + bn - 1) / bn;
        g.a_mn = q.a.mn_major ? 1 : 0; g.b_mn = q.b.mn_major ? 1 : 0;
        g.a_lo_on = q.a.lo ? 1 : 0; g.b_lo_on = q.b.lo ? 1 : 0;
        g.c = q.c; g.ldc = q.ldc; g.bias = q.bias; g.act = q.act;
        const int kb_total = (q.k + 63) >> 6;
        int split = q.split_k;
        if (split < 0) return "split_k must be >= 0";
        if (split > kb_total) split = kb_total;
        if (ordered) split = ordered_slices(q);
        g.split_k = split;                                   // 0 = decided below (auto), 1 = no split
        g.mode = split == 1 ? (q.accumulate ? 1 : 0) : ordered ? 3 : 2;
        if (g.mode >= 2 && (q.bias || q.act)) return "split-K products cannot carry a bias or an activation";
        if (g.mode == 3) {                                   // the kernel stores slice s at c + s * m * ldc
            ReduceProblem &r = red.p[red.n_problems++];
            r.c = q.c; r.ldc = q.ldc; r.p = ws_next;
            r.m = q.m; r.n = q.n; r.n_pad = (q.n + 7) & ~7; r.slices = split;
            r.vec = (q.ldc & 3) == 0 && (reinterpret_cast<uintptr_t>(q.c) & 15) == 0;
            r.unit0 = red.total_units;
            red.total_units += (long long)q.m * (r.n_pad >> 2);
            g.c = ws_next; g.ldc = r.n_pad;
            ws_next += (size_t)split * ordered_slice_floats(q);
        }
        const int b_tile = g.b_mn ? ((bn + 63) / 64) * 8192 : bn * 128;
        g.stage_tx = (unsigned)(kABytes * (1 + g.a_lo_on) + b_tile * (1 + g.b_lo_on));
        if (b_tile > max_b_bytes) max_b_bytes = b_tile;
        total_kb_items += (long long)kb_total * g.m_tiles * g.n_tiles;
    }
    const int cluster = forced_cluster == 1 ? 1 : pick_cluster(args, n_problems, forced_cluster);
    args.cluster = cluster;
    for (int i = 0; i < n_problems; ++i) {
        const CnGemm &q = problems[i];
        GemmProblem &g = args.p[i];
        // A: K-major [m, k] box 128 rows; MN-major [k, m] box 64 k-rows.  B: this CTA's 1/c slice of the tile -- K-major
        // [n, k] box bn/c rows; MN-major [k, n] box 64/c k-rows (of every 64-wide atom).
        const int b_rows = g.b_mn ? 64 / cluster : g.bn / cluster;
        const bool ok = (g.a_mn ? make_map(&g.a_hi, q.a.hi, q.k, q.m, q.a.ld, 64) : make_map(&g.a_hi, q.a.hi, q.m, q.k, q.a.ld, kTileM)) &&
                        (!q.a.lo || (g.a_mn ? make_map(&g.a_lo, q.a.lo, q.k, q.m, q.a.ld, 64) : make_map(&g.a_lo, q.a.lo, q.m, q.k, q.a.ld, kTileM))) &&
                        (g.b_mn ? make_map(&g.b_hi, q.b.hi, q.k, q.n, q.b.ld, b_rows) : make_map(&g.b_hi, q.b.hi, q.n, q.k, q.b.ld, b_rows)) &&
                        (!q.b.lo || (g.b_mn ? make_map(&g.b_lo, q.b.lo, q.k, q.n, q.b.ld, b_rows) : make_map(&g.b_lo, q.b.lo, q.n, q.k, q.b.ld, b_rows)));
        if (!ok) return "cuTensorMapEncodeTiled failed (driver entry point missing, or an operand it cannot describe)";
        g.m_groups = (g.m_tiles + cluster - 1) / cluster;
        g.b_slice_bytes = b_rows * 128;
    }
    int max_clusters = num_sms / cluster;
    if (cluster > 1) {      // clusters that can be co-resident (GPC boundaries): a persistent grid larger than that runs in two waves
        static int active[5] = {0, 0, 0, 0, 0};
        if (active[cluster] == 0) {
            cudaLaunchConfig_t probe = {};
            probe.gridDim = dim3((unsigned)num_sms / cluster * cluster); probe.blockDim = dim3(kThreads);
            probe.dynamicSmemBytes = kSmemLimit + 1024;
            cudaLaunchAttribute pa[1];
            pa[0].id = cudaLaunchAttributeClusterDimension;
            pa[0].val.clusterDim.x = (unsigned)cluster; pa[0].val.clusterDim.y = 1; pa[0].val.clusterDim.z = 1;
            probe.attrs = pa; probe.numAttrs = 1;
            int n = 0;
            if (cudaOccupancyMaxActiveClusters(&n, gemm_bf16x3_kernel<false>, &probe) != cudaSuccess || n < 1) n = num_sms / cluster;
            active[cluster] = n;
        }
        if (active[cluster] < max_clusters) max_clusters = active[cluster];
    }
    // split-K "auto" (0): cut the k range so that the launch has about two items per cluster, shared out in proportion to the work
    int item0 = 0;
    for (int i = 0; i < n_problems; ++i) {
        GemmProblem &g = args.p[i];
        const int kb_total = (g.k + 63) >> 6;
        if (g.split_k == 0) {
            const long long tiles = (long long)g.m_groups * g.n_tiles;
            const double share = (double)kb_total * g.m_tiles * g.n_tiles / (double)total_kb_items;
            int split = (int)(share * 2.0 * max_clusters / (double)tiles + 0.5);
            if (split < 1) split = 1;
            if (split > kb_total) split = kb_total;
            g.split_k = split;
        }
        g.kb_per_split = (kb_total + g.split_k - 1) / g.split_k;
        g.split_k = (kb_total + g.kb_per_split - 1) / g.kb_per_split;     // no empty slices
        g.item0 = item0;
        g.items = g.split_k * g.m_groups * g.n_tiles;
        item0 += g.items;
    }
    args.n_problems = n_problems;
    args.total_items = item0;
    args.b_off_lo = max_b_bytes;
    args.stage_bytes = 2 * kABytes + 2 * max_b_bytes;
    int stages = (kSmemLimit - kScratchBytes - 256) / args.stage_bytes;
    if (stages > kMaxStages) stages = kMaxStages;
    if (stages < 2) return "tile does not fit two pipeline stages";
    args.stages = stages;
    const int smem = stages * args.stage_bytes + kScratchBytes + 256 + 1024;
    const int clusters = args.total_items < max_clusters ? args.total_items : max_clusters;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(clusters * cluster));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = (size_t)smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (g_timer.enabled) {
        std::pair<cudaEvent_t, cudaEvent_t> p;
        if (!g_timer.pool.empty()) { p = g_timer.pool.back(); g_timer.pool.pop_back(); }
        else { cudaEventCreate(&p.first); cudaEventCreate(&p.second); }
        cudaEventRecord(p.first, stream);
        g_timer.pending.push_back(p);
        for (int i = 0; i < n_problems; ++i) g_timer.flops += 2.0 * problems[i].m * (double)problems[i].n * problems[i].k;
    }
    cudaError_t err = ordered ? cudaLaunchKernelEx(&cfg, gemm_bf16x3_kernel<true>, args) : cudaLaunchKernelEx(&cfg, gemm_bf16x3_kernel<false>, args);
    if (err == cudaSuccess && red.n_problems > 0) {
        long long blocks = (red.total_units + 255) / 256;
        if (blocks > 148 * 4) blocks = 148 * 4;
        splitk_reduce_kernel<<<(unsigned)blocks, 256, 0, stream>>>(red);
        err = cudaGetLastError();
    }
    if (g_timer.enabled) cudaEventRecord(g_timer.pending.back().second, stream);
    if (items_out) *items_out = args.total_items;
    return err == cudaSuccess ? nullptr : cudaGetErrorString(err);
}
