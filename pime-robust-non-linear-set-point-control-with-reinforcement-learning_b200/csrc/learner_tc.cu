// learner_tc.cu -- the PPO minibatch step of AgentPPO.update_net (elegantrl/agent.py:635-658) for LARGE batches
// (4096 .. 2^20 rows: BASELINE configs[4] trains on 131 072-row minibatches) on the tcgen05 tensor cores.
//
// The small-batch step (learner.cu) keeps R rows per CTA and streams every weight matrix past them; at thousands of rows
// that re-reads the weights once per 2-8 rows.  Here the ratio is inverted: the batch is cut into tiles of 128 rows (the
// 128 TMEM lanes = the M of every tcgen05.mma), the layers run one after the other as GEMMs over all row tiles, and each
// GEMM CTA streams its operands through shared memory with cp.async.bulk (TMA) exactly once.
//
// fp32-grade sums on fp16 tensor cores: every operand X is kept as X = X_hi + X_lo (two fp16 numbers, 22 significant bits)
// and every product is three MMAs, A_hi B_hi + A_lo B_hi + A_hi B_lo (the dropped A_lo B_lo term is 2^-22 relative),
// accumulated in fp32 in TMEM -- the same split the rollout engine uses for its first layer (tc_mlp.cuh).
//
// "T-format" of a [rows][units] matrix (activations, pre-activation gradients, weights): tiles of 128 rows x 64 units, a
// hi block then a lo block per tile, each block [8 unit groups][128 rows][8 fp16] = 16 KB.  That is the no-swizzle canonical
// shared-memory operand layout of tcgen05, so a block is ONE bulk copy, and it is BOTH
//   * a K-major operand (rows = M or N of the MMA, units = K): forward  Z = A W^T  and data gradient  dA = dZ W, and
//   * an MN-major operand (units = M or N, rows = K): weight gradient  dW = dZ^T A, contracted over the batch rows,
// -- the same bytes, only the descriptor strides and the major bits of the instruction descriptor differ -- so no matrix
// is ever transposed.  Every GEMM epilogue (TMEM -> registers -> activation / derivative -> hi, lo) writes its result
// straight back in T-format for the next GEMM.
//
// One step = weights -> T-format (tiny), gather (+ first-layer operand with a ones column that carries the bias), forward
// GEMMs, the objectives kernel (clipped surrogate / entropy / SmoothL1, output layers, their gradients), data-gradient
// GEMMs, weight-gradient GEMMs into a flat fp32 gradient in theta's layout; the caller all-reduces that buffer when the job
// is data parallel and applies Adam with pime_ppo_apply_grad (learner.cu).
#include "ppo_common.cuh"

namespace pime {
namespace tcl {

using tc::bulk_g2s; using tc::elect_one; using tc::fence_barrier_init; using tc::make_desc; using tc::mbar_arrive_expect_tx;
using tc::mbar_init; using tc::mbar_wait; using tc::mma_commit; using tc::mma_f16; using tc::smem_u32; using tc::tc_fence_after;
using tc::tc_fence_before; using tc::tmem_alloc; using tc::tmem_dealloc; using tc::tmem_ld32;
using ppo::Net;

constexpr int kBlk = 16384;        // bytes of one T-format block: [8 unit groups][128 rows][8 fp16]
constexpr int kUg = 2048;          // bytes of one unit group: 128 rows x 16 B
constexpr int kMaxProb = 8;
constexpr int kBiasCol = 63;       // first-layer operand: unit 63 of the gathered row is 1.0, column 63 of the padded weight is the bias

enum { ACT_TANH = 0, ACT_RELU = 1 };

__host__ __device__ __forceinline__ size_t tblock(int row_tile, int chunks, int chunk, int hl) {
    return ((size_t)((size_t)row_tile * chunks + chunk) * 2 + hl) * kBlk;
}

// x = hi + lo with hi = fp16(x), lo = fp16(x - hi): pairs of values through the packed conversions
__device__ __forceinline__ void split8(const float (&x)[8], uint4 &hi, uint4 &lo) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const __half2 hh = __floats2half2_rn(x[2 * q], x[2 * q + 1]);
        const float2 back = __half22float2(hh);
        const __half2 ll = __floats2half2_rn(x[2 * q] - back.x, x[2 * q + 1] - back.y);
        h[q] = *reinterpret_cast<const uint32_t *>(&hh);
        l[q] = *reinterpret_cast<const uint32_t *>(&ll);
    }
    hi = make_uint4(h[0], h[1], h[2], h[3]);
    lo = make_uint4(l[0], l[1], l[2], l[3]);
}
__device__ __forceinline__ void join8(const uint4 &hi, const uint4 &lo, float (&x)[8]) {
    const uint32_t h[4] = {hi.x, hi.y, hi.z, hi.w}, l[4] = {lo.x, lo.y, lo.z, lo.w};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float2 a = __half22float2(*reinterpret_cast<const __half2 *>(&h[q]));
        const float2 b = __half22float2(*reinterpret_cast<const __half2 *>(&l[q]));
        x[2 * q] = a.x + b.x;
        x[2 * q + 1] = a.y + b.y;
    }
}
__device__ __forceinline__ float act_grad(int act, float a) { return act == ACT_TANH ? 1.0f - a * a : (a > 0.0f ? 1.0f : 0.0f); }

// tanh to ~4e-7 absolute without the slow branches of tanhf: 1 - 2 / (1 + e^{2x}) = 1 - 2 rcp(1 + ex2(2 log2(e) x)) with
// ex2.approx / rcp.approx (2^-22, 1 ulp); the clamp keeps e^{2x} finite.  7 instructions, 2 of them MUFU.  (The rollout
// engine's tanh.approx.f32, 5e-4, is too coarse for fp32-grade gradients.)
__device__ __forceinline__ float tanh_acc(float x) {
    float t, r;
    const float y = 2.8853900817779268f * fminf(fmaxf(x, -15.0f), 15.0f);
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(y));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(t + 1.0f));
    return fmaf(-2.0f, r, 1.0f);
}

// Column sums of a [32 lanes][N values] register tile in N - 1 + (32 / N >= 1 ? log2(32 / N) : 0) shuffles: at every stage a
// lane keeps one half of its values and receives the partner's copy of that half ("transpose-reduce").  Returns, in lane l,
// the sum over the 32 lanes of column col_of(l); for N = 8 four lanes hold each column after three stages and two plain
// butterfly stages finish the sum (every lane of a group of four then holds the same total).
template <int N> __device__ __forceinline__ float colsum(float (&v)[N], int lane, int &col) {
    static_assert(N == 8 || N == 32, "tile width");
    int base = 0;
#pragma unroll
    for (int w = N / 2, o = 16; w >= 1; w >>= 1, o >>= 1) {
        const bool upper = (lane & o) != 0;
#pragma unroll
        for (int i = 0; i < w; ++i) {
            const float keep = upper ? v[i + w] : v[i];
            const float send = upper ? v[i] : v[i + w];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
        base += upper ? w : 0;
    }
    float s = v[0];
    if (N == 8) {
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        s += __shfl_xor_sync(0xffffffffu, s, 1);
    }
    col = base;
    return s;
}

// instruction descriptor kind::f16, D = f32, A = B = f16; MAJOR = 1: both operands MN-major (bits 15, 16)
__host__ __device__ constexpr uint32_t idesc(int M, int N, int mn_major) {
    return tc::make_idesc(M, N) | (mn_major ? ((1u << 15) | (1u << 16)) : 0u);
}

// ------------------------------------------------------------------------------------------------ forward / data-gradient GEMM
// OUT[rows][n] = epi( sum_k A[rows][k] * W[n][k] ), both operands K-major.  One CTA = one 128-row tile x one tile of <= 128
// output units; the K chunks (64 units) stream through a 3-stage ring.
struct GemmProb {
    const uint8_t *A; int a_chunks, a_c0, kc;            // A operand: T-format matrix, chunks per row tile, first chunk, chunks contracted
    const uint8_t *W; int w_chunks;                      // W operand: T-format [N rows][K units]; block (n tile, chunk)
    int n_tiles, n_cols;                                 // output tiles of this problem, MMA N of a tile (64 or 128)
    int mode;                                            // 0: forward (bias + activation), 1: data gradient (x act'(APREV))
    int act;
    const float *bias;                                   // forward: fp32 bias[N] (NULL: the bias rides in the operand's ones column)
    uint8_t *OUT; int out_chunks, out_c0;                // result, T-format; unit = out_c0 * 64 + tile * 128 + column
    const uint8_t *APREV; int ap_chunks, ap_c0;          // data gradient: the activation whose derivative multiplies
    float *db, *db2; int db_split;                       // data gradient: bias gradients of the layer(s) that produced APREV: column sums of the
                                                         // result go to db[unit] (unit < db_split) or db2[unit - db_split]; NULL: none
    float db_scale;                                      // 1 / (gradient scale of this net), see StepCommon::dz_scale
};
struct GemmBatch {
    GemmProb p[kMaxProb];
    int n, row_tiles;
};

// One 32-column piece of a GEMM epilogue for the row of this thread: forward (bias + activation) or data gradient
// (x act'(stored activation)), hi / lo split, T-format stores.  Data gradient: returns, in lane l, the sum over the warp's 32
// rows of column l of the piece (the bias gradient of the producing layer).
__device__ __forceinline__ float epi_piece(const GemmProb &P, int rt, int nt, int j, int row, int lane, float (&v)[32]) {
    if (P.mode == 0) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int unit = nt * 128 + j * 32 + q * 8;     // output unit inside the problem
            float x[8], bz[8];
            if (P.bias) {   // every bias vector starts on a 16-byte boundary of theta? not guaranteed: scalar loads unless aligned
                if ((reinterpret_cast<uintptr_t>(P.bias + unit) & 15) == 0) {
                    const float4 b0 = __ldg(reinterpret_cast<const float4 *>(P.bias + unit)), b1 = __ldg(reinterpret_cast<const float4 *>(P.bias + unit) + 1);
                    bz[0] = b0.x; bz[1] = b0.y; bz[2] = b0.z; bz[3] = b0.w; bz[4] = b1.x; bz[5] = b1.y; bz[6] = b1.z; bz[7] = b1.w;
                } else {
#pragma unroll
                    for (int e = 0; e < 8; ++e) bz[e] = __ldg(P.bias + unit + e);
                }
            } else {
#pragma unroll
                for (int e = 0; e < 8; ++e) bz[e] = 0.0f;
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const float z = v[q * 8 + e] + bz[e];
                x[e] = P.act == ACT_TANH ? tanh_acc(z) : fmaxf(z, 0.0f);
            }
            uint4 hi, lo;
            split8(x, hi, lo);
            const int ou = P.out_c0 * 64 + unit;
            const size_t o = (size_t)(((ou & 63) >> 3) * 128 + row) * 16;
            *reinterpret_cast<uint4 *>(P.OUT + tblock(rt, P.out_chunks, ou >> 6, 0) + o) = hi;
            *reinterpret_cast<uint4 *>(P.OUT + tblock(rt, P.out_chunks, ou >> 6, 1) + o) = lo;
        }
        return 0.0f;
    }
    uint4 ah[4], al[4];                       // the four 8-unit groups of the activation: loads in flight together
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int pu = P.ap_c0 * 64 + nt * 128 + j * 32 + q * 8;
        const size_t o = (size_t)(((pu & 63) >> 3) * 128 + row) * 16;
        ah[q] = *reinterpret_cast<const uint4 *>(P.APREV + tblock(rt, P.ap_chunks, pu >> 6, 0) + o);
        al[q] = *reinterpret_cast<const uint4 *>(P.APREV + tblock(rt, P.ap_chunks, pu >> 6, 1) + o);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        float a[8], x[8];
        join8(ah[q], al[q], a);
#pragma unroll
        for (int e = 0; e < 8; ++e) { x[e] = v[q * 8 + e] * act_grad(P.act, a[e]); v[q * 8 + e] = x[e]; }
        uint4 hi, lo;
        split8(x, hi, lo);
        const int ou = P.out_c0 * 64 + nt * 128 + j * 32 + q * 8;
        const size_t o = (size_t)(((ou & 63) >> 3) * 128 + row) * 16;
        *reinterpret_cast<uint4 *>(P.OUT + tblock(rt, P.out_chunks, ou >> 6, 0) + o) = hi;
        *reinterpret_cast<uint4 *>(P.OUT + tblock(rt, P.out_chunks, ou >> 6, 1) + o) = lo;
    }
    if (!P.db) return 0.0f;
    int col;
    return colsum<32>(v, lane, col);          // col == lane
}

// 1: 65 KB per CTA, three CTAs per SM overlap one another's load / MMA / epilogue phases (3 stages, one CTA per SM: 2.21 ms
// against 1.46 ms for this single stage)
constexpr int kGemmStages = 1;
constexpr int kGemmStage = 4 * kBlk;                      // A_hi, A_lo, W_hi, W_lo
constexpr int kGemmSmem = kGemmStages * kGemmStage + 1024;
constexpr int kGemmThreads = 320;                         // warp 0: TMA, warp 1: MMA, warps 2-9: epilogue (two threads per row: column halves)

__global__ void __launch_bounds__(kGemmThreads, kGemmStages == 1 ? 3 : 1) gemm_kk_kernel(const __grid_constant__ GemmBatch gb) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const GemmProb &P = gb.p[blockIdx.z];
    const int nt = blockIdx.x, rt = blockIdx.y;
    if (nt >= P.n_tiles) return;
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + kGemmStages * kGemmStage);
    uint64_t *empty = full + kGemmStages;
    uint64_t *acc_ready = empty + kGemmStages;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(acc_ready + 1);
    float *s_db = reinterpret_cast<float *>(tmem_slot + 2);   // [128] column sums (data gradient)
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int s = 0; s < kGemmStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(acc_ready, 1);
        fence_barrier_init();
    }
    if (tid < 128) s_db[tid] = 0.0f;
    if (warp == 1) tmem_alloc(tmem_slot, 128);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            uint32_t st = 0, ph = 0;
            for (int c = 0; c < P.kc; ++c) {
                mbar_wait(&empty[st], ph ^ 1);
                uint8_t *dst = smem + st * kGemmStage;
                const uint32_t wbytes = (uint32_t)P.n_cols * 128u;   // the n_cols rows of every unit group: 8 groups x n_cols x 16 B
                mbar_arrive_expect_tx(&full[st], 2 * kBlk + 2 * (P.n_cols == 128 ? kBlk : 0) + (P.n_cols == 128 ? 0 : 2 * wbytes));
                bulk_g2s(dst, P.A + tblock(rt, P.a_chunks, P.a_c0 + c, 0), kBlk, &full[st]);
                bulk_g2s(dst + kBlk, P.A + tblock(rt, P.a_chunks, P.a_c0 + c, 1), kBlk, &full[st]);
                if (P.n_cols == 128) {
                    bulk_g2s(dst + 2 * kBlk, P.W + tblock(nt, P.w_chunks, c, 0), kBlk, &full[st]);
                    bulk_g2s(dst + 3 * kBlk, P.W + tblock(nt, P.w_chunks, c, 1), kBlk, &full[st]);
                } else {   // 64 output units: rows 0..63 of each unit group (1 KB pieces)
                    for (int hl = 0; hl < 2; ++hl)
                        for (int ug = 0; ug < 8; ++ug)
                            bulk_g2s(dst + (2 + hl) * kBlk + ug * kUg, P.W + tblock(nt, P.w_chunks, c, hl) + ug * kUg, (uint32_t)P.n_cols * 16u, &full[st]);
                }
                if (++st == kGemmStages) { st = 0; ph ^= 1; }
            }
        }
    } else if (warp == 1) {
        uint32_t st = 0, ph = 0;
        const uint32_t id = P.n_cols == 128 ? idesc(128, 128, 0) : idesc(128, 64, 0);
        for (int c = 0; c < P.kc; ++c) {
            mbar_wait(&full[st], ph);
            tc_fence_after();
            if (elect_one()) {
                const uint32_t base = smem_u32(smem) + st * kGemmStage;
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {   // K = 16 per MMA = two unit groups
                    const uint64_t a_hi = make_desc(base + kk * 2 * kUg, kUg, 128), a_lo = make_desc(base + kBlk + kk * 2 * kUg, kUg, 128);
                    const uint64_t w_hi = make_desc(base + 2 * kBlk + kk * 2 * kUg, kUg, 128), w_lo = make_desc(base + 3 * kBlk + kk * 2 * kUg, kUg, 128);
                    mma_f16(tmem, a_hi, w_hi, id, (c == 0 && kk == 0) ? 0u : 1u);
                    mma_f16(tmem, a_lo, w_hi, id, 1u);
                    mma_f16(tmem, a_hi, w_lo, id, 1u);
                }
                mma_commit(&empty[st]);
                if (c == P.kc - 1) mma_commit(acc_ready);
            }
            __syncwarp();
            if (++st == kGemmStages) { st = 0; ph ^= 1; }
        }
    } else {
        mbar_wait(acc_ready, 0);
        tc_fence_after();
        const int row = 32 * (warp & 3) + lane;          // TMEM lane quarter = warp % 4; warps 2-5 / 6-9 take the two column halves
        const int half = (warp - 2) >> 2;
        const uint32_t taddr = tmem + ((uint32_t)(32 * (warp & 3)) << 16);
        const int jn = P.n_cols / 64;                     // 32-column pieces per half
        for (int j = half * jn; j < (half + 1) * jn; ++j) {
            float v[32];
            tmem_ld32(taddr + j * 32, v);
            const float cs = epi_piece(P, rt, nt, j, row, lane, v);
            if (P.mode == 1 && P.db) atomicAdd(&s_db[j * 32 + lane], cs);
        }
        tc_fence_before();
    }
    __syncthreads();
    if (P.mode == 1 && P.db && tid < P.n_cols) {
        const int unit = nt * 128 + tid;
        atomicAdd(unit < P.db_split ? P.db + unit : P.db2 + (unit - P.db_split), s_db[tid] * P.db_scale);
    }
    if (warp == 1) tc_fence_after();
    if (warp == 1) tmem_dealloc(tmem, 128);
}


// ------------------------------------------------------------------------------------------------ weight-gradient GEMM
// G[m][n] = sum over the batch rows of MOP[row][m] * NOP[row][n]: both operands MN-major (units = M / N of the MMA, rows = K),
// read from the very same T-format blocks.  One CTA = 128 m-units x (64 or 128) n-units, looping over the row tiles
// blockIdx.y, blockIdx.y + gridDim.y, ...; the partial sums go to the flat gradient with atomics.
struct WgProb {
    const uint8_t *MOP; int m_chunks, m_c0, m_tiles;     // operand whose units become the MMA's M (tiles of 128 units = 2 chunks)
    const uint8_t *NOP; int n_chunks, n_c0, n_tiles, n_cols;   // operand whose units become the MMA's N (n_cols = 64: one chunk per tile)
    int swap;                                            // 0: (m, n) = (output unit, input unit); 1: the other way round
    int w_off, ldw;                                      // dW[out][in] -> grad[w_off + out * ldw + (in - in_lo)] for in in [in_lo, in_hi)
    int in_lo, in_hi, out_n;
    int bias_col, b_off;                                 // first layers: input unit bias_col (the ones column) -> grad[b_off + out]; -1: none
    float scale;                                         // 1 / (gradient scale of this net)
};
struct WgBatch {
    WgProb p[kMaxProb];
    int n, row_tiles;
    float *grad;
};
constexpr int kWgSmem = 12 * kBlk + 1024;   // two hi buffers (M_hi 2 blocks + N_hi 2 blocks) + one lo buffer
constexpr int kWgThreads = 192;

// Shared memory: H[0], H[1] (the hi blocks of row tile i, i + 1: 64 KB each) and L (the lo blocks of row tile i: 64 KB).  A row
// tile's products are  M_hi N_hi  (needs H only)  then  M_lo N_hi + M_hi N_lo  (needs L too): while those run, the hi blocks
// of the next row tile are already landing in the other H buffer, and its lo blocks follow as soon as L is released.
__global__ void __launch_bounds__(kWgThreads, 1) wgrad_mn_kernel(const __grid_constant__ WgBatch wb) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const WgProb &P = wb.p[blockIdx.z];
    if ((int)blockIdx.x >= P.m_tiles * P.n_tiles) return;
    const int mt = blockIdx.x / P.n_tiles, ntile = blockIdx.x % P.n_tiles;
    uint64_t *h_full = reinterpret_cast<uint64_t *>(smem + 12 * kBlk);   // [2]
    uint64_t *h_empty = h_full + 2;                                      // [2]
    uint64_t *l_full = h_empty + 2, *l_empty = l_full + 1, *acc_ready = l_empty + 1;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(acc_ready + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int b = 0; b < 2; ++b) { mbar_init(&h_full[b], 1); mbar_init(&h_empty[b], 1); }
        mbar_init(l_full, 1); mbar_init(l_empty, 1); mbar_init(acc_ready, 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, 128);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const int my_tiles = (wb.row_tiles - (int)blockIdx.y + (int)gridDim.y - 1) / (int)gridDim.y;
    const int nblk = P.n_cols == 128 ? 2 : 1;            // chunks of the N operand per tile
    uint8_t *sL = smem + 8 * kBlk;
    if (warp == 0) {
        if (lane == 0) {
            for (int i = 0; i < my_tiles; ++i) {
                const int rt = blockIdx.y + i * gridDim.y;
                const uint32_t buf = (uint32_t)i & 1u;
                uint8_t *sH = smem + buf * 4 * kBlk;
                for (int hl = 0; hl < 2; ++hl) {
                    uint64_t *bar = hl == 0 ? &h_full[buf] : l_full;
                    uint8_t *dst = hl == 0 ? sH : sL;
                    if (hl == 0) mbar_wait(&h_empty[buf], (((uint32_t)i >> 1) & 1u) ^ 1u);
                    else mbar_wait(l_empty, ((uint32_t)i & 1u) ^ 1u);
                    mbar_arrive_expect_tx(bar, (2 + nblk) * kBlk);
                    for (int c = 0; c < 2; ++c) bulk_g2s(dst + c * kBlk, P.MOP + tblock(rt, P.m_chunks, P.m_c0 + 2 * mt + c, hl), kBlk, bar);
                    for (int c = 0; c < nblk; ++c)
                        bulk_g2s(dst + (2 + c) * kBlk, P.NOP + tblock(rt, P.n_chunks, P.n_c0 + nblk * ntile + c, hl), kBlk, bar);
                }
            }
        }
    } else if (warp == 1) {
        const uint32_t id = P.n_cols == 128 ? idesc(128, 128, 1) : idesc(128, 64, 1);
        for (int i = 0; i < my_tiles; ++i) {
            const uint32_t buf = (uint32_t)i & 1u;
            const uint32_t hb = smem_u32(smem) + buf * 4 * kBlk, lb = smem_u32(sL);
            // MN-major, no swizzle: K groups (8 rows) 128 B apart (LBO), MN groups (8 units) one unit group apart (SBO);
            // 16 batch rows per MMA = 256 B further into every unit group
            mbar_wait(&h_full[buf], ((uint32_t)i >> 1) & 1u);
            tc_fence_after();
            if (elect_one()) {
#pragma unroll
                for (int kk = 0; kk < 8; ++kk)
                    mma_f16(tmem, make_desc(hb + kk * 256, 128, kUg), make_desc(hb + 2 * kBlk + kk * 256, 128, kUg), id, (i == 0 && kk == 0) ? 0u : 1u);
            }
            __syncwarp();
            mbar_wait(l_full, (uint32_t)i & 1u);
            tc_fence_after();
            if (elect_one()) {
#pragma unroll
                for (int kk = 0; kk < 8; ++kk) {
                    mma_f16(tmem, make_desc(lb + kk * 256, 128, kUg), make_desc(hb + 2 * kBlk + kk * 256, 128, kUg), id, 1u);   // M_lo N_hi
                    mma_f16(tmem, make_desc(hb + kk * 256, 128, kUg), make_desc(lb + 2 * kBlk + kk * 256, 128, kUg), id, 1u);   // M_hi N_lo
                }
                mma_commit(l_empty);
                mma_commit(&h_empty[buf]);
                if (i == my_tiles - 1) mma_commit(acc_ready);
            }
            __syncwarp();
        }
    } else if (my_tiles > 0) {
        mbar_wait(acc_ready, 0);
        tc_fence_after();
        const int m_unit = mt * 128 + 32 * (warp & 3) + lane;
        const uint32_t taddr = tmem + ((uint32_t)(32 * (warp & 3)) << 16);
        for (int j = 0; j < P.n_cols / 32; ++j) {
            float v[32];
            tmem_ld32(taddr + j * 32, v);
#pragma unroll
            for (int e = 0; e < 32; ++e) {
                const int n_unit = ntile * P.n_cols + j * 32 + e;
                const int out = P.swap ? n_unit : m_unit, in = P.swap ? m_unit : n_unit;
                if (out < P.out_n) {
                    if (in >= P.in_lo && in < P.in_hi) atomicAdd(wb.grad + P.w_off + (size_t)out * P.ldw + (in - P.in_lo), v[e] * P.scale);
                    else if (in == P.bias_col) atomicAdd(wb.grad + P.b_off + out, v[e] * P.scale);
                }
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, 128);
}

// ------------------------------------------------------------------------------------------------ small kernels
// fp32 torch-layout weights (theta) -> T-format hi / lo blocks: W (rows = output units) and, for hidden layers, W^T.
struct WLayer {
    int w_off, b_off, N, K;      // W[N][K], bias[N] in theta
    int kpad, k_lo, first;       // first layers: K padded to 64, source column j at k_lo + j, the bias in column kBiasCol
    long long dst, dst_t;        // byte offsets in the work buffer (dst_t < 0: no transposed copy)
};
struct WSplit {
    WLayer l[kMaxProb];
    int n;
};
__global__ void __launch_bounds__(256) split_weights_kernel(const __grid_constant__ WSplit ws, const float *__restrict__ theta, uint8_t *work) {
    const WLayer L = ws.l[blockIdx.y];
    const int rows_pad = (L.N + 127) / 128 * 128;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < rows_pad * L.kpad; e += gridDim.x * blockDim.x) {
        const int n = e / L.kpad, k = e % L.kpad;
        float v = 0.0f;
        if (n < L.N) {
            if (L.first) v = (k >= L.k_lo && k < L.k_lo + L.K) ? theta[L.w_off + n * L.K + (k - L.k_lo)] : (k == kBiasCol ? theta[L.b_off + n] : 0.0f);
            else v = theta[L.w_off + n * L.K + k];
        }
        __half hi, lo;
        tc::split_h(v, hi, lo);
        const size_t o = (size_t)(((k & 63) >> 3) * 128 + (n & 127)) * 16 + (k & 7) * 2;
        *reinterpret_cast<__half *>(work + L.dst + tblock(n >> 7, L.kpad / 64, k >> 6, 0) + o) = hi;
        *reinterpret_cast<__half *>(work + L.dst + tblock(n >> 7, L.kpad / 64, k >> 6, 1) + o) = lo;
        if (L.dst_t >= 0 && n < L.N) {   // W^T: rows = input units (K, a multiple of 128 for hidden layers), units = output units
            const int npad = (L.N + 63) / 64 * 64;
            const size_t ot = (size_t)(((n & 63) >> 3) * 128 + (k & 127)) * 16 + (n & 7) * 2;
            *reinterpret_cast<__half *>(work + L.dst_t + tblock(k >> 7, npad / 64, n >> 6, 0) + ot) = hi;
            *reinterpret_cast<__half *>(work + L.dst_t + tblock(k >> 7, npad / 64, n >> 6, 1) + ot) = lo;
        }
    }
}

struct StepCommon {
    const float *buf_state, *buf_action, *buf_r_sum, *buf_logprob, *buf_adv;
    const int64_t *idx;
    int B, S, row_tiles;
    float ratio_clip, lambda_entropy, lr, beta1, beta2;
    int *step_dev;
    float *adam_c, *loss_ring;
    int ring_len;
    float *grad;
    int n_theta;
    float *rowv;        // [row_tiles * 128][4]: action, r_sum, old logprob, advantage
    float *inv_cs;      // 1 / (r_sum.std() + 1e-5) of the minibatch
    const float *theta;
    // Gradient scaling.  d united / d out is O(1 / B) per row (and another 1 / std(r_sum) for the critic): at B = 2^17 the
    // pre-activation gradients would sit in fp16's subnormal range and lose the lo part.  They are therefore carried
    // multiplied by a power of two (exact), per net, through the whole data-gradient chain (which is linear in them), and
    // every sum that leaves for the fp32 gradient is multiplied by the inverse.  Saturated at +-6e4 instead of overflowing.
    float dz_scale[2];
};

// gathered rows -> first-layer operand X (64 units: the S observations, zeros, 1.0 in unit kBiasCol), T-format
__global__ void __launch_bounds__(128) gather_kernel(const StepCommon c, uint8_t *X) {
    const int rt = blockIdx.x, row = threadIdx.x, b = rt * 128 + row;
    const bool live = b < c.B;
    const int64_t i = live ? __ldg(c.idx + b) : 0;
    if (rt == 0 && row == 0) ppo::adam_prepare(c.step_dev, c.lr, c.beta1, c.beta2, c.adam_c);
#pragma unroll
    for (int ug = 0; ug < 8; ++ug) {
        float x[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int u = ug * 8 + e;
            x[e] = u == kBiasCol ? 1.0f : (live && u < c.S ? __ldg(c.buf_state + i * c.S + u) : 0.0f);
        }
        uint4 hi, lo;
        split8(x, hi, lo);
        const size_t o = (size_t)(ug * 128 + row) * 16;
        *reinterpret_cast<uint4 *>(X + tblock(rt, 1, 0, 0) + o) = hi;
        *reinterpret_cast<uint4 *>(X + tblock(rt, 1, 0, 1) + o) = lo;
    }
    float4 rv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (live) rv = make_float4(__ldg(c.buf_action + i), __ldg(c.buf_r_sum + i), __ldg(c.buf_logprob + i), __ldg(c.buf_adv + i));
    reinterpret_cast<float4 *>(c.rowv)[b] = rv;
}

// r_sum.std() of the minibatch (agent.py:652, unbiased), two passes, one CTA
__global__ void __launch_bounds__(1024) rstd_kernel(const StepCommon c) {
    __shared__ float red[32];
    __shared__ float s_mean;
    auto block_sum = [&](float v) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
        __syncthreads();
        float s = 0.0f;
        for (int w = 0; w < 32; ++w) s += red[w];
        return s;
    };
    float s = 0.0f;
    for (int i = threadIdx.x; i < c.B; i += 1024) s += c.rowv[(size_t)i * 4 + 1];
    const float mean = block_sum(s) / (float)c.B;
    if (threadIdx.x == 0) s_mean = mean;
    __syncthreads();
    s = 0.0f;
    for (int i = threadIdx.x; i < c.B; i += 1024) { const float d = c.rowv[(size_t)i * 4 + 1] - s_mean; s = fmaf(d, d, s); }
    const float var = block_sum(s) / (float)(c.B > 1 ? c.B - 1 : 1);
    if (threadIdx.x == 0) *c.inv_cs = 1.0f / (sqrtf(var) + 1e-5f);
}

// Output layers Linear(H -> 1), the objectives and their gradients (agent.py:635-652) for one row tile of one net:
// out = w . a_last + b; d united / d out; dZ_last = d_out * w * act'(a_last) (T-format); output-layer gradients.
struct OutNet {
    const uint8_t *LAST; uint8_t *DZ; int chunks;   // last hidden activation and its pre-activation gradient ([rows][H])
    int w_off, b_off, db_last_off, act, H;          // output layer in theta / grad; bias gradient of the last hidden layer
};
__global__ void __launch_bounds__(256) out_obj_kernel(const StepCommon c, const OutNet na, const OutNet nc) {
    __shared__ float part[32][129];
    __shared__ float dout[128];
    __shared__ float gw[257];
    __shared__ float gb_last[256];
    __shared__ float red4[8][4];
    const int rt = blockIdx.x, net = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
    const OutNet &N = net == 0 ? na : nc;
    const int H = N.H, UG = H / 8;
    const float *w = c.theta + N.w_off;
    for (int j = tid; j < H + 1; j += 256) gw[j] = 0.0f;
    for (int j = tid; j < H; j += 256) gb_last[j] = 0.0f;
    for (int item = tid; item < 128 * UG; item += 256) {
        const int row = item & 127, ug = item >> 7;
        const size_t o = (size_t)((ug & 7) * 128 + row) * 16;
        float a[8];
        join8(*reinterpret_cast<const uint4 *>(N.LAST + tblock(rt, N.chunks, ug >> 3, 0) + o),
              *reinterpret_cast<const uint4 *>(N.LAST + tblock(rt, N.chunks, ug >> 3, 1) + o), a);
        float s = 0.0f;
#pragma unroll
        for (int e = 0; e < 8; ++e) s = fmaf(a[e], __ldg(w + ug * 8 + e), s);
        part[ug][row] = s;
    }
    __syncthreads();
    if (tid < 128) {
        const int row = tid, b = rt * 128 + row;
        const bool live = b < c.B;
        float out = __ldg(c.theta + N.b_off);
        for (int ug = 0; ug < UG; ++ug) out += part[ug][row];
        const float4 rv = reinterpret_cast<const float4 *>(c.rowv)[b];   // action, r_sum, old logprob, advantage
        const ppo::RowObj ob = ppo::row_objectives(net, out, rv.x, rv.y, rv.z, rv.w, __ldg(c.theta + c.n_theta - 1), *c.inv_cs,
                                                   c.ratio_clip, c.lambda_entropy, 1.0f / (float)c.B, live);
        const float d = ob.d_out;
        float o_act = ob.o_act, o_cri = ob.o_cri, o_ent = ob.o_ent, g_asl = ob.g_asl;
        dout[row] = d;
        float db = d;
#pragma unroll
        for (int o2 = 16; o2 > 0; o2 >>= 1) {
            o_act += __shfl_xor_sync(0xffffffffu, o_act, o2); o_cri += __shfl_xor_sync(0xffffffffu, o_cri, o2);
            o_ent += __shfl_xor_sync(0xffffffffu, o_ent, o2); g_asl += __shfl_xor_sync(0xffffffffu, g_asl, o2);
            db += __shfl_xor_sync(0xffffffffu, db, o2);
        }
        if (lane == 0) { red4[tid >> 5][0] = o_act; red4[tid >> 5][1] = o_cri; red4[tid >> 5][2] = o_ent; red4[tid >> 5][3] = g_asl; atomicAdd(&gw[H], db); }
    }
    __syncthreads();
    if (tid == 0) {
        float o_act = 0.f, o_cri = 0.f, o_ent = 0.f, g_asl = 0.f;
        for (int q = 0; q < 4; ++q) { o_act += red4[q][0]; o_cri += red4[q][1]; o_ent += red4[q][2]; g_asl += red4[q][3]; }
        float *row = c.loss_ring + (size_t)(*c.step_dev % c.ring_len) * 4;
        if (net == 0) { atomicAdd(row + 0, o_act); atomicAdd(row + 1, o_act); atomicAdd(row + 3, o_ent); atomicAdd(c.grad + c.n_theta - 1, g_asl); }
        else { atomicAdd(row + 0, o_cri * *c.inv_cs); atomicAdd(row + 2, o_cri); }
    }
    for (int item = tid; item < 128 * UG; item += 256) {
        const int row = item & 127, ug = item >> 7;
        const size_t o = (size_t)((ug & 7) * 128 + row) * 16;
        float a[8], x[8];
        join8(*reinterpret_cast<const uint4 *>(N.LAST + tblock(rt, N.chunks, ug >> 3, 0) + o),
              *reinterpret_cast<const uint4 *>(N.LAST + tblock(rt, N.chunks, ug >> 3, 1) + o), a);
        const float d = dout[row], ds = d * c.dz_scale[net];
#pragma unroll
        for (int e = 0; e < 8; ++e) x[e] = fminf(fmaxf(ds * __ldg(w + ug * 8 + e) * act_grad(N.act, a[e]), -6e4f), 6e4f);
        uint4 hi, lo;
        split8(x, hi, lo);   // (colsum below consumes x)
        *reinterpret_cast<uint4 *>(N.DZ + tblock(rt, N.chunks, ug >> 3, 0) + o) = hi;
        *reinterpret_cast<uint4 *>(N.DZ + tblock(rt, N.chunks, ug >> 3, 1) + o) = lo;
        float s8[8];                    // lanes = 32 consecutive rows of the same unit group: column sums over the rows
#pragma unroll
        for (int e = 0; e < 8; ++e) s8[e] = d * a[e];
        int col;
        const float sw = colsum<8>(s8, lane, col);
        const float sb = colsum<8>(x, lane, col);
        if ((lane & 3) == 0) { atomicAdd(&gw[ug * 8 + col], sw); atomicAdd(&gb_last[ug * 8 + col], sb); }
    }
    __syncthreads();
    const float unscale = 1.0f / c.dz_scale[net];
    for (int j = tid; j < H; j += 256) { atomicAdd(c.grad + N.w_off + j, gw[j]); atomicAdd(c.grad + N.db_last_off + j, gb_last[j] * unscale); }
    if (tid == 0) atomicAdd(c.grad + N.b_off, gw[H]);
}

__global__ void close_step_kernel(int *step_dev, float *loss_ring, int ring_len) { ppo::close_step(step_dev, loss_ring, ring_len); }

// ------------------------------------------------------------------------------------------------ host side: the step's program
// work buffer layout (bytes).  Activation / gradient matrices are [row_tiles * 128][units] in T-format (hi + lo: 4 B per element).
struct Plan {
    Net act, cri;
    int B, row_tiles, H, n_theta;
    size_t X, rowv, inv_cs;
    size_t A[8], Z[8];          // activations / pre-activation gradients of the hidden layers (see build_plan)
    size_t W[8], WT[8];         // T-format weights of the up to 8 matrix layers
    size_t total;
    WSplit ws;
};

static size_t mat_bytes(int row_tiles, int units) { return (size_t)row_tiles * (units / 64) * 2 * kBlk; }

// layer numbering.  modular actor: 0 other_net.0, 1 integrator_net.0, 2 other_net.2, 3 integrator_net.2, 4 net.0;
// plain actor: 0 net.0, 2 net.2, 4 net.4 (1, 3 unused); critic: 5 net.0, 6 net.2, 7 net.4.
// activations: A[0] = other_net.0 (H) / plain net.0, A[1] = integrator_net.0 (H), A[2] = cat (H) / plain net.2, A[4] = net.0 (H) /
// plain net.4, A[5..7] = critic; Z[i] = the pre-activation gradient with the shape of A[i].
static bool build_plan(const pime_actor_config &actor, int B, Plan &pl) {
    const int H = actor.mid_dim, S = actor.state_dim;
    if (!(H == 128 || H == 256) || S > 56) return false;
    if (!(actor.kind == PIME_ACTOR_MODULAR || actor.kind == PIME_ACTOR_PLAIN)) return false;
    if (!ppo::theta_layout(actor, pl.act, pl.cri, pl.n_theta)) return false;
    pl.B = B; pl.H = H; pl.row_tiles = (B + 127) / 128;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += (bytes + 1023) & ~(size_t)1023; return r; };
    pl.X = take(mat_bytes(pl.row_tiles, 64));
    pl.rowv = take((size_t)pl.row_tiles * 128 * 16);
    pl.inv_cs = take(1024);
    const bool mod = actor.kind == PIME_ACTOR_MODULAR;
    for (int i = 0; i < 8; ++i) {
        const bool used = i >= 5 || i == 0 || i == 2 || i == 4 || (mod && i == 1);
        pl.A[i] = used ? take(mat_bytes(pl.row_tiles, H)) : 0;
        pl.Z[i] = used ? take(mat_bytes(pl.row_tiles, H)) : 0;
    }
    // weights
    const int Hh = H / 2;
    pl.ws = WSplit{};
    auto layer = [&](int li, const Net &d, int w, int b, int N, int K, bool first, int k_lo, bool need_t) {
        WLayer &L = pl.ws.l[pl.ws.n++];
        L.w_off = d.theta_off + d.src[w]; L.b_off = d.theta_off + d.src[b]; L.N = N; L.K = K;
        L.first = first ? 1 : 0; L.kpad = first ? 64 : K; L.k_lo = k_lo;
        const int rows_pad = (N + 127) / 128 * 128;
        pl.W[li] = take((size_t)rows_pad * L.kpad * 4);
        L.dst = (long long)pl.W[li];
        pl.WT[li] = need_t ? take((size_t)K * ((N + 63) / 64 * 64) * 4) : 0;
        L.dst_t = need_t ? (long long)pl.WT[li] : -1;
    };
    if (mod) {
        layer(0, pl.act, 0, 1, H, pl.act.So, true, 0, false);                 // other_net.0
        layer(1, pl.act, 4, 5, H, S - pl.act.So, true, pl.act.So, false);     // integrator_net.0
        layer(2, pl.act, 2, 3, Hh, H, false, 0, true);                        // other_net.2
        layer(3, pl.act, 6, 7, Hh, H, false, 0, true);                        // integrator_net.2
        layer(4, pl.act, 8, 9, H, H, false, 0, true);                         // net.0
    } else {
        layer(0, pl.act, 0, 1, H, S, true, 0, false);
        layer(2, pl.act, 2, 3, H, H, false, 0, true);
        layer(4, pl.act, 4, 5, H, H, false, 0, true);
    }
    layer(5, pl.cri, 0, 1, H, S, true, 0, false);
    layer(6, pl.cri, 2, 3, H, H, false, 0, true);
    layer(7, pl.cri, 4, 5, H, H, false, 0, true);
    pl.total = o;
    return true;
}

static GemmProb fwd(uint8_t *w, const Plan &pl, size_t A, int a_chunks, int a_c0, int kc, size_t W, int w_chunks, int N, const float *bias, int act,
                    size_t OUT, int out_c0) {
    GemmProb p{};
    p.A = w + A; p.a_chunks = a_chunks; p.a_c0 = a_c0; p.kc = kc;
    p.W = w + W; p.w_chunks = w_chunks;
    p.n_cols = N >= 128 ? 128 : 64; p.n_tiles = N >= 128 ? N / 128 : 1;
    p.mode = 0; p.act = act; p.bias = bias;
    p.OUT = w + OUT; p.out_chunks = pl.H / 64; p.out_c0 = out_c0;
    return p;
}
static GemmProb bwd(uint8_t *w, const Plan &pl, float unscale, size_t DZ, int dz_c0, int kc, size_t WT, int wt_chunks, int K, int act, size_t APREV,
                    size_t OUT, float *db, float *db2 = nullptr, int db_split = 1 << 30) {
    GemmProb p{};
    p.A = w + DZ; p.a_chunks = pl.H / 64; p.a_c0 = dz_c0; p.kc = kc;
    p.W = w + WT; p.w_chunks = wt_chunks;
    p.n_cols = 128; p.n_tiles = K / 128;
    p.mode = 1; p.act = act;
    p.OUT = w + OUT; p.out_chunks = pl.H / 64; p.out_c0 = 0;
    p.APREV = w + APREV; p.ap_chunks = pl.H / 64; p.ap_c0 = 0;
    p.db = db; p.db2 = db2; p.db_split = db_split; p.db_scale = unscale;
    return p;
}
// dW[out][in] = sum_rows DZ[row][out] * A[row][in]
static WgProb wg(uint8_t *w, const Plan &pl, float unscale, size_t DZ, int dz_c0, int out_n, size_t A, int a_chunks, int in_units, int w_off, int ldw,
                 int in_lo, int in_hi, int bias_col, int b_off) {
    WgProb p{};
    p.scale = unscale;
    const bool swap = out_n < 128;   // 64 output units (H = 128: the H/2-wide layers): they become the MMA's N, the inputs its M
    const uint8_t *dz = w + DZ, *a = w + A;
    if (!swap) {
        p.MOP = dz; p.m_chunks = pl.H / 64; p.m_c0 = dz_c0; p.m_tiles = out_n / 128;
        p.NOP = a; p.n_chunks = a_chunks; p.n_c0 = 0; p.n_cols = in_units >= 128 ? 128 : 64; p.n_tiles = in_units >= 128 ? in_units / 128 : 1;
    } else {
        p.MOP = a; p.m_chunks = a_chunks; p.m_c0 = 0; p.m_tiles = in_units / 128;
        p.NOP = dz; p.n_chunks = pl.H / 64; p.n_c0 = dz_c0; p.n_cols = 64; p.n_tiles = 1;
    }
    p.swap = swap ? 1 : 0;
    p.w_off = w_off; p.ldw = ldw; p.in_lo = in_lo; p.in_hi = in_hi; p.out_n = out_n; p.bias_col = bias_col; p.b_off = b_off;
    return p;
}

template <typename Batch, typename Kern>
static int launch_batch(Kern kern, const Batch &b, dim3 grid, int threads, int smem, cudaStream_t s) {
    PIME_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    kern<<<grid, threads, smem, s>>>(b);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

}  // namespace tcl
}  // namespace pime

using namespace pime;

extern "C" {

int64_t pime_ppo_tc_work_bytes(const pime_actor_config *actor, int32_t batch) {
    tcl::Plan pl;
    if (!actor || batch < 1 || !tcl::build_plan(*actor, batch, pl)) return -1;
    return (int64_t)pl.total;
}

// named buffers of the work area (tests compare the intermediate matrices with torch): out[2 * i] = byte offset, out[2 * i + 1] =
// units, for i = 0: X, 1..8: A[0..7], 9..16: Z[0..7]
int pime_ppo_tc_layout(const pime_actor_config *actor, int32_t batch, int64_t *out34) {
    tcl::Plan pl;
    PIME_REQUIRE(actor && out34 && tcl::build_plan(*actor, batch, pl), "unsupported network dimensions for the tensor-core learner");
    out34[0] = (int64_t)pl.X; out34[1] = 64;
    for (int i = 0; i < 8; ++i) {
        out34[2 + 2 * i] = (int64_t)pl.A[i]; out34[3 + 2 * i] = pl.A[i] || i == 0 ? pl.H : 0;
        out34[18 + 2 * i] = (int64_t)pl.Z[i]; out34[19 + 2 * i] = pl.Z[i] ? pl.H : 0;
    }
    return PIME_OK;
}

int pime_ppo_close_step(const pime_ppo_args *a, void *stream) {
    PIME_REQUIRE(a && a->state && a->loss_ring && a->ring_len >= 2, "null ppo args / state / loss ring");
    if (int rc = require_device()) return rc;
    tcl::close_step_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(ppo::State(a->state).step, a->loss_ring, a->ring_len);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

int pime_ppo_grad_tc(const pime_ppo_args *a, void *work_tc, float *grad, void *stream) {
    using namespace tcl;
    if (int rc = ppo::validate_ppo_args(a)) return rc;
    PIME_REQUIRE(work_tc && grad, "null work_tc / grad");
    Plan pl;
    PIME_REQUIRE(build_plan(*a->actor, a->batch, pl), "the tensor-core learner needs mid_dim 128 or 256 and a plain / modular actor");
    PIME_REQUIRE(((uintptr_t)work_tc & 255) == 0, "work_tc must be 256-byte aligned");
    if (int rc = require_device()) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    uint8_t *w = (uint8_t *)work_tc;
    const int H = pl.H, Hh = H / 2, HC = H / 64, RT = pl.row_tiles;
    const bool mod = a->actor->kind == PIME_ACTOR_MODULAR;
    const float *th = a->theta;

    StepCommon c{};
    c.buf_state = a->buf_state; c.buf_action = a->buf_action; c.buf_r_sum = a->buf_r_sum; c.buf_logprob = a->buf_logprob; c.buf_adv = a->buf_advantage;
    c.idx = a->idx; c.B = a->batch; c.S = a->actor->state_dim; c.row_tiles = RT;
    c.ratio_clip = a->ratio_clip; c.lambda_entropy = a->lambda_entropy; c.lr = a->lr; c.beta1 = a->beta1; c.beta2 = a->beta2;
    const ppo::State st(a->state);
    c.step_dev = st.step; c.adam_c = st.adam_c; c.loss_ring = a->loss_ring; c.ring_len = a->ring_len;
    c.grad = grad; c.n_theta = pl.n_theta; c.rowv = (float *)(w + pl.rowv); c.inv_cs = (float *)(w + pl.inv_cs); c.theta = th;

    float pow2B = 1.0f;
    while (pow2B < (float)a->batch) pow2B *= 2.0f;
    c.dz_scale[0] = pow2B;            // actor: |d out| B is O(advantage * ratio / std)
    c.dz_scale[1] = pow2B * 16.0f;    // critic: |d out| B <= 1 / (std(r_sum) + 1e-5)
    const float un_a = 1.0f / c.dz_scale[0], un_c = 1.0f / c.dz_scale[1];

    const Net &A = pl.act, &C = pl.cri;
    const int actA = ACT_TANH, actC = ACT_RELU;
    PIME_CUDA(cudaMemsetAsync(grad, 0, (size_t)pl.n_theta * sizeof(float), s));
    split_weights_kernel<<<dim3(64, pl.ws.n), 256, 0, s>>>(pl.ws, th, w);
    PIME_LAUNCH_CHECK();
    gather_kernel<<<RT, 128, 0, s>>>(c, w + pl.X);
    PIME_LAUNCH_CHECK();
    rstd_kernel<<<1, 1024, 0, s>>>(c);
    PIME_LAUNCH_CHECK();

    auto B_ = [&](const Net &d, int j) { return th + d.theta_off + d.src[j]; };
    auto run_gemm = [&](GemmBatch &gb) {
        gb.row_tiles = RT;
        int nt = 1;
        for (int i = 0; i < gb.n; ++i) nt = gb.p[i].n_tiles > nt ? gb.p[i].n_tiles : nt;
        return launch_batch(gemm_kk_kernel, gb, dim3(nt, RT, gb.n), kGemmThreads, kGemmSmem, s);
    };
    // ---- forward
    {
        GemmBatch g{};
        if (mod) {
            g.p[g.n++] = fwd(w, pl, pl.X, 1, 0, 1, pl.W[0], 1, H, nullptr, actA, pl.A[0], 0);          // other_net.0 (bias in the ones column)
            g.p[g.n++] = fwd(w, pl, pl.X, 1, 0, 1, pl.W[1], 1, H, nullptr, actA, pl.A[1], 0);          // integrator_net.0
        } else {
            g.p[g.n++] = fwd(w, pl, pl.X, 1, 0, 1, pl.W[0], 1, H, nullptr, actA, pl.A[0], 0);          // net.0
        }
        g.p[g.n++] = fwd(w, pl, pl.X, 1, 0, 1, pl.W[5], 1, H, nullptr, actC, pl.A[5], 0);              // critic net.0
        if (int rc = run_gemm(g)) return rc;
    }
    {
        GemmBatch g{};
        if (mod) {
            g.p[g.n++] = fwd(w, pl, pl.A[0], HC, 0, HC, pl.W[2], HC, Hh, B_(A, 3), actA, pl.A[2], 0);          // other_net.2 -> cat[:, :H/2]
            g.p[g.n++] = fwd(w, pl, pl.A[1], HC, 0, HC, pl.W[3], HC, Hh, B_(A, 7), actA, pl.A[2], Hh / 64);    // integrator_net.2 -> cat[:, H/2:]
        } else {
            g.p[g.n++] = fwd(w, pl, pl.A[0], HC, 0, HC, pl.W[2], HC, H, B_(A, 3), actA, pl.A[2], 0);           // net.2
        }
        g.p[g.n++] = fwd(w, pl, pl.A[5], HC, 0, HC, pl.W[6], HC, H, B_(C, 3), actC, pl.A[6], 0);               // critic net.2
        if (int rc = run_gemm(g)) return rc;
    }
    {
        GemmBatch g{};
        g.p[g.n++] = fwd(w, pl, pl.A[2], HC, 0, HC, pl.W[4], HC, H, B_(A, mod ? 9 : 5), actA, pl.A[4], 0);     // net.0 on cat / plain net.4
        g.p[g.n++] = fwd(w, pl, pl.A[6], HC, 0, HC, pl.W[7], HC, H, B_(C, 5), actC, pl.A[7], 0);               // critic net.4
        if (int rc = run_gemm(g)) return rc;
    }
    // ---- output layers, objectives, their gradients
    {
        OutNet na{}, nc{};
        na.LAST = w + pl.A[4]; na.DZ = w + pl.Z[4]; na.chunks = HC; na.act = actA; na.H = H;
        na.w_off = A.theta_off + A.src[mod ? 10 : 6]; na.b_off = A.theta_off + A.src[mod ? 11 : 7]; na.db_last_off = A.theta_off + A.src[mod ? 9 : 5];
        nc.LAST = w + pl.A[7]; nc.DZ = w + pl.Z[7]; nc.chunks = HC; nc.act = actC; nc.H = H;
        nc.w_off = C.theta_off + C.src[6]; nc.b_off = C.theta_off + C.src[7]; nc.db_last_off = C.theta_off + C.src[5];
        out_obj_kernel<<<dim3(RT, 2), 256, 0, s>>>(c, na, nc);
        PIME_LAUNCH_CHECK();
    }
    // ---- data gradients.  The epilogue that produces a pre-activation gradient also takes its column sums = the bias
    // gradient of that layer (first layers excepted: their bias is a weight column, see the ones column of X).
    {
        GemmBatch g{};
        float *ga = grad + A.theta_off, *gc = grad + C.theta_off;
        if (mod)   // dZ(cat) = (dZ(net.0) W_net.0) * tanh'(cat); its halves are the bias gradients of other_net.2 | integrator_net.2
            g.p[g.n++] = bwd(w, pl, un_a, pl.Z[4], 0, HC, pl.WT[4], HC, H, actA, pl.A[2], pl.Z[2], ga + A.src[3], ga + A.src[7], Hh);
        else       // dZ(net.2) = (dZ(net.4) W_net.4) * tanh'
            g.p[g.n++] = bwd(w, pl, un_a, pl.Z[4], 0, HC, pl.WT[4], HC, H, actA, pl.A[2], pl.Z[2], ga + A.src[3]);
        g.p[g.n++] = bwd(w, pl, un_c, pl.Z[7], 0, HC, pl.WT[7], HC, H, actC, pl.A[6], pl.Z[6], gc + C.src[3]);
        if (int rc = run_gemm(g)) return rc;
    }
    {
        GemmBatch g{};
        if (mod) {
            g.p[g.n++] = bwd(w, pl, un_a, pl.Z[2], 0, Hh / 64, pl.WT[2], Hh / 64, H, actA, pl.A[0], pl.Z[0], nullptr);          // -> dZ(other_net.0)
            g.p[g.n++] = bwd(w, pl, un_a, pl.Z[2], Hh / 64, Hh / 64, pl.WT[3], Hh / 64, H, actA, pl.A[1], pl.Z[1], nullptr);    // -> dZ(integrator_net.0)
        } else {
            g.p[g.n++] = bwd(w, pl, un_a, pl.Z[2], 0, HC, pl.WT[2], HC, H, actA, pl.A[0], pl.Z[0], nullptr);
        }
        g.p[g.n++] = bwd(w, pl, un_c, pl.Z[6], 0, HC, pl.WT[6], HC, H, actC, pl.A[5], pl.Z[5], nullptr);
        if (int rc = run_gemm(g)) return rc;
    }
    // ---- weight gradients: all matrices in one launch
    {
        WgBatch g{};
        g.grad = grad; g.row_tiles = RT;
        auto W_ = [&](const Net &d, int j) { return d.theta_off + d.src[j]; };
        const int S = c.S;
        if (mod) {
            g.p[g.n++] = wg(w, pl, un_a, pl.Z[0], 0, H, pl.X, 1, 64, W_(A, 0), A.So, 0, A.So, kBiasCol, W_(A, 1));                 // other_net.0
            g.p[g.n++] = wg(w, pl, un_a, pl.Z[1], 0, H, pl.X, 1, 64, W_(A, 4), S - A.So, A.So, S, kBiasCol, W_(A, 5));            // integrator_net.0
            g.p[g.n++] = wg(w, pl, un_a, pl.Z[2], 0, Hh, pl.A[0], HC, H, W_(A, 2), H, 0, H, -1, 0);                               // other_net.2
            g.p[g.n++] = wg(w, pl, un_a, pl.Z[2], Hh / 64, Hh, pl.A[1], HC, H, W_(A, 6), H, 0, H, -1, 0);                         // integrator_net.2
            g.p[g.n++] = wg(w, pl, un_a, pl.Z[4], 0, H, pl.A[2], HC, H, W_(A, 8), H, 0, H, -1, 0);                                // net.0
        } else {
            g.p[g.n++] = wg(w, pl, un_a, pl.Z[0], 0, H, pl.X, 1, 64, W_(A, 0), S, 0, S, kBiasCol, W_(A, 1));
            g.p[g.n++] = wg(w, pl, un_a, pl.Z[2], 0, H, pl.A[0], HC, H, W_(A, 2), H, 0, H, -1, 0);
            g.p[g.n++] = wg(w, pl, un_a, pl.Z[4], 0, H, pl.A[2], HC, H, W_(A, 4), H, 0, H, -1, 0);
        }
        g.p[g.n++] = wg(w, pl, un_c, pl.Z[5], 0, H, pl.X, 1, 64, W_(C, 0), S, 0, S, kBiasCol, W_(C, 1));
        g.p[g.n++] = wg(w, pl, un_c, pl.Z[6], 0, H, pl.A[5], HC, H, W_(C, 2), H, 0, H, -1, 0);
        g.p[g.n++] = wg(w, pl, un_c, pl.Z[7], 0, H, pl.A[6], HC, H, W_(C, 4), H, 0, H, -1, 0);
        int mx = 1;
        for (int i = 0; i < g.n; ++i) mx = g.p[i].m_tiles * g.p[i].n_tiles > mx ? g.p[i].m_tiles * g.p[i].n_tiles : mx;
        int split = RT < 32 ? RT : 32;
        if (int rc = launch_batch(wgrad_mn_kernel, g, dim3(mx, split, g.n), kWgThreads, kWgSmem, s)) return rc;
    }
    return PIME_OK;
}

}  // extern "C"
