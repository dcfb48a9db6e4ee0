// learner.cu -- one PPO minibatch step of AgentPPO.update_net (elegantrl/agent.py:635-658) on the GPU-resident replay
// as TWO launches instead of the ~100 small kernels of the autograd step (the reference's batch sizes, 128-512 rows, are
// launch-latency bound):
//
//   ppo_rows_kernel   one CTA per R minibatch rows: gather the rows, actor and critic forward (fp32, activations in
//                     shared memory), the clipped-surrogate / entropy / SmoothL1 objectives and their gradients, the
//                     data-gradient chain through both networks.  Rows are independent, so no grid-wide step exists;
//                     a ninth warp streams the hidden-layer weights from L2 through a cp.async.bulk ring (forward from
//                     the transposed copy, backward from the torch layout, so that thread n / thread k reads its own
//                     column).  Activations and pre-activation gradients go to a scratch buffer.
//   ppo_wgrad_kernel  one CTA per 32 x 64 tile of a weight matrix: dW = dZ^T . A over the minibatch (cp.async double-buffered), bias gradient, and
//                     the Adam update (torch.optim.Adam arithmetic) applied in place to the weights, their transposed
//                     copy and the moments.  Every gradient element is produced by exactly one thread: no atomics.
//
// fp32 throughout (the reference trains in fp32); sums run in a different order than cuBLAS, nothing else differs.
#include "ppo_common.cuh"

namespace pime {
namespace ppo {

constexpr int kThreads = 256;          // compute threads of the rows kernel (one more warp streams the weights)
constexpr int kRowsThreads = kThreads + 32;
constexpr int kSlabRows = 16;          // weight rows per streamed slab
constexpr int kSlabFloats = kSlabRows * 256;
constexpr int kMaxStages = 8;          // slabs in flight (cp.async.bulk ring): 8 (128 KB) up to 4 rows per CTA, 4 at 8 rows
constexpr int kMaxPasses = 12;
constexpr int kMaxLayers = 10;
constexpr int kOutAcc = 272;           // floats per output-layer accumulator (H + 1 <= 257)
static_assert(State::kGOut + 2 * kOutAcc <= 1024, "the two output-layer accumulators must fit in the state block");
constexpr int kXInt = 4;               // modular: aligned copy of the integrator observation inside the gathered row
constexpr int kXStride = 32;      // gathered state row (S <= 32)
constexpr int kRowVals = 8;       // per-row scalars in shared memory
constexpr int kTileN = 32, kTileK = 64;   // weight-gradient tile
constexpr int kBk = 32;           // minibatch rows per shared-memory stage of the weight-gradient kernel
constexpr int kWgStages = 2;

enum { ACT_NONE = 0, ACT_TANH = 1, ACT_RELU = 2 };

struct LayerDesc {
    int net;              // 0 actor, 1 critic
    int N, K;
    int w_off, b_off;     // offsets into theta
    int dz_col;           // column of this layer's dZ in the net's gradient rows; -1: the output gradient DOUT[:, net]
    int in_col;           // column of the layer's input in the net's activation rows; -1: the gathered state X[:, x_col:]
    int x_col;
    int tile0, tn, tk;    // first tile, tiles along N and K
};

struct StreamPass {       // one hidden-layer weight matrix streamed through the shared-memory ring, 16 rows per slab
    int off;              // offset in theta (backward: torch layout [N][K]) or theta_t (forward: [K][N])
    int transposed;       // 1: theta_t
    int net;              // 0 actor, 1 critic
    int rows, cols;
};

struct StepParams {
    Net act, cri;
    int LA[2];                // activation columns per row of the actor and the critic (act_cols)
    int n_layers, n_tiles;
    int n_passes;
    StreamPass pass[kMaxPasses];
    LayerDesc layer[kMaxLayers];
    float *theta, *theta_t, *m, *v, *grad_out;
    int n_theta;              // actor + critic + a_std_log
    const float *buf_state, *buf_action, *buf_r_sum, *buf_logprob, *buf_adv;
    const int64_t *idx;
    int B;
    float ratio_clip, lambda_entropy, lr, beta1, beta2, eps;
    State st;                 // adam_c is written by the rows kernel; g_out holds [2][kOutAcc]: weight[H], bias
    float *X, *ACT_A, *DZ_A, *ACT_C, *DZ_C, *DOUT;
    float *loss_ring;
    int ring_len;
};

__device__ __forceinline__ float act_apply(int act, float x) { return act == ACT_TANH ? tanhf(x) : (act == ACT_RELU ? fmaxf(x, 0.0f) : x); }
__device__ __forceinline__ float act_grad(int act, float a) { return act == ACT_TANH ? 1.0f - a * a : (act == ACT_RELU ? (a > 0.0f ? 1.0f : 0.0f) : 1.0f); }

// out[r][n] = act(b[n] + sum_k in[r][k] Wt[k][n]); thread n, R rows in registers, weights coalesced along n
template <int R>
__device__ __forceinline__ void fwd_layer(const float *in, int in_stride, int K, const float *__restrict__ Wt,
                                          const float *__restrict__ bias, int N, int act, float *out, int out_stride) {
    for (int n = threadIdx.x; n < N; n += kThreads) {
        float acc[R];
        const float b = __ldg(bias + n);
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = b;
        int k = 0;
        for (; k + 8 <= K; k += 8) {
            float w[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) w[j] = __ldg(Wt + (size_t)(k + j) * N + n);
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const float4 a0 = *reinterpret_cast<const float4 *>(in + r * in_stride + k);
                const float4 a1 = *reinterpret_cast<const float4 *>(in + r * in_stride + k + 4);
                acc[r] = fmaf(a0.x, w[0], acc[r]); acc[r] = fmaf(a0.y, w[1], acc[r]);
                acc[r] = fmaf(a0.z, w[2], acc[r]); acc[r] = fmaf(a0.w, w[3], acc[r]);
                acc[r] = fmaf(a1.x, w[4], acc[r]); acc[r] = fmaf(a1.y, w[5], acc[r]);
                acc[r] = fmaf(a1.z, w[6], acc[r]); acc[r] = fmaf(a1.w, w[7], acc[r]);
            }
        }
        for (; k < K; ++k) {
            const float w = __ldg(Wt + (size_t)k * N + n);
#pragma unroll
            for (int r = 0; r < R; ++r) acc[r] = fmaf(in[r * in_stride + k], w, acc[r]);
        }
#pragma unroll
        for (int r = 0; r < R; ++r) out[r * out_stride + n] = act_apply(act, acc[r]);
    }
}

// barrier of the 8 compute warps of the rows kernel (the streaming warp never joins)
__device__ __forceinline__ void sync_compute() { asm volatile("bar.sync 1, %0;" ::"n"(kThreads) : "memory"); }

// The weight ring: warp 8 streams every hidden-layer matrix of the step, slab by slab (cp.async.bulk, kStages in flight,
// so the L2 latency is paid once); the 8 compute warps consume the slabs in the same order.
struct Ring {
    float *buf;
    uint64_t *full, *empty;
    uint32_t st, ph, nst;
    __device__ __forceinline__ const float *acquire() {
        tc::mbar_wait(&full[st], ph);
        return buf + st * kSlabFloats;
    }
    __device__ __forceinline__ void release() {
        __syncwarp();
        if ((threadIdx.x & 31) == 0) tc::mbar_arrive(&empty[st]);
        if (++st == nst) { st = 0; ph ^= 1; }
    }
};

// One streamed matrix [ROWS][COLS] against R operand rows x[r][0..ROWS): part[g][r][c] = sum over the slab rows of group g
// of x[r][row] * W[row][c].  Thread = (4 adjacent columns) x (one of G = 1024 / COLS row groups): a float4 of weights and a
// few operand values per 4*R..16*R FMAs, instead of one shared-memory load per R FMAs with a thread per column.  The
// caller sums the G partials.  COLS in {64, 128, 256}.
template <int R, int COLS>
__device__ __forceinline__ void ring_gemm(Ring &ring, const float *x, int xs, int ROWS, float *part) {
    constexpr int CG = COLS / 4, G = kThreads / CG, RPG = kSlabRows / G;   // 256: G=4, 4 rows per group and slab; 128: 8, 2; 64: 16, 1
    const int cg = threadIdx.x % CG, g = threadIdx.x / CG;
    float acc[R][4];
#pragma unroll
    for (int r = 0; r < R; ++r) acc[r][0] = acc[r][1] = acc[r][2] = acc[r][3] = 0.0f;
    for (int r0 = 0; r0 < ROWS; r0 += kSlabRows) {
        const float *w = ring.acquire() + (g * RPG) * COLS + cg * 4;
        float4 wv[RPG];
#pragma unroll
        for (int i = 0; i < RPG; ++i) wv[i] = *reinterpret_cast<const float4 *>(w + i * COLS);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            float xv[RPG];
            const float *xp = x + r * xs + r0 + g * RPG;
            if constexpr (RPG == 4) { const float4 t = *reinterpret_cast<const float4 *>(xp); xv[0] = t.x; xv[1] = t.y; xv[2] = t.z; xv[3] = t.w; }
            else if constexpr (RPG == 2) { const float2 t = *reinterpret_cast<const float2 *>(xp); xv[0] = t.x; xv[1] = t.y; }
            else xv[0] = xp[0];
#pragma unroll
            for (int i = 0; i < RPG; ++i) {
                acc[r][0] = fmaf(xv[i], wv[i].x, acc[r][0]); acc[r][1] = fmaf(xv[i], wv[i].y, acc[r][1]);
                acc[r][2] = fmaf(xv[i], wv[i].z, acc[r][2]); acc[r][3] = fmaf(xv[i], wv[i].w, acc[r][3]);
            }
        }
        ring.release();
    }
    sync_compute();   // every thread has left the previous layer's reduction, which reads part
#pragma unroll
    for (int r = 0; r < R; ++r)
        *reinterpret_cast<float4 *>(part + (g * R + r) * COLS + cg * 4) = make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]);
    sync_compute();
}
template <int R, int COLS> __device__ __forceinline__ float part_sum(const float *part, int r, int c) {
    constexpr int G = kThreads / (COLS / 4);
    float s = 0.0f;
#pragma unroll
    for (int g = 0; g < G; ++g) s += part[(g * R + r) * COLS + c];
    return s;
}

template <int R> __device__ __forceinline__ void fwd_ring_narrow(Ring &ring, const float *in, int in_stride, int K, const float *__restrict__ bias,
                                                                 int N, int act, float *out, int out_stride);
template <int R> __device__ __forceinline__ void bwd_ring_narrow(Ring &ring, const float *dz_out, int dzo_stride, int N, int K, const float *a_in,
                                                                 int a_stride, int act_in, float *dz_in, int dzi_stride);

// hidden layer forward through the ring: out[r][n] = act(b[n] + sum_k in[r][k] Wt[k][n])
template <int R>
__device__ __forceinline__ void fwd_ring(Ring &ring, const float *in, int in_stride, int K, const float *__restrict__ bias, int N, int act,
                                         float *out, int out_stride, float *part) {
    if (N == 256) ring_gemm<R, 256>(ring, in, in_stride, K, part);
    else if (N == 128) ring_gemm<R, 128>(ring, in, in_stride, K, part);
    else if (N == 64) ring_gemm<R, 64>(ring, in, in_stride, K, part);
    else { fwd_ring_narrow<R>(ring, in, in_stride, K, bias, N, act, out, out_stride); return; }
    const int n = threadIdx.x;
    if (n < N) {
        const float b = __ldg(bias + n);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const float s = N == 256 ? part_sum<R, 256>(part, r, n) : (N == 128 ? part_sum<R, 128>(part, r, n) : part_sum<R, 64>(part, r, n));
            out[r * out_stride + n] = act_apply(act, b + s);
        }
    }
}

// hidden layer backward through the ring: dz_in[r][k] = act'(a_in[r][k]) * sum_n dz_out[r][n] W[n][k]
template <int R>
__device__ __forceinline__ void bwd_ring(Ring &ring, const float *dz_out, int dzo_stride, int N, int K, const float *a_in, int a_stride,
                                         int act_in, float *dz_in, int dzi_stride, float *part) {
    if (K == 256) ring_gemm<R, 256>(ring, dz_out, dzo_stride, N, part);
    else if (K == 128) ring_gemm<R, 128>(ring, dz_out, dzo_stride, N, part);
    else if (K == 64) ring_gemm<R, 64>(ring, dz_out, dzo_stride, N, part);
    else { bwd_ring_narrow<R>(ring, dz_out, dzo_stride, N, K, a_in, a_stride, act_in, dz_in, dzi_stride); return; }
    const int k = threadIdx.x;
    if (k < K) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const float s = K == 256 ? part_sum<R, 256>(part, r, k) : (K == 128 ? part_sum<R, 128>(part, r, k) : part_sum<R, 64>(part, r, k));
            dz_in[r * dzi_stride + k] = s * act_grad(act_in, a_in[r * a_stride + k]);
        }
    }
}

// narrow layers (fewer than 64 columns): a thread per column
template <int R>
__device__ __forceinline__ void fwd_ring_narrow(Ring &ring, const float *in, int in_stride, int K, const float *__restrict__ bias, int N, int act,
                                         float *out, int out_stride) {
    const int n = threadIdx.x;
    const bool on = n < N;
    float acc[R];
    const float b = on ? __ldg(bias + n) : 0.0f;
#pragma unroll
    for (int r = 0; r < R; ++r) acc[r] = b;
    for (int k0 = 0; k0 < K; k0 += kSlabRows) {
        const float *w = ring.acquire();
        if (on) {
#pragma unroll
            for (int kk = 0; kk < kSlabRows; kk += 4) {
                const float w0 = w[(kk + 0) * N + n], w1 = w[(kk + 1) * N + n], w2 = w[(kk + 2) * N + n], w3 = w[(kk + 3) * N + n];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const float4 a = *reinterpret_cast<const float4 *>(in + r * in_stride + k0 + kk);
                    acc[r] = fmaf(a.x, w0, acc[r]); acc[r] = fmaf(a.y, w1, acc[r]);
                    acc[r] = fmaf(a.z, w2, acc[r]); acc[r] = fmaf(a.w, w3, acc[r]);
                }
            }
        }
        ring.release();
    }
    if (on) {
#pragma unroll
        for (int r = 0; r < R; ++r) out[r * out_stride + n] = act_apply(act, acc[r]);
    }
}

// hidden layer backward through the ring: dz_in[r][k] = act'(a_in[r][k]) * sum_n dz_out[r][n] W[n][k], thread k (K == kThreads or less)
template <int R>
__device__ __forceinline__ void bwd_ring_narrow(Ring &ring, const float *dz_out, int dzo_stride, int N, int K, const float *a_in, int a_stride,
                                                int act_in, float *dz_in, int dzi_stride) {
    const int k = threadIdx.x;
    const bool on = k < K;
    float acc[R];
#pragma unroll
    for (int r = 0; r < R; ++r) acc[r] = 0.0f;
    for (int n0 = 0; n0 < N; n0 += kSlabRows) {
        const float *w = ring.acquire();
        if (on) {
#pragma unroll
            for (int nn = 0; nn < kSlabRows; nn += 4) {
                const float w0 = w[(nn + 0) * K + k], w1 = w[(nn + 1) * K + k], w2 = w[(nn + 2) * K + k], w3 = w[(nn + 3) * K + k];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const float4 d = *reinterpret_cast<const float4 *>(dz_out + r * dzo_stride + n0 + nn);
                    acc[r] = fmaf(d.x, w0, acc[r]); acc[r] = fmaf(d.y, w1, acc[r]);
                    acc[r] = fmaf(d.z, w2, acc[r]); acc[r] = fmaf(d.w, w3, acc[r]);
                }
            }
        }
        ring.release();
    }
    if (on) {
#pragma unroll
        for (int r = 0; r < R; ++r) dz_in[r * dzi_stride + k] = acc[r] * act_grad(act_in, a_in[r * a_stride + k]);
    }
}

// Linear(K -> 1): one warp per row
template <int R>
__device__ __forceinline__ void fwd_out(const float *in, int in_stride, int K, const float *__restrict__ w, float b, float *out,
                                        int out_stride) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int r = warp; r < R; r += kThreads / 32) {
        float s = 0.0f;
        for (int k = lane; k < K; k += 32) s = fmaf(in[r * in_stride + k], __ldg(w + k), s);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) out[r * out_stride] = s + b;
    }
}

// backward of Linear(K -> 1): dz_in[r][k] = act'(a_in[r][k]) * d_out[r] * w[k]
template <int R>
__device__ __forceinline__ void bwd_out(const float *d_out, int d_stride, const float *__restrict__ w, int K, const float *a_in,
                                        int a_stride, int act_in, float *dz_in, int dzi_stride) {
    for (int k = threadIdx.x; k < K; k += kThreads) {
        const float wk = __ldg(w + k);
#pragma unroll
        for (int r = 0; r < R; ++r) dz_in[r * dzi_stride + k] = d_out[r * d_stride] * wk * act_grad(act_in, a_in[r * a_stride + k]);
    }
}

__device__ __forceinline__ float block_sum(float v, float *scratch) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    sync_compute();
    if (lane == 0) scratch[warp] = v;
    sync_compute();
    float s = 0.0f;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) s += scratch[w];
    return s;
}

// forward (and its mirror, the data-gradient chain) of one net on R rows held in shared memory.  Compute warps only; the
// hidden layers take their weights from the ring in the order fill_passes() lists them.
template <int R>
__device__ __forceinline__ void net_forward(Ring &ring, const Net &d, const float *__restrict__ th, const float *__restrict__ tt,
                                            const float *sX, float *A, int as, float *out, int out_stride, float *part) {
    const int H = d.H;
    if (d.kind == PIME_ACTOR_MODULAR) {   // net_residual.py:150-170
        const int Hh = H / 2;
        fwd_layer<R>(sX, kXStride, d.So, tt + d.src[0], th + d.src[1], H, ACT_TANH, A, as);                       // other_net.0
        fwd_layer<R>(sX + d.So, kXStride, d.S - d.So, tt + d.src[4], th + d.src[5], H, ACT_TANH, A + H, as);     // integrator_net.0
        sync_compute();
        fwd_ring<R>(ring, A, as, H, th + d.src[3], Hh, ACT_TANH, A + 2 * H, as, part);                                  // other_net.2
        fwd_ring<R>(ring, A + H, as, H, th + d.src[7], Hh, ACT_TANH, A + 2 * H + Hh, as, part);                         // integrator_net.2
        sync_compute();
        fwd_ring<R>(ring, A + 2 * H, as, H, th + d.src[9], H, ACT_TANH, A + 3 * H, as, part);                           // net.0 on cat
        sync_compute();
        fwd_out<R>(A + 3 * H, as, H, th + d.src[10], __ldg(th + d.src[11]), out, out_stride);                     // net.2
    } else {                               // plain actor (tanh) / CriticAdv (relu)
        const int act = d.kind == PIME_CRITIC_ADV ? ACT_RELU : ACT_TANH;
        fwd_layer<R>(sX, kXStride, d.S, tt + d.src[0], th + d.src[1], H, act, A, as);
        sync_compute();
        fwd_ring<R>(ring, A, as, H, th + d.src[3], H, act, A + H, as, part);
        sync_compute();
        fwd_ring<R>(ring, A + H, as, H, th + d.src[5], H, act, A + 2 * H, as, part);
        sync_compute();
        fwd_out<R>(A + 2 * H, as, H, th + d.src[6], __ldg(th + d.src[7]), out, out_stride);
    }
    sync_compute();
}

template <int R>
__device__ __forceinline__ void net_backward(Ring &ring, const Net &d, const float *__restrict__ th, const float *A, float *Z, int as,
                                             const float *d_out, int d_stride, float *part) {
    const int H = d.H;
    if (d.kind == PIME_ACTOR_MODULAR) {
        const int Hh = H / 2;
        bwd_out<R>(d_out, d_stride, th + d.src[10], H, A + 3 * H, as, ACT_TANH, Z + 3 * H, as);                   // -> dZ(net.0)
        sync_compute();
        bwd_ring<R>(ring, Z + 3 * H, as, H, H, A + 2 * H, as, ACT_TANH, Z + 2 * H, as, part);                           // net.0 -> dZ(other_net.2 | integrator_net.2)
        sync_compute();
        bwd_ring<R>(ring, Z + 2 * H, as, Hh, H, A, as, ACT_TANH, Z, as, part);                                          // other_net.2 -> dZ(other_net.0)
        bwd_ring<R>(ring, Z + 2 * H + Hh, as, Hh, H, A + H, as, ACT_TANH, Z + H, as, part);                             // integrator_net.2 -> dZ(integrator_net.0)
    } else {
        const int act = d.kind == PIME_CRITIC_ADV ? ACT_RELU : ACT_TANH;
        bwd_out<R>(d_out, d_stride, th + d.src[6], H, A + 2 * H, as, act, Z + 2 * H, as);
        sync_compute();
        bwd_ring<R>(ring, Z + 2 * H, as, H, H, A + H, as, act, Z + H, as, part);                                        // net.4
        sync_compute();
        bwd_ring<R>(ring, Z + H, as, H, H, A, as, act, Z, as, part);                                                    // net.2
    }
    sync_compute();
}

// grid = (row tiles, 2): blockIdx.y = 0 runs the actor (forward, policy objectives, backward), 1 the critic.  The two
// nets share nothing but the gathered rows (obj_united = obj_actor + obj_critic / (std + 1e-5) is a sum), so splitting
// them halves the chain of dependent layers a CTA walks through.
template <int R>
__global__ void __launch_bounds__(kRowsThreads, 1) ppo_rows_kernel(const StepParams p) {
    extern __shared__ __align__(128) float sm[];
    const int net = blockIdx.y;
    const Net &d = net == 0 ? p.act : p.cri;
    const int LA = p.LA[net];
    Ring ring;
    constexpr int kStages = R <= 4 ? kMaxStages : 4;
    ring.buf = sm;                          // [kStages][kSlabFloats]
    ring.full = reinterpret_cast<uint64_t *>(sm + kStages * kSlabFloats);
    ring.empty = ring.full + kStages;
    ring.st = 0; ring.ph = 0; ring.nst = kStages;
    if (threadIdx.x == 0) {
        for (int j = 0; j < kStages; ++j) { tc::mbar_init(&ring.full[j], 1); tc::mbar_init(&ring.empty[j], kThreads / 32); }
        tc::fence_barrier_init();
    }
    __syncthreads();
    if (threadIdx.x >= kThreads) {          // warp 8: streams every hidden-layer matrix of this net through the ring
        if (threadIdx.x == kThreads) {
            uint32_t st = 0, ph = 0;
            for (int q = 0; q < p.n_passes; ++q) {
                const StreamPass P = p.pass[q];
                if (P.net != net) continue;
                const float *src = (P.transposed ? p.theta_t : p.theta) + P.off;
                const uint32_t bytes = (uint32_t)(kSlabRows * P.cols * sizeof(float));
                for (int r0 = 0; r0 < P.rows; r0 += kSlabRows) {
                    tc::mbar_wait(&ring.empty[st], ph ^ 1);
                    tc::mbar_arrive_expect_tx(&ring.full[st], bytes);
                    tc::bulk_g2s(ring.buf + st * kSlabFloats, src + (size_t)r0 * P.cols, bytes, &ring.full[st]);
                    if (++st == kStages) { st = 0; ph ^= 1; }
                }
            }
        }
        return;
    }
    float *sX = reinterpret_cast<float *>(ring.empty + kStages);   // [R][kXStride]
    float *sA = sX + R * kXStride;          // [R][LA] activations of this net
    float *sZ = sA + R * LA;                // [R][LA] pre-activation gradients
    float *sV = sZ + R * LA;                // [R][kRowVals]: action, r_sum, logprob_old, advantage, net output, -, d output, -
    float *sRed = sV + R * kRowVals;        // [8]
    float *sPart = sRed + 8;                // 1024 R floats: partial sums of ring_gemm
    const int tid = threadIdx.x;
    const int B = p.B;
    const int b0 = blockIdx.x * R;

    if (blockIdx.x == 0 && net == 0 && tid == 0) adam_prepare(p.st.step, p.lr, p.beta1, p.beta2, p.st.adam_c);
    float inv_cs = 0.0f;
    if (net == 1) {   // r_sum.std() of the minibatch (agent.py:652; unbiased), two passes
        float s = 0.0f;
        for (int i = tid; i < B; i += kThreads) s += __ldg(p.buf_r_sum + __ldg(p.idx + i));
        const float mean = block_sum(s, sRed) / (float)B;
        s = 0.0f;
        for (int i = tid; i < B; i += kThreads) {
            const float dlt = __ldg(p.buf_r_sum + __ldg(p.idx + i)) - mean;
            s = fmaf(dlt, dlt, s);
        }
        const float rstd = sqrtf(block_sum(s, sRed) / (float)(B > 1 ? B - 1 : 1));
        inv_cs = 1.0f / (rstd + 1e-5f);
    }

    // gather
    for (int j = tid; j < R * kXStride; j += kThreads) {
        const int r = j / kXStride, c = j % kXStride, b = b0 + r;
        float x = 0.0f;
        if (b < B && c < p.act.S) x = __ldg(p.buf_state + __ldg(p.idx + b) * p.act.S + c);
        else if (b < B && p.act.kind == PIME_ACTOR_MODULAR && c >= kXInt && c - kXInt < p.act.S - p.act.So)   // 16-byte aligned copy
            x = __ldg(p.buf_state + __ldg(p.idx + b) * p.act.S + p.act.So + (c - kXInt));                      // for the weight-gradient kernel
        sX[j] = x;
    }
    if (tid < R) {
        const int b = b0 + tid;
        const bool live = b < B;
        const int64_t i = live ? __ldg(p.idx + b) : 0;
        sV[tid * kRowVals + 0] = live ? __ldg(p.buf_action + i) : 0.0f;
        sV[tid * kRowVals + 1] = live ? __ldg(p.buf_r_sum + i) : 0.0f;
        sV[tid * kRowVals + 2] = live ? __ldg(p.buf_logprob + i) : 0.0f;
        sV[tid * kRowVals + 3] = live ? __ldg(p.buf_adv + i) : 0.0f;
    }
    sync_compute();

    const float *th = p.theta + d.theta_off, *tt = p.theta_t + d.theta_off;
    net_forward<R>(ring, d, th, tt, sX, sA, LA, sV + 4, kRowVals, sPart);

    // objectives and their gradients (agent.py:635-652), one thread per row
    if (tid < R) {
        float *rv = sV + tid * kRowVals;
        const bool live = b0 + tid < B;
        const RowObj ob = row_objectives(net, rv[4], rv[0], rv[1], rv[2], rv[3], __ldg(p.theta + p.n_theta - 1), inv_cs,
                                         p.ratio_clip, p.lambda_entropy, 1.0f / (float)B, live);
        rv[6] = ob.d_out;
        float o_act = ob.o_act, o_cri = ob.o_cri, o_ent = ob.o_ent, g_asl = ob.g_asl;
#pragma unroll
        for (int o = 1; o < R; o <<= 1) {   // R is a power of two <= 32, the rows sit in one warp
            o_act += __shfl_xor_sync((1u << R) - 1u, o_act, o);
            o_cri += __shfl_xor_sync((1u << R) - 1u, o_cri, o);
            o_ent += __shfl_xor_sync((1u << R) - 1u, o_ent, o);
            g_asl += __shfl_xor_sync((1u << R) - 1u, g_asl, o);
        }
        if (tid == 0) {
            float *row = p.loss_ring + (size_t)(*p.st.step % p.ring_len) * 4;
            atomicAdd(row + 0, o_act + o_cri * inv_cs);
            if (net == 0) { atomicAdd(row + 1, o_act); atomicAdd(row + 3, o_ent); atomicAdd(p.st.g_astd, g_asl); }
            else atomicAdd(row + 2, o_cri);
        }
    }
    sync_compute();

    net_backward<R>(ring, d, th, sA, sZ, LA, sV + 6, kRowVals, sPart);

    // output layer Linear(H -> 1): weight / bias gradients of this CTA's rows, straight into the accumulators
    for (int k = tid; k < d.H + 1; k += kThreads) {
        const float *Alast = sA + (d.kind == PIME_ACTOR_MODULAR ? 3 : 2) * d.H;
        float g = 0.0f;
#pragma unroll
        for (int r = 0; r < R; ++r) g = fmaf(sV[r * kRowVals + 6], k < d.H ? Alast[r * LA + k] : 1.0f, g);
        atomicAdd(p.st.g_out + net * kOutAcc + k, g);
    }

    // rows -> scratch (inputs of the weight-gradient kernel)
    float *ACT = net == 0 ? p.ACT_A : p.ACT_C, *DZ = net == 0 ? p.DZ_A : p.DZ_C;
    for (int r = 0; r < R; ++r) {
        const int b = b0 + r;
        if (b >= B) break;
        for (int c = tid; c < LA; c += kThreads) {
            ACT[(size_t)b * LA + c] = sA[r * LA + c];
            DZ[(size_t)b * LA + c] = sZ[r * LA + c];
        }
        if (net == 0 && tid < kXStride) p.X[(size_t)b * kXStride + tid] = sX[r * kXStride + tid];
        if (tid == 0) p.DOUT[(size_t)b * 2 + net] = sV[r * kRowVals + 6];
    }
}

__device__ __forceinline__ void cp_async16(void *dst_smem, const void *src, bool valid) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst_smem);
    const int bytes = valid ? 16 : 0;   // 0: the 16 bytes are zero-filled, nothing is read
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async4(void *dst_smem, const void *src, bool valid) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst_smem);
    const int bytes = valid ? 4 : 0;
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(d), "l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__global__ void __launch_bounds__(kThreads) ppo_wgrad_kernel(const StepParams p) {
    __shared__ __align__(16) float sD[kWgStages][kBk][kTileN + 4];   // dZ[b][n0 + .], kWgStages stages in flight
    __shared__ __align__(16) float sI[kWgStages][kBk][kTileK + 4];   // input[b][k0 + .]
    __shared__ bool is_last;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;   // tx: 4 columns of k, ty: 2 rows of n
    int li = 0;
    while (li + 1 < p.n_layers && (int)blockIdx.x >= p.layer[li + 1].tile0) ++li;
    const LayerDesc L = p.layer[li];
    const int t_in = blockIdx.x - L.tile0;
    const int n0 = (t_in / L.tk) * kTileN, k0 = (t_in % L.tk) * kTileK;
    const int B = p.B;
    const float *dz; int dz_stride;
    if (L.dz_col < 0) { dz = p.DOUT + L.net; dz_stride = 2; }
    else if (L.net == 0) { dz = p.DZ_A + L.dz_col; dz_stride = p.LA[0]; }
    else { dz = p.DZ_C + L.dz_col; dz_stride = p.LA[1]; }
    const float *in; int in_stride, in_avail;   // in_avail: readable columns of an input row (the products beyond K are dropped)
    if (L.in_col < 0) { in = p.X + L.x_col; in_stride = kXStride; in_avail = kXStride - L.x_col; }
    else if (L.net == 0) { in = p.ACT_A + L.in_col; in_stride = p.LA[0]; in_avail = L.K; }
    else { in = p.ACT_C + L.in_col; in_stride = p.LA[1]; in_avail = L.K; }
    // 16-byte cp.async needs aligned rows: true for every hidden layer; the output layers (dZ = DOUT, stride 2) and the
    // integrator branch's first layer (input column So of X) take the scalar path -- they are a handful of tiny tiles
    const bool fast = L.dz_col >= 0 && (L.in_col >= 0 || (L.x_col & 3) == 0);

    auto fill = [&](int stage, int bb) {
        if (fast) {
            {
                const int r = tid >> 3, c = (tid & 7) * 4, b = bb + r;
                const bool ok = b < B && n0 + c < L.N;
                cp_async16(&sD[stage][r][c], ok ? dz + (size_t)b * dz_stride + n0 + c : dz, ok);
            }
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int j = tid + h * kThreads, r = j >> 4, c = (j & 15) * 4, b = bb + r;
                const bool ok = b < B && k0 + c + 4 <= in_avail;
                cp_async16(&sI[stage][r][c], ok ? in + (size_t)b * in_stride + k0 + c : in, ok);
            }
        } else {   // element-wise asynchronous copies (only the columns that exist are touched; the rest is zero-filled)
            for (int j = tid; j < kBk * kTileN; j += kThreads) {
                const int r = j / kTileN, c = j % kTileN, b = bb + r;
                const bool ok = b < B && n0 + c < L.N;
                cp_async4(&sD[stage][r][c], ok ? dz + (size_t)b * dz_stride + n0 + c : dz, ok);
            }
            for (int j = tid; j < kBk * kTileK; j += kThreads) {
                const int r = j / kTileK, c = j % kTileK, b = bb + r;
                const bool ok = b < B && k0 + c < L.K;
                cp_async4(&sI[stage][r][c], ok ? in + (size_t)b * in_stride + k0 + c : in, ok);
            }
        }
        cp_async_commit();
    };

    float acc[2][4], accb[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        accb[i] = 0.0f;
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
    }
    const int nst = (B + kBk - 1) / kBk;
    for (int j = 0; j < kWgStages - 1; ++j) {   // one commit group per stage, empty groups past the end keep the count uniform
        if (j < nst) fill(j, j * kBk); else cp_async_commit();
    }
    for (int it = 0; it < nst; ++it) {
        const int cur = it % kWgStages;
        if (it + kWgStages - 1 < nst) fill((it + kWgStages - 1) % kWgStages, (it + kWgStages - 1) * kBk); else cp_async_commit();
        cp_async_wait<kWgStages - 1>();
        __syncthreads();
#pragma unroll 8
        for (int r = 0; r < kBk; ++r) {
            const float2 d = *reinterpret_cast<const float2 *>(&sD[cur][r][ty * 2]);
            const float4 a = *reinterpret_cast<const float4 *>(&sI[cur][r][tx * 4]);
            const float dv[2] = {d.x, d.y}, av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                accb[i] += dv[i];
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(dv[i], av[j], acc[i][j]);
            }
        }
        __syncthreads();
    }

    const AdamCoef c = adam_coef(p.st.adam_c, p.beta1, p.beta2, p.eps);
    auto apply = [&](int idx, int idx_t, float g) {
        if (p.grad_out) { p.grad_out[idx] = g; return; }
        float m = p.m[idx], v = p.v[idx];
        const float th = adam_update(c, g, p.theta[idx], m, v);
        p.m[idx] = m; p.v[idx] = v; p.theta[idx] = th; p.theta_t[idx_t] = th;
    };
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const int n = n0 + ty * 2 + i;
        if (n >= L.N) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0 + tx * 4 + j;
            if (k < L.K) apply(L.w_off + n * L.K + k, L.w_off + k * L.N + n, acc[i][j]);
        }
        if (k0 == 0 && tx == 0) apply(L.b_off + n, L.b_off + n, accb[i]);
    }

    // the last CTA to finish closes the step: a_std_log, step counter, the next ring row, the accumulators
    __threadfence();
    __syncthreads();
    if (tid == 0) is_last = atomicAdd(p.st.ticket, 1u) == (unsigned)p.n_tiles - 1u;
    __syncthreads();
    if (is_last) {
        __threadfence();
        for (int j = tid; j < 2 * (p.act.H + 1); j += kThreads) {   // the output layers, accumulated by the rows kernel
            const int net = j / (p.act.H + 1), k = j % (p.act.H + 1);
            const Net &d = net == 0 ? p.act : p.cri;
            const int wi = d.kind == PIME_ACTOR_MODULAR ? 10 : 6;
            const int idx = d.theta_off + (k < d.H ? d.src[wi] + k : d.src[wi + 1]);
            float *acc_p = p.st.g_out + net * kOutAcc + k;
            apply(idx, idx, *reinterpret_cast<volatile float *>(acc_p));
            *acc_p = 0.0f;
        }
        if (tid == 0) {
            const float g = *reinterpret_cast<volatile float *>(p.st.g_astd);
            apply(p.n_theta - 1, p.n_theta - 1, g);
            *p.st.g_astd = 0.0f;
            *p.st.ticket = 0u;
            close_step(p.st.step, p.loss_ring, p.ring_len);
        }
    }
}


// Adam on a flat gradient in theta's layout (the distributed path: pime_ppo_step(grad_out) -> all-reduce -> this).  One
// thread per parameter of every layer (grid.y = layer); the transposed copy is kept in step.  adam_c was written by the
// rows kernel of the same step (adam_prepare), so the bias corrections belong to the step whose gradient this is.
__global__ void __launch_bounds__(kThreads) ppo_adam_kernel(const StepParams p, const float *__restrict__ grad, float scale) {
    const LayerDesc L = p.layer[blockIdx.y];
    const AdamCoef c = adam_coef(p.st.adam_c, p.beta1, p.beta2, p.eps);
    const int nw = L.N * L.K, total = nw + L.N;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < total; j += gridDim.x * blockDim.x) {
        int idx, idx_t;
        if (j < nw) { const int n = j / L.K, k = j % L.K; idx = L.w_off + j; idx_t = L.w_off + k * L.N + n; }
        else { idx = idx_t = L.b_off + (j - nw); }
        float m = p.m[idx], v = p.v[idx];
        const float th = adam_update(c, grad[idx] * scale, p.theta[idx], m, v);
        p.m[idx] = m; p.v[idx] = v; p.theta[idx] = th; p.theta_t[idx_t] = th;
    }
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) {   // a_std_log
        const int idx = p.n_theta - 1;
        float m = p.m[idx], v = p.v[idx];
        const float th = adam_update(c, grad[idx] * scale, p.theta[idx], m, v);
        p.m[idx] = m; p.v[idx] = v; p.theta[idx] = th; p.theta_t[idx] = th;
    }
}

__global__ void ppo_transpose_kernel(StepParams p) {
    for (int li = 0; li < p.n_layers; ++li) {
        const LayerDesc L = p.layer[li];
        for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < L.N * L.K; j += gridDim.x * blockDim.x) {
            const int n = j / L.K, k = j % L.K;
            p.theta_t[L.w_off + k * L.N + n] = p.theta[L.w_off + j];
        }
        for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < L.N; j += gridDim.x * blockDim.x) p.theta_t[L.b_off + j] = p.theta[L.b_off + j];
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) p.theta_t[p.n_theta - 1] = p.theta[p.n_theta - 1];
}

// ------------------------------------------------------------------------------------------------ host side
static void add_layer(StepParams &p, int net, const Net &d, int N, int K, int w, int b, int dz_col, int in_col, int x_col) {
    LayerDesc &L = p.layer[p.n_layers++];
    L.net = net; L.N = N; L.K = K; L.w_off = d.theta_off + d.src[w]; L.b_off = d.theta_off + d.src[b];
    L.dz_col = dz_col; L.in_col = in_col; L.x_col = x_col;
    L.tn = N == 1 ? 0 : (N + kTileN - 1) / kTileN; L.tk = (K + kTileK - 1) / kTileK;   // Linear(H -> 1): see g_out
    L.tile0 = p.n_tiles;
    p.n_tiles += L.tn * L.tk;
}

static void add_net_layers(StepParams &p, int net, const Net &d) {
    const int H = d.H;
    if (d.kind == PIME_ACTOR_MODULAR) {
        add_layer(p, net, d, H, d.So, 0, 1, 0, -1, 0);                      // other_net.0
        add_layer(p, net, d, H / 2, H, 2, 3, 2 * H, 0, 0);                  // other_net.2
        add_layer(p, net, d, H, d.S - d.So, 4, 5, H, -1, kXInt);            // integrator_net.0 (aligned copy of its input)
        add_layer(p, net, d, H / 2, H, 6, 7, 2 * H + H / 2, H, 0);          // integrator_net.2
        add_layer(p, net, d, H, H, 8, 9, 3 * H, 2 * H, 0);                  // net.0
        add_layer(p, net, d, 1, H, 10, 11, -1, 3 * H, 0);                   // net.2
    } else {
        add_layer(p, net, d, H, d.S, 0, 1, 0, -1, 0);
        add_layer(p, net, d, H, H, 2, 3, H, 0, 0);
        add_layer(p, net, d, H, H, 4, 5, 2 * H, H, 0);
        add_layer(p, net, d, 1, H, 6, 7, -1, 2 * H, 0);
    }
}

static void add_pass(StepParams &p, const Net &d, int src, bool transposed, int rows, int cols) {
    StreamPass &q = p.pass[p.n_passes++];
    q.net = &d == &p.cri ? 1 : 0;
    q.off = d.theta_off + d.src[src]; q.transposed = transposed ? 1 : 0; q.rows = rows; q.cols = cols;
}
// the order in which net_forward / net_backward consume the ring
static void fill_passes(StepParams &p) {
    for (int dir = 0; dir < 2; ++dir)
        for (const Net *d : {&p.act, &p.cri}) {
            const int H = d->H, Hh = H / 2;
            if (d->kind == PIME_ACTOR_MODULAR) {
                if (dir == 0) { add_pass(p, *d, 2, true, H, Hh); add_pass(p, *d, 6, true, H, Hh); add_pass(p, *d, 8, true, H, H); }
                else { add_pass(p, *d, 8, false, H, H); add_pass(p, *d, 2, false, Hh, H); add_pass(p, *d, 6, false, Hh, H); }
            } else {
                if (dir == 0) { add_pass(p, *d, 2, true, H, H); add_pass(p, *d, 4, true, H, H); }
                else { add_pass(p, *d, 4, false, H, H); add_pass(p, *d, 2, false, H, H); }
            }
        }
}

// activation columns per row of a net in shared memory and in the scratch rows
static int act_cols(const Net &d) { return d.kind == PIME_ACTOR_MODULAR ? 4 * d.H : 3 * d.H; }

static int fill_params(const pime_ppo_args *a, StepParams &p) {
    PIME_REQUIRE(a && a->actor, "null ppo args / actor config");
    PIME_REQUIRE(a->actor->kind == PIME_ACTOR_PLAIN || a->actor->kind == PIME_ACTOR_MODULAR, "actor kind");
    p = StepParams{};
    PIME_REQUIRE(theta_layout(*a->actor, p.act, p.cri, p.n_theta), "unsupported network dimensions");
    p.LA[0] = act_cols(p.act); p.LA[1] = act_cols(p.cri);
    add_net_layers(p, 0, p.act);
    add_net_layers(p, 1, p.cri);
    fill_passes(p);
    p.theta = a->theta; p.theta_t = a->theta_t; p.m = a->adam_m; p.v = a->adam_v; p.grad_out = a->grad_out;
    return PIME_OK;
}

static int64_t work_floats_per_row(const StepParams &p) { return kXStride + 2 * (int64_t)(p.LA[0] + p.LA[1]) + 2; }

template <int R> static int launch_rows(const StepParams &p, cudaStream_t s) {
    constexpr int kStages = R <= 4 ? kMaxStages : 4;
    const int LAmax = p.LA[0] > p.LA[1] ? p.LA[0] : p.LA[1];
    const size_t smem = sizeof(float) * (size_t)(kStages * kSlabFloats + R * (kXStride + 2 * LAmax + kRowVals) + 8 + 1024 * R) +
                        2 * kStages * sizeof(uint64_t);
    auto kern = ppo_rows_kernel<R>;
    PIME_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<dim3((p.B + R - 1) / R, 2), kRowsThreads, smem, s>>>(p);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

}  // namespace ppo
}  // namespace pime

using namespace pime;

extern "C" {

int64_t pime_ppo_theta_count(const pime_actor_config *actor) {
    int64_t lay[3];
    return pime_ppo_theta_layout(actor, lay) == PIME_OK ? lay[2] : -1;
}

int pime_ppo_theta_layout(const pime_actor_config *actor, int64_t *out) {
    PIME_REQUIRE(actor && out, "null pointer");
    ppo::Net act, cri;
    int n_theta;
    PIME_REQUIRE(ppo::theta_layout(*actor, act, cri, n_theta), "unsupported network dimensions");
    out[0] = cri.theta_off;
    out[1] = n_theta - 1;
    out[2] = n_theta;
    return PIME_OK;
}

int64_t pime_ppo_work_floats(const pime_actor_config *actor, int32_t batch) {
    ppo::StepParams p;
    pime_ppo_args a{};
    a.actor = actor;
    if (!actor || ppo::fill_params(&a, p) != PIME_OK) return -1;
    return ppo::work_floats_per_row(p) * (int64_t)batch;
}

int pime_ppo_transpose(const pime_actor_config *actor, const float *theta, float *theta_t, void *stream) {
    PIME_REQUIRE(actor && theta && theta_t, "null pointer");
    ppo::StepParams p;
    pime_ppo_args a{};
    a.actor = actor; a.theta = const_cast<float *>(theta); a.theta_t = theta_t;
    if (int rc = ppo::fill_params(&a, p)) return rc;
    if (int rc = require_device()) return rc;
    ppo::ppo_transpose_kernel<<<kNumSMs, 256, 0, (cudaStream_t)stream>>>(p);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

int pime_ppo_apply_grad(const pime_ppo_args *a, const float *grad, float scale, void *stream) {
    ppo::StepParams p;
    if (int rc = ppo::fill_params(a, p)) return rc;
    PIME_REQUIRE(a->theta && a->theta_t && a->adam_m && a->adam_v && a->state && grad, "null theta / theta_t / moments / state / grad");
    if (int rc = require_device()) return rc;
    p.lr = a->lr; p.beta1 = a->beta1; p.beta2 = a->beta2; p.eps = a->eps;
    p.st = ppo::State(a->state);
    ppo::ppo_adam_kernel<<<dim3(32, p.n_layers), ppo::kThreads, 0, (cudaStream_t)stream>>>(p, grad, scale);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

int pime_ppo_step(const pime_ppo_args *a, void *stream) {
    if (int rc = ppo::validate_ppo_args(a)) return rc;
    ppo::StepParams p;
    if (int rc = ppo::fill_params(a, p)) return rc;
    PIME_REQUIRE(a->theta_t && a->work, "null theta_t / work");
    PIME_REQUIRE(a->grad_out || (a->adam_m && a->adam_v), "Adam moments are required unless grad_out is given");
    if (int rc = require_device()) return rc;
    p.buf_state = a->buf_state; p.buf_action = a->buf_action; p.buf_r_sum = a->buf_r_sum; p.buf_logprob = a->buf_logprob;
    p.buf_adv = a->buf_advantage; p.idx = a->idx; p.B = a->batch;
    p.ratio_clip = a->ratio_clip; p.lambda_entropy = a->lambda_entropy;
    p.lr = a->lr; p.beta1 = a->beta1; p.beta2 = a->beta2; p.eps = a->eps;
    p.st = ppo::State(a->state);
    p.loss_ring = a->loss_ring; p.ring_len = a->ring_len;
    const int64_t B = a->batch;
    float *w = a->work;
    p.X = w; w += B * ppo::kXStride;
    p.ACT_A = w; w += B * p.LA[0];
    p.DZ_A = w; w += B * p.LA[0];
    p.ACT_C = w; w += B * p.LA[1];
    p.DZ_C = w; w += B * p.LA[1];
    p.DOUT = w;
    cudaStream_t s = (cudaStream_t)stream;
    const int R = B <= 128 ? 2 : (B <= 256 ? 4 : 8);   // at most 128 CTAs (64 per net) up to 512 rows: one wave
    int rc = R == 2 ? ppo::launch_rows<2>(p, s) : (R == 4 ? ppo::launch_rows<4>(p, s) : ppo::launch_rows<8>(p, s));
    if (rc) return rc;
    ppo::ppo_wgrad_kernel<<<p.n_tiles, ppo::kThreads, 0, s>>>(p);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

}  // extern "C"
