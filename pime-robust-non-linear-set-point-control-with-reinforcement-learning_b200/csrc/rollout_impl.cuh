// rollout_impl.cuh -- the fused kernel: T steps of plant + prior + float32 observation + residual actor for 128 envs
// per CTA, state in registers for the whole launch.  Replaces the per-step Python loop of
// AgentResidualPPO.explore_env (elegantrl/agent_residual.py:52-69) and get_episode_return (elegantrl/run.py:600-619).
#pragma once

#include "plants.cuh"
#include "mlp_fp32.cuh"
#include "tc_mlp.cuh"

namespace pime {

constexpr int kMaxS = 32;

struct RolloutParams {
    int64_t n;
    int64_t ld;             // row length of the per-step buffers (>= n)
    int T, deterministic, auto_reset, has_actor, keep_params;
    float a_std;            // exp(a_std_log)
    double reward_scale, gamma;
    uint64_t seed, env_offset;
    uint32_t tick0;
    int S;
    double priorK[kMaxS];
    float priorKf[kMaxS];   // float(priorK): the f32 path multiplies in fp32, as obs32 @ priorK does (agent_residual.py:61)
    float reward_scale_f, gamma_f;
    int reward_scale_exact;  // reward_scale is a float: float(double(rew) * reward_scale) == rew * float(reward_scale)
    const float *eps;
    const void *pn1, *pn2;
    float *buf_state, *buf_other;
    void *env_action;
    double *stats;
    int32_t *status;
};

// ------------------------------------------------------------------------------------------------ plant glue
// STACK selects the observation-history variant (NonLinearWaterTank...Stacking): the last num_stack frames of
// (h1, h2, r) live in registers (every loop below is unrolled to the maximum, 10 frames, and predicated), which keeps
// them out of local memory; the goal / integrator variant carries no history at all.
constexpr int kMaxFrames = 30;

template <typename T, bool STACK> struct WtGlue {
    using Real = T;
    static constexpr int kObsMax = STACK ? kMaxFrames : 4;   // widest observation of this plant (loop bounds)
    static constexpr bool kSegmented = false;
    WtConst<T> c;
    WtPtrs<T> p;

    struct Env {
        WtEnv<T> e;
        T ret;
        uint32_t episode;
        T fr[STACK ? kMaxFrames : 1];  // obs history, oldest first
    };

    __device__ __forceinline__ void load(Env &v, int64_t i, int64_t n) const {
        p.load(v.e, i, c.obs_mode == PIME_WT_OBS_INTEGRATOR);
        v.ret = p.ep_return ? p.ep_return[i] : (T)0;
        v.episode = p.episode[i];
        if constexpr (STACK) {
            const int m = 3 * c.num_stack;
#pragma unroll
            for (int j = 0; j < kMaxFrames; ++j) v.fr[j] = j < m ? p.frames[(int64_t)j * n + i] : (T)0;
        }
    }
    __device__ __forceinline__ void store(const Env &v, int64_t i, int64_t n) const {
        p.store(v.e, i, c.obs_mode == PIME_WT_OBS_INTEGRATOR);
        if (p.ep_return) p.ep_return[i] = v.ret;
        p.episode[i] = v.episode;
        if constexpr (STACK) {
            const int m = 3 * c.num_stack;
#pragma unroll
            for (int j = 0; j < kMaxFrames; ++j)
                if (j < m) p.frames[(int64_t)j * n + i] = v.fr[j];
        }
    }
    // float32(obs): elegantrl/env.py:46,72.  obs[] is indexed with compile-time indices only (registers).
    __device__ __forceinline__ void observe(const Env &v, float (&obs)[kMaxS]) const {
        if constexpr (STACK) {
#pragma unroll
            for (int j = 0; j < kMaxFrames; ++j) obs[j] = (float)v.fr[j];
        } else {
            obs[0] = (float)v.e.h1; obs[1] = (float)v.e.h2; obs[2] = (float)v.e.r;
            obs[3] = c.obs_mode == PIME_WT_OBS_INTEGRATOR ? (float)v.e.I : 0.0f;
        }
    }
    __device__ __forceinline__ bool uses_process_noise() const { return c.noise_scale > (T)0; }
    __device__ __forceinline__ T noise_sigma() const { return c.noise_scale; }
    __device__ __forceinline__ bool advance(Env &v, T action, T nz1, T nz2, T &rew, bool &done) const {
        wt_advance(c, v.e, action, nz1, nz2, rew, done);
        if constexpr (STACK) {  // frames.append(state) (nonlinear_watertank.py:1145-1146)
            const int m = 3 * c.num_stack;
#pragma unroll
            for (int j = 0; j < kMaxFrames - 3; ++j) v.fr[j] = j < m - 3 ? v.fr[j + 3] : v.fr[j];
#pragma unroll
            for (int j = 0; j < kMaxFrames; j += 3)
                if (j == m - 3) { v.fr[j] = v.e.h1; v.fr[j + 1] = v.e.h2; v.fr[j + 2] = v.e.r; }
        }
        return true;
    }
    __device__ __forceinline__ T tracking_error(const Env &v) const { return Num<T>::abs(v.e.r - v.e.h2); }
    // `done` bookkeeping of reset_from_last_state (:819-821)
    __device__ __forceinline__ void record_done(const Env &v, int64_t i) const {
        if (p.last_h1) { p.last_h1[i] = v.e.h1; p.last_h2[i] = v.e.h2; }
    }
    // the in-kernel reset always follows a `done`, so "the levels of the last finished episode" are the current ones
    __device__ __forceinline__ bool reset(Env &v, uint64_t seed, uint64_t index, bool resample) const {
        double u[6];
        reset_uniforms(seed, index, v.episode, u);
        const T k1 = v.e.h1, k2 = v.e.h2;
        wt_reset(c, v.e, u, resample);
        if (c.from_last) { v.e.h1 = k1; v.e.h2 = k2; }
        v.episode += 1;
        fill_frames(v);
        return true;
    }
    // every frame = the current state (nonlinear_watertank.py:1183-1184)
    __device__ __forceinline__ void fill_frames(Env &v) const {
        if constexpr (STACK) {
            const int m = 3 * c.num_stack;
#pragma unroll
            for (int j = 0; j < kMaxFrames; j += 3)
                if (j < m) { v.fr[j] = v.e.h1; v.fr[j + 1] = v.e.h2; v.fr[j + 2] = v.e.r; }
        }
    }

    // Segment begin of a scheduled launch: reset() exactly as wt_reset_kernel (step.cu) computes it, then set_state() of
    // the levels before it and set_r(r) (utils/test.py:102-106).  set_state / set_r leave the frame history alone, so
    // the segment's first observations still show the frames of the reset.
    __device__ __forceinline__ bool restart(Env &v, T r, uint64_t seed, uint64_t index, int64_t i, bool resample) const {
        const T h1 = v.e.h1, h2 = v.e.h2;
        double u[6];
        reset_uniforms(seed, index, v.episode, u);
        wt_reset(c, v.e, u, resample);
        if (c.from_last) wt_reset_levels_from_last(v.e, u, p.last_h1[i], p.last_h2[i]);
        v.episode += 1;
        fill_frames(v);
        v.e.h1 = h1; v.e.h2 = h2; v.e.r = r;
        return true;
    }
    // the controlled output (the level tracking_error compares with r)
    __device__ __forceinline__ T output(const Env &v) const { return v.e.h2; }
    // what the reset writes and store() does not: I = 0 when the observation does not carry the integrator
    __device__ __forceinline__ void store_reset_extra(int64_t i) const {
        if (c.obs_mode != PIME_WT_OBS_INTEGRATOR && p.I) p.I[i] = (T)0;
    }
};

template <typename T> struct PhGlue {
    using Real = T;
    static constexpr int kObsMax = 3;
    static constexpr bool kSegmented = false;
    PhConst<T> c;
    const T *table;
    PhPtrs<T> p;

    struct Env {
        PhEnv<T> e;
        T qww, qc, ret;
        uint32_t episode;
    };
    __device__ __forceinline__ void load(Env &v, int64_t i, int64_t) const {
        p.load(v.e, i, c.integrator_mode != PIME_PH_NO_INTEGRATOR, true);
        v.qww = p.qww[i]; v.qc = p.qc[i];
        v.ret = p.ep_return ? p.ep_return[i] : (T)0;
        v.episode = p.episode[i];
    }
    __device__ __forceinline__ void store(const Env &v, int64_t i, int64_t) const {
        p.store(v.e, i, c.integrator_mode != PIME_PH_NO_INTEGRATOR);
        p.qww[i] = v.qww; p.qc[i] = v.qc;
        if (p.ep_return) p.ep_return[i] = v.ret;
        p.episode[i] = v.episode;
    }
    __device__ __forceinline__ void observe(const Env &v, float (&obs)[kMaxS]) const {
        obs[0] = (float)v.e.y; obs[1] = (float)v.e.r;
        obs[2] = c.integrator_mode != PIME_PH_NO_INTEGRATOR ? (float)v.e.I : 0.0f;
    }
    __device__ __forceinline__ bool uses_process_noise() const { return false; }
    __device__ __forceinline__ T noise_sigma() const { return (T)0; }
    __device__ __forceinline__ bool advance(Env &v, T action, T, T, T &rew, bool &done) const {
        return ph_advance(c, table, v.e, action, rew, done);
    }
    __device__ __forceinline__ T tracking_error(const Env &v) const { return Num<T>::abs(v.e.r - v.e.y); }
    __device__ __forceinline__ void record_done(const Env &v, int64_t i) const {   // ph.py:345-346
        if (p.last_x) p.last_x[i] = v.e.x;
    }
    __device__ __forceinline__ bool reset(Env &v, uint64_t seed, uint64_t index, bool resample) const {
        double u[6];
        reset_uniforms(seed, index, v.episode, u);
        bool ok = ph_reset(c, table, v.e, v.qww, v.qc, u, resample, c.from_last ? v.e.x : nan_of<double>());
        v.episode += 1;
        return ok;
    }
    // Segment begin of a scheduled launch: reset() exactly as ph_reset_kernel (step.cu) computes it, then the state x
    // before it restored with its observation y under the new C, and r set (utils/test.py:1386-1388).
    __device__ __forceinline__ bool restart(Env &v, T r, uint64_t seed, uint64_t index, int64_t i, bool resample) const {
        const double x = v.e.x;
        double u[6];
        reset_uniforms(seed, index, v.episode, u);
        bool ok = ph_reset(c, table, v.e, v.qww, v.qc, u, resample, c.from_last ? p.last_x[i] : nan_of<double>());
        v.episode += 1;
        v.e.x = x;
        ok = ph_lookup(table, c.table_len, (double)v.e.C, x, v.e.y) && ok;   // observe_state (ph.py:187-189)
        v.e.r = r;
        return ok;
    }
    __device__ __forceinline__ T output(const Env &v) const { return v.e.y; }
    __device__ __forceinline__ void store_reset_extra(int64_t i) const {
        if (c.integrator_mode == PIME_PH_NO_INTEGRATOR && p.I) p.I[i] = (T)0;
    }
};

// ------------------------------------------------------------------------------------------------ scheduled launch
// T = K L steps in K segments of L steps (pime_schedule); segment k tracks set-point r[k].  Segmented<Glue> is the plant
// glue of such a launch: Stepper restarts each env at every segment begin and keeps its tracking metrics in registers.
// Every plain glue has kSegmented = false, for which none of this generates code.
struct SegParams {
    int K, L, resample;
    double r[PIME_MAX_SEGMENTS];
    double *metrics;   // [4][K][n] (ret, iae, final_err, overshoot), or NULL
};

template <typename Glue> struct Segmented : Glue {
    static constexpr bool kSegmented = true;
    SegParams sg;
    struct Env : Glue::Env {
        double m_ret, m_iae, m_err, m_ovs;   // this segment's sum of rewards, sum of |e|, last |e|, overshoot
        bool up;                             // r >= y at the segment begin: the overshoot is y - r, else r - y
    };
    __device__ __forceinline__ void store(const Env &v, int64_t i, int64_t n) const {
        Glue::store(v, i, n);
        Glue::store_reset_extra(i);
    }
};

template <typename T> __device__ __forceinline__ T prior_k(const RolloutParams &rp, int k);
template <> __device__ __forceinline__ float prior_k<float>(const RolloutParams &rp, int k) { return rp.priorKf[k]; }
template <> __device__ __forceinline__ double prior_k<double>(const RolloutParams &rp, int k) { return rp.priorK[k]; }

// ------------------------------------------------------------------------------------------------ one env step
// Everything of one step that follows the actor forward, for the env owned by the calling thread:
// noise, action = tanh(a_raw) + obs32 . priorK, plant step, replay row, statistics, auto-reset.
template <typename Plant> struct Stepper {
    using T = typename Plant::Real;
    using N = Num<T>;
    double s_ret = 0.0, s_ret2 = 0.0, s_cnt = 0.0, s_err = 0.0, s_rew = 0.0, s_steps = 0.0;
    bool fault = false;

    // The part of a step that does not depend on the network output: exploration / process noise (Philox + Box-Muller, or
    // the injected arrays) and the prior term obs32 . priorK.  The fused kernel runs it BEFORE it waits for net(obs), i.e.
    // in the time the owner would otherwise spend on the barrier -- ~500 cycles off the owners' critical path per step.
    float p_eps = 0.0f, p_prior_f = 0.0f;
    T p_nz1 = (T)0, p_nz2 = (T)0, p_prior = (T)0;
    __device__ __forceinline__ void prepare(const Plant &plant, const RolloutParams &rp, const float (&obs)[kMaxS], int s, int64_t ii) {
        const int S = rp.S;
        float eps = 0.0f, z0 = 0.0f, z1 = 0.0f;
        const int64_t q = (int64_t)s * rp.ld + ii;
        const bool need_eps = !rp.deterministic && rp.eps == nullptr;
        const bool need_pn = plant.uses_process_noise() && rp.pn1 == nullptr;
        if (need_eps || need_pn) {
            const Philox4 w = philox4x32_10(rp.seed, rp.env_offset + (uint64_t)ii, rp.tick0 + (uint32_t)s, kStreamStep);
            if (need_pn) box_muller(w.v[0], w.v[1], z0, z1);
            if (need_eps) { float e1; box_muller(w.v[2], w.v[3], eps, e1); }
        }
        if (!rp.deterministic && rp.eps) eps = rp.eps[q];
        T nz1 = (T)0, nz2 = (T)0;
        if (plant.uses_process_noise()) {
            if (rp.pn1) { nz1 = ((const T *)rp.pn1)[q]; nz2 = ((const T *)rp.pn2)[q]; }
            else { nz1 = (T)z0 * plant.noise_sigma(); nz2 = (T)z1 * plant.noise_sigma(); }
        } else if (rp.pn1) { nz1 = ((const T *)rp.pn1)[q]; nz2 = ((const T *)rp.pn2)[q]; }
        p_eps = eps; p_nz1 = nz1; p_nz2 = nz2;
        // ---- prior term of action = tanh(a_raw) + obs32 . priorK   (agent_residual.py:61 / net_residual.py:167-170)
        if (rp.deterministic) {
            float prior = 0.0f;
#pragma unroll
            for (int k = 0; k < Plant::kObsMax; ++k)
                if (k < S) prior = fmaf(obs[k], rp.priorKf[k], prior);
            p_prior_f = prior;
        } else {
            T prior = (T)0;
#pragma unroll
            for (int k = 0; k < Plant::kObsMax; ++k)
                if (k < S) prior = N::add(prior, N::mul((T)obs[k], prior_k<T>(rp, k)));
            p_prior = prior;
        }
    }

    __device__ __forceinline__ void step(const Plant &plant, const RolloutParams &rp, typename Plant::Env &env,
                                         const float (&obs)[kMaxS], float a_avg, int s, int64_t ii, bool live) {
        prepare(plant, rp, obs, s, ii);
        finish(plant, rp, env, obs, a_avg, s, ii, live);
    }

    // the rest of the step, after prepare(): action, plant step, replay row, statistics, auto-reset
    __device__ __forceinline__ void finish(const Plant &plant, const RolloutParams &rp, typename Plant::Env &env,
                                           const float (&obs)[kMaxS], float a_avg, int s, int64_t ii, bool live) {
        const int S = rp.S;
        const int64_t q = (int64_t)s * rp.ld + ii;
        const float eps = p_eps;
        const T nz1 = p_nz1, nz2 = p_nz2;
        float a_raw;
        T action;
        if (rp.deterministic) {
            a_raw = a_avg;
            action = (T)(tanhf(a_avg) + p_prior_f);
        } else {
            a_raw = a_avg + eps * rp.a_std;   // net_residual.py:176-180
            action = N::add((T)tanhf(a_raw), p_prior);
        }
        // ---- plant step
        T rew;
        bool done;
        if (!plant.advance(env, action, nz1, nz2, rew, done)) fault = true;
        env.ret += rew;
        if (live) {
            if (rp.buf_state) {  // replay row (agent_residual.py:64-65; replay.py:278-291), time-major
                float *bs = rp.buf_state + q * S;
                if (S == 4) {
                    *reinterpret_cast<float4 *>(bs) = make_float4(obs[0], obs[1], obs[2], obs[3]);
                } else if ((S & 1) == 0) {   // rows of an even number of floats are 8-byte aligned
#pragma unroll
                    for (int k = 0; k + 1 < Plant::kObsMax; k += 2)
                        if (k < S) *reinterpret_cast<float2 *>(bs + k) = make_float2(obs[k], obs[k + 1]);
                } else {
#pragma unroll
                    for (int k = 0; k < Plant::kObsMax; ++k)
                        if (k < S) bs[k] = obs[k];
                }
                const float rs = (sizeof(T) == 4 && rp.reward_scale_exact) ? (float)rew * rp.reward_scale_f
                                                                           : (float)((double)rew * rp.reward_scale);
                *reinterpret_cast<float4 *>(rp.buf_other + q * 4) = make_float4(rs, done ? 0.0f : rp.gamma_f, a_raw, eps);
            }
            if (rp.env_action) ((T *)rp.env_action)[q] = action;
            s_rew += (double)rew;
            s_steps += 1.0;
            if (done) {
                plant.record_done(env, ii);
                s_ret += (double)env.ret;
                s_ret2 += (double)env.ret * (double)env.ret;
                s_cnt += 1.0;
                s_err += (double)plant.tracking_error(env);
            }
        }
        if (done && rp.auto_reset) {  // env.reset() -> reset_all(): new ensemble member (T4 in SURVEY.md), or reset_r()
            if (!plant.reset(env, rp.seed, rp.env_offset + (uint64_t)ii, rp.keep_params == 0)) fault = true;
            env.ret = (T)0;
        }
        if constexpr (Plant::kSegmented) track(plant, rp, env, rew, s, ii, live);
    }

    // Segment k begins for the env: reset + restore + set-point (the glue's restart), metrics cleared.  The kernels call
    // it for k = 0 right after an env is loaded; track() calls it for the later segments.  No code for a plain launch.
    __device__ __forceinline__ void begin_segment(const Plant &plant, const RolloutParams &rp, typename Plant::Env &env, int k,
                                                  int64_t ii) {
        if constexpr (Plant::kSegmented) {
            const T r = (T)plant.sg.r[k];
            if (!plant.restart(env, r, rp.seed, rp.env_offset + (uint64_t)ii, ii, plant.sg.resample != 0)) fault = true;
            env.ret = (T)0;
            env.m_ret = env.m_iae = env.m_err = env.m_ovs = 0.0;
            env.up = r >= plant.output(env);
        }
    }

    // after step s: the metrics of the step; at a segment end, their store (live envs only) and the next segment's begin
    __device__ __forceinline__ void track(const Plant &plant, const RolloutParams &rp, typename Plant::Env &env, T rew, int s,
                                          int64_t ii, bool live) {
        const double y = (double)plant.output(env), r = (double)env.e.r;
        env.m_ret += (double)rew;
        env.m_err = fabs(r - y);
        env.m_iae += env.m_err;
        env.m_ovs = fmax(env.m_ovs, env.up ? y - r : r - y);
        const int k = (s + 1) / plant.sg.L;
        if (k * plant.sg.L != s + 1) return;
        if (live && plant.sg.metrics) {   // metrics[m][k - 1][ii]
            const int64_t stride = (int64_t)plant.sg.K * rp.n;
            double *m = plant.sg.metrics + (int64_t)(k - 1) * rp.n + ii;
            m[0] = env.m_ret; m[stride] = env.m_iae; m[2 * stride] = env.m_err; m[3 * stride] = env.m_ovs;
        }
        if (s + 1 < rp.T) begin_segment(plant, rp, env, k, ii);
    }

    // warp-shuffle reduction of the episode / set-point statistics; lane 0 of each calling warp adds to red[][slot]
    __device__ __forceinline__ void reduce_warp(double (*red)[4], int slot) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s_ret += __shfl_xor_sync(0xffffffffu, s_ret, o);
            s_ret2 += __shfl_xor_sync(0xffffffffu, s_ret2, o);
            s_cnt += __shfl_xor_sync(0xffffffffu, s_cnt, o);
            s_err += __shfl_xor_sync(0xffffffffu, s_err, o);
            s_rew += __shfl_xor_sync(0xffffffffu, s_rew, o);
            s_steps += __shfl_xor_sync(0xffffffffu, s_steps, o);
        }
        if ((threadIdx.x & 31) == 0) {
            red[0][slot] = s_ret; red[1][slot] = s_ret2; red[2][slot] = s_cnt;
            red[3][slot] = s_err; red[4][slot] = s_rew; red[5][slot] = s_steps;
        }
    }
};

// ------------------------------------------------------------------------------------------------ the kernels
// Fused rollout with an actor: 256 envs per tile (two groups of 128), see tc_mlp.cuh for the roles.  PERSISTENT: one CTA
// per SM walks over the tiles blockIdx.x, blockIdx.x + gridDim.x, ... as ONE continuous sequence of network passes -- TMEM
// allocation, barrier initialisation, the fp32 layer tables, the fill / drain of the software pipeline and the statistics
// tail are paid once per SM instead of once per tile (the pH sweep of BASELINE configs[3] is 32 768 tiles of only 50 steps).
// At a tile boundary the owner stores its env, loads the env of the next tile and writes that observation as the next pass's
// input, so the workers / MMA / TMA roles never notice the boundary.
template <typename Plant, int KIND, int H>
__global__ void __launch_bounds__(tc::kThreads, 1) rollout_kernel(Plant plant, tc::MlpParams mp, RolloutParams rp, int n_tiles) {
    extern __shared__ __align__(1024) uint8_t smem[];
    tc::Engine<KIND, H> eng;
    eng.setup(smem, mp);
    double (*red)[4] = eng.red();
    const int tid = threadIdx.x, warp = tid >> 5;
    const int my_tiles = (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int passes = 2 * rp.T * my_tiles;
    bool fault = false;

    if (warp < 8) {
        eng.worker_loop(passes);
    } else if (warp < 12) {
        const int row = tid - tc::kWorkerThreads;
        const int64_t n = rp.n;
        Stepper<Plant> sp;
        float obs[kMaxS];
        typename Plant::Env env0, env1;
        int64_t i0 = (int64_t)blockIdx.x * tc::kTileEnvs + row, i1 = i0 + tc::kRows;
        bool live0 = i0 < n, live1 = i1 < n;
        int64_t ii0 = live0 ? i0 : n - 1, ii1 = live1 ? i1 : n - 1;  // tail rows shadow the last env and write nothing
        plant.load(env0, ii0, n);
        plant.load(env1, ii1, n);
        sp.begin_segment(plant, rp, env0, 0, ii0);
        sp.begin_segment(plant, rp, env1, 0, ii1);
        plant.observe(env0, obs);
        eng.write_obs(row, 0, obs);
        plant.observe(env1, obs);
        eng.write_obs(row, 1, obs);
#ifdef PIME_PROFILE_OWNER
        long long c_wait = 0, c_work = 0, c0 = clock64();
#define PIME_TICK(acc) { const long long c1 = clock64(); acc += c1 - c0; c0 = c1; }
#else
#define PIME_TICK(acc)
#endif
        int q = 0;   // running pass index of this CTA (group g of step s of tile k: q = 2 (k T + s) + g)
        for (int k = 0; k < my_tiles; ++k) {
            const bool next_tile = k + 1 < my_tiles;
            const int64_t j0 = i0 + (int64_t)gridDim.x * tc::kTileEnvs, j1 = j0 + tc::kRows;   // this row's envs in the next tile
            for (int s = 0; s < rp.T; ++s) {
                const bool more = s + 1 < rp.T;
                {   // group 0: the workers run group 1's pass while this thread steps the plant
                    plant.observe(env0, obs);
                    sp.prepare(plant, rp, obs, s, ii0);                    // noise + prior: before the wait for net(obs)
                    PIME_TICK(c_work)
                    const float a_avg = eng.read_out(row, q++);
                    PIME_TICK(c_wait)
                    sp.finish(plant, rp, env0, obs, a_avg, s, ii0, live0);
                    if (!more && next_tile) {
                        if (live0) plant.store(env0, i0, n);
                        i0 = j0; live0 = i0 < n; ii0 = live0 ? i0 : n - 1;
                        plant.load(env0, ii0, n);
                        sp.begin_segment(plant, rp, env0, 0, ii0);
                    }
                    if (more || next_tile) { plant.observe(env0, obs); eng.write_obs(row, 0, obs); }
                    PIME_TICK(c_work)
                }
                {
                    plant.observe(env1, obs);
                    sp.prepare(plant, rp, obs, s, ii1);
                    PIME_TICK(c_work)
                    const float a_avg = eng.read_out(row, q++);
                    PIME_TICK(c_wait)
                    sp.finish(plant, rp, env1, obs, a_avg, s, ii1, live1);
                    if (!more && next_tile) {
                        if (live1) plant.store(env1, i1, n);
                        i1 = j1; live1 = i1 < n; ii1 = live1 ? i1 : n - 1;
                        plant.load(env1, ii1, n);
                        sp.begin_segment(plant, rp, env1, 0, ii1);
                    }
                    if (more || next_tile) { plant.observe(env1, obs); eng.write_obs(row, 1, obs); }
                    PIME_TICK(c_work)
                }
            }
        }
#ifdef PIME_PROFILE_OWNER
        if (blockIdx.x == 0 && row == 0 && rp.stats) { rp.stats[6] = (double)c_wait; rp.stats[7] = (double)c_work; }
#endif
        if (live0) plant.store(env0, i0, n);
        if (live1) plant.store(env1, i1, n);
        fault = sp.fault;
        if (rp.stats) sp.reduce_warp(red, warp - 8);
    } else if (warp == tc::kMmaWarp) {
        eng.mma_loop(passes);
    } else if ((tid & 31) == 0) {
        eng.producer_loop(passes);
    }

    eng.teardown();  // __syncthreads inside: red[][] is complete
    if (rp.stats && tid < 6) atomicAdd(rp.stats + tid, red[tid][0] + red[tid][1] + red[tid][2] + red[tid][3]);
    if (fault && rp.status) atomicMin(rp.status, (int32_t)PIME_ERANGE);
}

// Fidelity mode of the fused rollout (actor.precision = PIME_PRECISION_FP32): the same Stepper, the network in fp32 on the
// CUDA cores (mlp_fp32.cuh).  32 envs per CTA: threads 0..31 own one env each, all 256 threads evaluate the layers.
template <typename Plant>
__global__ void __launch_bounds__(f32::kFThreads) rollout_fp32_kernel(Plant plant, const __grid_constant__ tc::PackLayout L,
                                                                      const float *__restrict__ params, RolloutParams rp) {
    extern __shared__ __align__(16) float sm32[];
    __shared__ double red[6][4];
    float *tA = sm32, *tB = tA + f32::kTile, *sObs = tB + f32::kTile, *sOut = sObs + 32 * f32::kRS;
    const int tid = threadIdx.x;
    const bool owner = tid < f32::kFR;
    const int64_t n = rp.n;
    const int64_t i = (int64_t)blockIdx.x * f32::kFR + (owner ? tid : 0);
    const bool live = owner && i < n;
    const int64_t ii = i < n ? i : n - 1;
    typename Plant::Env env;
    if (owner) plant.load(env, ii, n);
    Stepper<Plant> sp;
    if (owner) sp.begin_segment(plant, rp, env, 0, ii);
    float obs[kMaxS];
    if (tid < 24) red[tid / 4][tid % 4] = 0.0;
    for (int s = 0; s < rp.T; ++s) {
        if (owner) {
            plant.observe(env, obs);
#pragma unroll
            for (int k = 0; k < Plant::kObsMax; ++k)
                if (k < rp.S) sObs[k * f32::kRS + tid] = obs[k];
        }
        __syncthreads();
        f32::forward(L, params, sObs, tA, tB, sOut);
        if (owner) sp.step(plant, rp, env, obs, sOut[tid], s, ii, live);
    }
    if (live) plant.store(env, i, n);
    if (rp.stats && owner) sp.reduce_warp(red, 0);
    __syncthreads();
    if (rp.stats && tid < 6) atomicAdd(rp.stats + tid, red[tid][0]);
    if (owner && sp.fault && rp.status) atomicMin(rp.status, (int32_t)PIME_ERANGE);
}

template <typename Plant>
int launch_rollout_fp32(const Plant &plant, const tc::PackLayout &L, const void *pack, const RolloutParams &rp, cudaStream_t stream) {
    auto kern = rollout_fp32_kernel<Plant>;
    PIME_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, f32::kSmemBytes));
    const int64_t grid = (rp.n + f32::kFR - 1) / f32::kFR;
    PIME_REQUIRE(grid <= 0x7fffffffLL, "too many envs for one launch");
    kern<<<(unsigned)grid, f32::kFThreads, f32::kSmemBytes, stream>>>(plant, L, reinterpret_cast<const float *>((const uint8_t *)pack + L.f32_off), rp);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

// Prior-only policy (no actor): one thread per env, nothing but the plant and the prior.
template <typename Plant>
__global__ void __launch_bounds__(128) rollout_prior_kernel(Plant plant, RolloutParams rp) {
    __shared__ double red[6][4];
    const int tid = threadIdx.x, warp = tid >> 5;
    const int64_t n = rp.n;
    const int64_t i = (int64_t)blockIdx.x * 128 + tid;
    const bool live = i < n;
    const int64_t ii = live ? i : n - 1;
    typename Plant::Env env;
    plant.load(env, ii, n);
    Stepper<Plant> sp;
    sp.begin_segment(plant, rp, env, 0, ii);
    float obs[kMaxS];
    for (int s = 0; s < rp.T; ++s) {
        plant.observe(env, obs);
        sp.step(plant, rp, env, obs, 0.0f, s, ii, live);
    }
    if (live) plant.store(env, i, n);
    if (rp.stats) sp.reduce_warp(red, warp);
    __syncthreads();
    if (rp.stats && tid < 6) atomicAdd(rp.stats + tid, red[tid][0] + red[tid][1] + red[tid][2] + red[tid][3]);
    if (sp.fault && rp.status) atomicMin(rp.status, (int32_t)PIME_ERANGE);
}

// ------------------------------------------------------------------------------------------------ launchers
template <typename Plant> int launch_rollout_prior(const Plant &plant, const RolloutParams &rp, cudaStream_t stream) {
    const int64_t grid = (rp.n + 127) / 128;
    PIME_REQUIRE(grid <= 0x7fffffffLL, "too many envs for one launch");
    rollout_prior_kernel<Plant><<<(unsigned)grid, 128, 0, stream>>>(plant, rp);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

template <typename Plant, int KIND, int H>
int launch_rollout_kh(const Plant &plant, const tc::PackLayout *L, const void *pack, const RolloutParams &rp, cudaStream_t stream) {
    using G = tc::Geo<KIND, H>;
    auto kern = rollout_kernel<Plant, KIND, H>;
    PIME_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, G::SmemBytes));
    const tc::MlpParams mp = tc::make_mlp_params(*L, pack);
    const int64_t tiles = (rp.n + tc::kTileEnvs - 1) / tc::kTileEnvs;
    const int sms = device_sm_count();
    const int64_t grid = tiles < sms ? tiles : sms;   // one persistent CTA per SM (227 KB of shared memory each)
    PIME_REQUIRE(tiles <= 0x7fffffffLL && 2 * (int64_t)rp.T * ((tiles + grid - 1) / grid) <= 0x7fffffffLL,
                 "too many env steps for one launch");
    kern<<<(unsigned)grid, tc::kThreads, G::SmemBytes, stream>>>(plant, mp, rp, (int)tiles);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

template <typename Plant, int KIND>
int launch_rollout_k(const Plant &plant, const tc::PackLayout *L, const void *pack, const RolloutParams &rp, int H,
                     cudaStream_t stream) {
    switch (H) {
        case 32: return launch_rollout_kh<Plant, KIND, 32>(plant, L, pack, rp, stream);
        case 64: return launch_rollout_kh<Plant, KIND, 64>(plant, L, pack, rp, stream);
        case 128: return launch_rollout_kh<Plant, KIND, 128>(plant, L, pack, rp, stream);
        case 256: return launch_rollout_kh<Plant, KIND, 256>(plant, L, pack, rp, stream);
    }
    set_error("mid_dim must be 32, 64, 128 or 256");
    return PIME_EINVAL;
}

// The kernel for the actor of `a`: the prior kernel without one, the fidelity kernel in fp32 precision, else the tcgen05
// kernel of its kind.  MODULAR = false for a plant without a modular instantiation (the caller has rejected that actor).
template <typename Plant, bool MODULAR>
int launch_rollout_actor(const Plant &plant, const RolloutParams &rp, const tc::PackLayout &L, const pime_rollout_args *a,
                         cudaStream_t stream) {
    if (!rp.has_actor) return launch_rollout_prior<Plant>(plant, rp, stream);
    if (a->actor->precision == PIME_PRECISION_FP32) return launch_rollout_fp32<Plant>(plant, L, a->actor_pack, rp, stream);
    if constexpr (MODULAR) {
        if (a->actor->kind == PIME_ACTOR_MODULAR)
            return launch_rollout_k<Plant, PIME_ACTOR_MODULAR>(plant, &L, a->actor_pack, rp, L.H, stream);
    }
    return launch_rollout_k<Plant, PIME_ACTOR_PLAIN>(plant, &L, a->actor_pack, rp, L.H, stream);
}

// the plain launch of glue g, or the scheduled one (Segmented<Glue>) when sg is given
template <bool MODULAR, typename Glue>
int launch_rollout_glue(const Glue &g, const SegParams *sg, const RolloutParams &rp, const tc::PackLayout &L,
                        const pime_rollout_args *a, cudaStream_t stream) {
    if (sg) return launch_rollout_actor<Segmented<Glue>, MODULAR>(Segmented<Glue>{g, *sg}, rp, L, a, stream);
    return launch_rollout_actor<Glue, MODULAR>(g, rp, L, a, stream);
}

// Checks a schedule against the argument block and fills SegParams (host arithmetic only).
inline int fill_seg_params(const pime_schedule *sc, const pime_rollout_args *a, SegParams &sg) {
    PIME_REQUIRE(sc && a, "null schedule / rollout args");
    PIME_REQUIRE(sc->num_segments >= 1 && sc->num_segments <= PIME_MAX_SEGMENTS, "num_segments must be in 1..16");
    PIME_REQUIRE(sc->segment_steps >= 1, "segment_steps must be >= 1");
    PIME_REQUIRE((int64_t)sc->num_segments * sc->segment_steps == (int64_t)a->T, "args->T must equal num_segments * segment_steps");
    PIME_REQUIRE(sc->setpoints_host, "setpoints_host is NULL");
    PIME_REQUIRE(a->auto_reset == 0, "a scheduled rollout resets at segment begins only: auto_reset must be 0");
    sg = SegParams{};
    sg.K = sc->num_segments; sg.L = sc->segment_steps; sg.resample = sc->resample_params != 0;
    for (int k = 0; k < sg.K; ++k) sg.r[k] = sc->setpoints_host[k];
    sg.metrics = sc->metrics;
    return PIME_OK;
}

// Fills RolloutParams from the public argument block; returns the pack layout in L when an actor is given.
inline int fill_rollout_params(const pime_rollout_args *a, int64_t n, int S, RolloutParams &rp, tc::PackLayout &L) {
    PIME_REQUIRE(a, "null rollout args");
    PIME_REQUIRE(a->T >= 1, "T must be >= 1");
    PIME_REQUIRE(a->priorK_host, "priorK_host is required (pass zeros for no prior)");
    PIME_REQUIRE(S >= 1 && S <= kMaxS, "observation dim");
    PIME_REQUIRE((a->buf_state == nullptr) == (a->buf_other == nullptr), "buf_state/buf_other must both be given or both NULL");
    PIME_REQUIRE((a->pnoise1 == nullptr) == (a->pnoise2 == nullptr), "pnoise1/pnoise2 must both be given or both NULL");
    rp = RolloutParams{};
    PIME_REQUIRE(a->ld == 0 || a->ld >= n, "ld must be 0 or >= n");
    rp.n = n; rp.ld = a->ld ? a->ld : n; rp.T = a->T; rp.deterministic = a->deterministic; rp.auto_reset = a->auto_reset;
    rp.has_actor = a->actor != nullptr;
    rp.keep_params = a->keep_params != 0;
    rp.a_std = expf(a->a_std_log);
    rp.reward_scale = a->reward_scale; rp.gamma = a->gamma; rp.seed = a->seed; rp.env_offset = a->env_offset; rp.tick0 = a->tick0;
    rp.S = S;
    for (int k = 0; k < kMaxS; ++k) {
        rp.priorK[k] = k < S ? a->priorK_host[k] : 0.0;
        rp.priorKf[k] = (float)rp.priorK[k];
    }
    rp.reward_scale_f = (float)a->reward_scale;
    rp.reward_scale_exact = (double)rp.reward_scale_f == a->reward_scale;
    rp.gamma_f = (float)a->gamma;
    rp.eps = a->eps; rp.pn1 = a->pnoise1; rp.pn2 = a->pnoise2;
    rp.buf_state = a->buf_state; rp.buf_other = a->buf_other; rp.env_action = a->env_action;
    rp.stats = a->stats; rp.status = a->status;
    if (rp.has_actor) {
        PIME_REQUIRE(a->actor_pack, "actor_pack is NULL");
        PIME_REQUIRE(a->actor->kind == PIME_ACTOR_PLAIN || a->actor->kind == PIME_ACTOR_MODULAR, "actor kind");
        PIME_REQUIRE(a->actor->state_dim == S, "actor state_dim does not match the env observation");
        PIME_REQUIRE(tc::make_pack_layout(*a->actor, L), "unsupported actor dimensions");
        PIME_REQUIRE(a->actor->precision == PIME_PRECISION_TC || a->actor->precision == PIME_PRECISION_FP32, "actor precision");
    }
    return PIME_OK;
}

}  // namespace pime
