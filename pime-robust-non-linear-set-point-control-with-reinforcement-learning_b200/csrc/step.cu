// step.cu -- stand-alone (gym-API) kernels: reset / step for both plants, titration table, prior action,
// GAE scan, episode statistics.  One thread per env, SoA state, grid-stride over a grid sized in multiples of
// the SM count.  HBM-bound in fp32 (57 B / env-step water tank, 53 B pH; DESIGN.md section 4).
#include <initializer_list>

#include "plants.cuh"

namespace pime {

constexpr int kBlock = 256;

// ---------------------------------------------------------------------------------------------- water tank
template <typename T>
__device__ __forceinline__ void wt_write_obs(const WtConst<T> &c, const WtPtrs<T> &p, const WtEnv<T> &e, int64_t i, int64_t n,
                                             T *obs_out, bool fill_frames) {
    if (c.obs_mode == PIME_WT_OBS_STACKING) {
        const int k = c.num_stack;
        if (fill_frames) {  // reset: every frame = the new state (nonlinear_watertank.py:1183-1184)
            for (int j = 0; j < k; ++j) {
                p.frames[(int64_t)(3 * j + 0) * n + i] = e.h1;
                p.frames[(int64_t)(3 * j + 1) * n + i] = e.h2;
                p.frames[(int64_t)(3 * j + 2) * n + i] = e.r;
            }
        } else {            // step: drop the oldest frame, append the new one (:1145-1146)
            for (int j = 0; j < 3 * (k - 1); ++j) p.frames[(int64_t)j * n + i] = p.frames[(int64_t)(j + 3) * n + i];
            p.frames[(int64_t)(3 * (k - 1) + 0) * n + i] = e.h1;
            p.frames[(int64_t)(3 * (k - 1) + 1) * n + i] = e.h2;
            p.frames[(int64_t)(3 * (k - 1) + 2) * n + i] = e.r;
        }
        if (obs_out)
            for (int j = 0; j < 3 * k; ++j) obs_out[(int64_t)j * n + i] = p.frames[(int64_t)j * n + i];
    } else if (obs_out) {
        obs_out[i] = e.h1;
        obs_out[n + i] = e.h2;
        obs_out[2 * n + i] = e.r;
        if (c.obs_mode == PIME_WT_OBS_INTEGRATOR) obs_out[3 * n + i] = e.I;
    }
}

template <typename T>
__global__ void __launch_bounds__(kBlock) wt_step_kernel(WtConst<T> c, int64_t i_begin, int64_t n, WtPtrs<T> p,
                                                         const T *__restrict__ action, const T *__restrict__ noise1,
                                                         const T *__restrict__ noise2, uint64_t seed, uint64_t env_offset,
                                                         uint32_t tick, T *obs_out, T *__restrict__ reward,
                                                         uint8_t *__restrict__ done) {
    const bool integ = c.obs_mode == PIME_WT_OBS_INTEGRATOR;
    for (int64_t i = i_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        WtEnv<T> e;
        p.load(e, i, integ);
        T nz1 = (T)0, nz2 = (T)0;
        if (noise1) {
            nz1 = noise1[i];
            nz2 = noise2[i];
        } else if (c.noise_scale > (T)0) {  // get_noise (:271-272), Philox instead of numpy's global stream
            Philox4 w = philox4x32_10(seed, env_offset + (uint64_t)i, tick, kStreamStep);
            float z0, z1;
            box_muller(w.v[0], w.v[1], z0, z1);
            nz1 = (T)z0 * c.noise_scale;
            nz2 = (T)z1 * c.noise_scale;
        }
        T rew;
        bool dn;
        wt_advance(c, e, action[i], nz1, nz2, rew, dn);
        p.store_step(e, i, integ);
        if (p.ep_return) p.ep_return[i] += rew;
        reward[i] = rew;
        done[i] = dn ? 1 : 0;
        if (dn && p.last_h1) { p.last_h1[i] = e.h1; p.last_h2[i] = e.h2; }                      // :819-821
        wt_write_obs(c, p, e, i, n, obs_out, false);
    }
}


// ---- float flavour, goal / integrator observation: FOUR consecutive envs per thread.  The SoA arrays are contiguous, so
// a thread's four envs are one 16-byte element of every array (float4 / int4 / uchar4 loads and stores; a warp moves 512
// contiguous bytes per array), and the four independent 20-sub-step Euler chains are interleaved so that the MUFU.SQRT
// latency of one chain is covered by the other three.  57 B of HBM traffic per env-step against 40 MUFU ops: the HBM floor
// and the MUFU floor of this kernel coincide (DESIGN.md section 4), hence nothing may be left serialised.
constexpr int kVec = 4;
constexpr int kVecBlock = 128;

__device__ __forceinline__ float4 ld4(const float *p, int64_t g) { return __ldcs(reinterpret_cast<const float4 *>(p) + g); }
__device__ __forceinline__ void st4(float *p, int64_t g, const float (&v)[4]) {
    __stcs(reinterpret_cast<float4 *>(p) + g, make_float4(v[0], v[1], v[2], v[3]));
}
__device__ __forceinline__ void unpack4(const float4 &v, float (&o)[4]) { o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w; }

__global__ void __launch_bounds__(kVecBlock) wt_step_vec4_kernel(WtConst<float> c, int64_t groups, int64_t n, WtPtrs<float> p,
                                                                 const float *__restrict__ action, const float *__restrict__ noise1,
                                                                 const float *__restrict__ noise2, uint64_t seed, uint64_t env_offset,
                                                                 uint32_t tick, float *obs_out, float *__restrict__ reward,
                                                                 uint8_t *__restrict__ done) {
    const bool integ = c.obs_mode == PIME_WT_OBS_INTEGRATOR;
    const bool philox = noise1 == nullptr && c.noise_scale > 0.0f;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += (int64_t)gridDim.x * blockDim.x) {
        float h1[4], h2[4], r[4], I[4], a1[4], a2[4], Kp[4], act[4], nz1[4], nz2[4], rew[4];
        int t[4];
        unpack4(ld4(p.h1, g), h1); unpack4(ld4(p.h2, g), h2); unpack4(ld4(p.r, g), r);
        unpack4(ld4(p.a1, g), a1); unpack4(ld4(p.a2, g), a2); unpack4(ld4(p.Kp, g), Kp);
        unpack4(ld4(action, g), act);
        if (integ) unpack4(ld4(p.I, g), I);
        else I[0] = I[1] = I[2] = I[3] = 0.0f;
        {
            const int4 tv = __ldcs(reinterpret_cast<const int4 *>(p.t) + g);
            t[0] = tv.x; t[1] = tv.y; t[2] = tv.z; t[3] = tv.w;
        }
        if (noise1) {
            unpack4(ld4(noise1, g), nz1); unpack4(ld4(noise2, g), nz2);
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                nz1[e] = nz2[e] = 0.0f;
                if (philox) {  // get_noise (:271-272), Philox instead of numpy's global stream
                    const Philox4 w = philox4x32_10(seed, env_offset + (uint64_t)(4 * g + e), tick, kStreamStep);
                    float z0, z1;
                    box_muller(w.v[0], w.v[1], z0, z1);
                    nz1[e] = z0 * c.noise_scale;
                    nz2[e] = z1 * c.noise_scale;
                }
            }
        }
        // the four Euler chains, sub-step by sub-step (same arithmetic as wt_integrate<float>)
        float k1[4], k2a[4], k2b[4], b1[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float u = wt_u(c, act[e]);                                                    // :260
            k1[e] = -a1[e] * c.sq2G_dt_over_A1;
            k2a[e] = a1[e] * c.sq2G_dt_over_A2;
            k2b[e] = -a2[e] * c.sq2G_dt_over_A2;
            b1[e] = Kp[e] * u * c.dt_over_A1;
        }
#pragma unroll 2
        for (int k = 0; k < c.n_discrete; ++k) {
            float s1[4], s2[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) { s1[e] = Num<float>::sqrt(h1[e]); s2[e] = Num<float>::sqrt(h2[e]); }
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float n1 = fmaf(k1[e], s1[e], h1[e] + b1[e]);
                const float n2 = fmaf(k2a[e], s1[e], fmaf(k2b[e], s2[e], h2[e]));
                h1[e] = fmaxf(n1, 0.0f);
                h2[e] = fmaxf(n2, 0.0f);
            }
        }
        uint32_t dn4 = 0;
        bool any_done = false;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            t[e] += 1;                                                                          // :801
            h1[e] = fmaxf(h1[e] + nz1[e], 0.0f);                                                // :810-813
            h2[e] = fmaxf(h2[e] + nz2[e], 0.0f);
            float rw = reward_of<float>(c.reward_type, fabsf(h2[e] - r[e]), c.z1, c.thr);       // :815
            const bool dn = t[e] >= c.max_step;                                                 // :816-821
            if (integ) {
                const float integ_raw = I[e] + (r[e] - h2[e]);                                  // :822-823
                rw = rw + (-c.Ipunish) * fabsf(integ_raw);                                      // :824
                I[e] = clampT(integ_raw, -c.Imax, c.Imax);                                      // :825
            }
            rew[e] = rw;
            dn4 |= (dn ? 1u : 0u) << (8 * e);
            any_done |= dn;
        }
        st4(p.h1, g, h1); st4(p.h2, g, h2);
        if (integ) st4(p.I, g, I);
        __stcs(reinterpret_cast<int4 *>(p.t) + g, make_int4(t[0], t[1], t[2], t[3]));
        if (p.ep_return) {
            float er[4];
            unpack4(ld4(p.ep_return, g), er);
#pragma unroll
            for (int e = 0; e < 4; ++e) er[e] += rew[e];
            st4(p.ep_return, g, er);
        }
        st4(reward, g, rew);
        __stcs(reinterpret_cast<uint32_t *>(done) + g, dn4);
        if (any_done && p.last_h1) {                                                            // :819-821
#pragma unroll
            for (int e = 0; e < 4; ++e)
                if ((dn4 >> (8 * e)) & 1u) { p.last_h1[4 * g + e] = h1[e]; p.last_h2[4 * g + e] = h2[e]; }
        }
        if (obs_out) {
            st4(obs_out, g, h1);
            st4(obs_out + n, g, h2);
            st4(obs_out + 2 * n, g, r);
            if (integ) st4(obs_out + 3 * n, g, I);
        }
    }
}

// every array the vectorised kernels touch must be 16-byte aligned (4 envs per element); n % 4 == 0 keeps obs_out rows aligned
static bool aligned16(std::initializer_list<const void *> ptrs) {
    for (const void *q : ptrs)
        if (q && ((uintptr_t)q & 15)) return false;
    return true;
}

template <typename T>
__global__ void __launch_bounds__(kBlock) wt_reset_kernel(WtConst<T> c, int64_t n, WtPtrs<T> p, uint64_t seed, uint64_t env_offset,
                                                          int resample, const uint8_t *__restrict__ mask, T *obs_out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (mask && !mask[i]) continue;
        WtEnv<T> e;
        p.load_params(e, i);
        uint32_t ep = p.episode[i];
        double u[6];
        reset_uniforms(seed, env_offset + (uint64_t)i, ep, u);
        wt_reset(c, e, u, resample != 0);
        if (c.from_last) wt_reset_levels_from_last(e, u, p.last_h1[i], p.last_h2[i]);
        p.episode[i] = ep + 1;
        p.store(e, i, p.I != nullptr);   // I = 0 and t = 0 after wt_reset; I is zeroed whenever the array exists
        if (p.ep_return) p.ep_return[i] = (T)0;
        wt_write_obs(c, p, e, i, n, obs_out, true);
    }
}

template <typename T>
static int wt_step_impl(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const T *action, const T *noise1,
                        const T *noise2, uint64_t seed, uint64_t env_offset, uint32_t tick, T *obs_out, T *reward, uint8_t *done,
                        void *stream) {
    if (int rc = validate_wt(cfg, n, st)) return rc;
    PIME_REQUIRE(action && reward && done, "null action/reward/done");
    PIME_REQUIRE((noise1 == nullptr) == (noise2 == nullptr), "noise1/noise2 must both be given or both be NULL");
    if (int rc = require_device()) return rc;
    if (n == 0) return PIME_OK;
    const WtPtrs<T> p(*st);
    int64_t i_begin = 0;
    if constexpr (sizeof(T) == 4) {   // float: 4 envs per thread where layout and alignment allow, scalar kernel for the tail
        const bool vec_ok = cfg->obs_mode != PIME_WT_OBS_STACKING && n >= kVec && (obs_out == nullptr || n % kVec == 0) &&
                            aligned16({p.h1, p.h2, p.r, p.I, p.a1, p.a2, p.Kp, p.t, p.ep_return, action, noise1, noise2, obs_out,
                                       reward}) && ((uintptr_t)done & 3) == 0;
        if (vec_ok) {
            const int64_t groups = n / kVec;
            wt_step_vec4_kernel<<<grid_for(groups, kVecBlock, 32), kVecBlock, 0, (cudaStream_t)stream>>>(
                make_wt_const<float>(*cfg), groups, n, p, (const float *)action, (const float *)noise1, (const float *)noise2, seed,
                env_offset, tick, (float *)obs_out, (float *)reward, done);
            PIME_LAUNCH_CHECK();
            i_begin = groups * kVec;
            if (i_begin == n) return PIME_OK;
        }
    }
    wt_step_kernel<T><<<grid_for(n - i_begin, kBlock), kBlock, 0, (cudaStream_t)stream>>>(make_wt_const<T>(*cfg), i_begin, n, p,
                                                                                        action, noise1, noise2, seed, env_offset,
                                                                                        tick, obs_out, reward, done);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

template <typename T>
static int wt_reset_impl(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, uint64_t seed, uint64_t env_offset,
                         int resample, const uint8_t *mask, T *obs_out, void *stream) {
    if (int rc = validate_wt(cfg, n, st)) return rc;
    if (int rc = require_device()) return rc;
    if (n == 0) return PIME_OK;
    wt_reset_kernel<T><<<grid_for(n, kBlock), kBlock, 0, (cudaStream_t)stream>>>(make_wt_const<T>(*cfg), n, WtPtrs<T>(*st), seed,
                                                                                env_offset, resample, mask, obs_out);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

// ---------------------------------------------------------------------------------------------- pH
template <typename T>
__device__ __forceinline__ void ph_write_obs(const PhConst<T> &c, const PhEnv<T> &e, int64_t i, int64_t n, T *obs_out) {
    if (!obs_out) return;
    obs_out[i] = e.y;
    obs_out[n + i] = e.r;
    if (c.integrator_mode != PIME_PH_NO_INTEGRATOR) obs_out[2 * n + i] = e.I;
}

template <typename T>
__global__ void __launch_bounds__(kBlock) ph_step_kernel(PhConst<T> c, const T *__restrict__ table, int64_t n, PhPtrs<T> p,
                                                         const T *__restrict__ action, T *obs_out, T *__restrict__ reward,
                                                         uint8_t *__restrict__ done, int32_t *status) {
    const bool integ = c.integrator_mode != PIME_PH_NO_INTEGRATOR;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        PhEnv<T> e;
        p.load(e, i, integ);
        T rew;
        bool dn;
        bool ok = ph_advance(c, table, e, action[i], rew, dn);
        if (!ok && status) atomicMin(status, (int32_t)PIME_ERANGE);
        p.store_step(e, i, integ);
        if (p.ep_return) p.ep_return[i] += rew;
        reward[i] = rew;
        done[i] = dn ? 1 : 0;
        if (dn && p.last_x) p.last_x[i] = e.x;                                                  // :345-346
        ph_write_obs(c, e, i, n, obs_out);
    }
}

template <typename T>
__global__ void __launch_bounds__(kBlock) ph_reset_kernel(PhConst<T> c, const T *__restrict__ table, int64_t n, PhPtrs<T> p,
                                                          uint64_t seed, uint64_t env_offset, int resample,
                                                          const uint8_t *__restrict__ mask, T *obs_out, int32_t *status) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (mask && !mask[i]) continue;
        PhEnv<T> e;
        p.load_system(e, i);
        T qww = p.qww[i], qc = p.qc[i];
        uint32_t ep = p.episode[i];
        double u[6];
        reset_uniforms(seed, env_offset + (uint64_t)i, ep, u);
        bool ok = ph_reset(c, table, e, qww, qc, u, resample != 0, c.from_last ? p.last_x[i] : nan_of<double>());
        if (!ok && status) atomicMin(status, (int32_t)PIME_ERANGE);
        p.episode[i] = ep + 1;
        p.qww[i] = qww; p.qc[i] = qc;
        p.store_system(e, i);                 // the new episode's system, set-point and step state
        p.r[i] = e.r;
        p.store_step(e, i, p.I != nullptr);   // I = 0 and t = 0 after ph_reset; I is zeroed whenever the array exists
        if (p.ep_return) p.ep_return[i] = (T)0;
        ph_write_obs(c, e, i, n, obs_out);
    }
}

template <typename T>
__global__ void __launch_bounds__(kBlock) ph_update_system_kernel(double sample_t, int64_t n, PhPtrs<T> p) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        PhEnv<T> e;
        ph_update_system<T>(sample_t, p.qww[i], p.qc[i], e.A, e.B, e.C);
        p.store_system(e, i);
    }
}

// Titration table (ph.py:72-84).  One thread per grid point: the quartic f(H) = H^4 + a H^3 + b H^2 + c H + d has
// d < 0 and exactly one positive root; bracket it by bisection on [1e-30, 4] (f(lo) < 0 < f(hi)), then run the
// reference's own iteration H <- |H - f/f'| until it stops moving (its fixed point is what the reference's
// warm-started 5-step chain converges to).
__global__ void __launch_bounds__(kBlock) ph_table_kernel(int table_len, double step, double kw, double kchem, double ka,
                                                          double MNaOH, double MHA, double MNH3, double *__restrict__ t64,
                                                          float *__restrict__ t32) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= table_len) return;
    double m = (double)i * step;
    double ak = MNH3 - m + MNaOH + kchem + ka;
    double bk = (kchem + ka) * MNaOH - (kchem + ka) * m - kw + MNH3 * ka + kchem * ka - ka * MHA;
    double ck = MNaOH * kchem * ka - kw * (ka + kchem) - m * kchem * ka - ka * kchem * MHA;
    double dk = -kchem * ka * kw;
    auto f = [&](double H) { return (((H + ak) * H + bk) * H + ck) * H + dk; };
    double lo = 1e-30, hi = 4.0;
    for (int it = 0; it < 200; ++it) {  // geometric bisection: the root spans 1e-12 .. 1
        double mid = sqrt(lo * hi);
        if (f(mid) > 0.0) hi = mid; else lo = mid;
        if (hi <= lo * (1.0 + 1e-9)) break;
    }
    double H = sqrt(lo * hi);
    for (int it = 0; it < 50; ++it) {
        double H2 = H * H, H3 = H2 * H, H4 = H3 * H;
        double num = H4 + ak * H3 + bk * H2 + ck * H + dk;
        double den = 4 * H3 + 3 * ak * H2 + 2 * bk * H + ck;
        double Hn = fabs(H - num / den);
        bool stop = fabs(Hn - H) <= 4e-16 * Hn;
        H = Hn;
        if (stop) break;
    }
    double v = -log10(H);
    t64[i] = v;
    if (t32) t32[i] = (float)v;
}

template <typename T>
static int ph_step_impl(const pime_ph_config *cfg, const T *table, int64_t n, const pime_ph_state *st, const T *action,
                        T *obs_out, T *reward, uint8_t *done, int32_t *status, void *stream) {
    if (int rc = validate_ph(cfg, n, st)) return rc;
    PIME_REQUIRE(table && action && reward && done, "null table/action/reward/done");
    if (int rc = require_device()) return rc;
    if (n == 0) return PIME_OK;
    ph_step_kernel<T><<<grid_for(n, kBlock), kBlock, 0, (cudaStream_t)stream>>>(make_ph_const<T>(*cfg), table, n, PhPtrs<T>(*st),
                                                                               action, obs_out, reward, done, status);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

template <typename T>
static int ph_reset_impl(const pime_ph_config *cfg, const T *table, int64_t n, const pime_ph_state *st, uint64_t seed,
                         uint64_t env_offset, int resample, const uint8_t *mask, T *obs_out, int32_t *status, void *stream) {
    if (int rc = validate_ph(cfg, n, st)) return rc;
    PIME_REQUIRE(table, "null table");
    if (int rc = require_device()) return rc;
    if (n == 0) return PIME_OK;
    ph_reset_kernel<T><<<grid_for(n, kBlock), kBlock, 0, (cudaStream_t)stream>>>(make_ph_const<T>(*cfg), table, n, PhPtrs<T>(*st),
                                                                                seed, env_offset, resample, mask, obs_out, status);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

template <typename T> static int ph_update_impl(const pime_ph_config *cfg, int64_t n, const pime_ph_state *st, void *stream) {
    if (int rc = validate_ph(cfg, n, st)) return rc;
    if (int rc = require_device()) return rc;
    if (n == 0) return PIME_OK;
    ph_update_system_kernel<T><<<grid_for(n, kBlock), kBlock, 0, (cudaStream_t)stream>>>(cfg->sample_t, n, PhPtrs<T>(*st));
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

// ---------------------------------------------------------------------------------------------- prior action
struct PriorK {
    double k[32];
};

template <typename T>
__global__ void __launch_bounds__(kBlock) prior_kernel(int64_t n, int S, const T *__restrict__ obs, PriorK K, int clip,
                                                       T *__restrict__ out) {
    using N = Num<T>;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        T acc = (T)0;
        for (int j = 0; j < S; ++j) acc = N::add(acc, N::mul(obs[(int64_t)j * n + i], (T)K.k[j]));
        acc = -acc;  // - state @ K.T  (nonlinear_watertank.py:757-758)
        if (clip) acc = clampT(acc, (T)-1, (T)1);
        out[i] = acc;
    }
}

template <typename T>
static int prior_impl(int64_t n, int32_t S, const T *obs, const double *K_host, int clip, T *out, void *stream) {
    PIME_REQUIRE(obs && K_host && out, "null pointer");
    PIME_REQUIRE(S >= 1 && S <= 32, "S must be in [1,32]");
    if (int rc = require_device()) return rc;
    if (n <= 0) return PIME_OK;
    PriorK K;
    for (int j = 0; j < 32; ++j) K.k[j] = j < S ? K_host[j] : 0.0;
    prior_kernel<T><<<grid_for(n, kBlock), kBlock, 0, (cudaStream_t)stream>>>(n, S, obs, K, clip, out);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

// ---------------------------------------------------------------------------------------------- GAE scan
// AgentPPO.compute_reward_gae (agent.py:685-708) per env column of a time-major replay.
__global__ void __launch_bounds__(kBlock) gae_kernel(int64_t n, int T, const float *__restrict__ reward,
                                                     const float *__restrict__ mask, int stride,
                                                     const float *__restrict__ value, float lam, float *__restrict__ r_sum,
                                                     float *__restrict__ adv) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float pre_r = 0.f, pre_a = 0.f;
        for (int s = T - 1; s >= 0; --s) {
            int64_t q = (int64_t)s * n + i;
            float rw = reward[q * stride], mk = mask[q * stride], v = value[q];
            float rs = rw + mk * pre_r;          // agent.py:701
            pre_r = rs;
            float a = rw + mk * (pre_a - v);     // agent.py:704
            pre_a = v + a * lam;                 // agent.py:705
            r_sum[q] = rs;
            adv[q] = a;
        }
    }
}

// ---------------------------------------------------------------------------------------------- episode stats
template <typename T>
__global__ void __launch_bounds__(kBlock) stats_kernel(int64_t n, const T *__restrict__ ret, double *stats) {
    double s = 0.0, s2 = 0.0, cnt = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double v = (double)ret[i];
        s += v; s2 += v * v; cnt += 1.0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        s2 += __shfl_xor_sync(0xffffffffu, s2, o);
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    }
    __shared__ double sh[3][kBlock / 32];
    int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) { sh[0][w] = s; sh[1][w] = s2; sh[2][w] = cnt; }
    __syncthreads();
    if (w == 0) {
        s = l < kBlock / 32 ? sh[0][l] : 0.0;
        s2 = l < kBlock / 32 ? sh[1][l] : 0.0;
        cnt = l < kBlock / 32 ? sh[2][l] : 0.0;
#pragma unroll
        for (int o = 4; o > 0; o >>= 1) {
            s += __shfl_xor_sync(0xffffffffu, s, o);
            s2 += __shfl_xor_sync(0xffffffffu, s2, o);
            cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        }
        if (l == 0) {
            atomicAdd(stats + 0, s);
            atomicAdd(stats + 1, s2);
            atomicAdd(stats + 2, cnt);
        }
    }
}

__global__ void philox_probe_kernel(uint64_t seed, uint64_t index, uint32_t tick, uint32_t stream_id, uint32_t *out) {
    Philox4 w = philox4x32_10(seed, index, tick, stream_id);
    for (int j = 0; j < 4; ++j) out[j] = w.v[j];
}

}  // namespace pime

// ================================================================================================ C ABI
using namespace pime;

extern "C" {

void pime_wt_default_config(pime_wt_config *c) {
    if (!c) return;
    *c = pime_wt_config{};
    c->A1 = 1; c->A2 = 1; c->G = 980; c->sample_t = 2.0; c->n_discrete = 20; c->max_step = 200; c->P_max_action = 10.0;
    c->reward_type = PIME_REWARD_SQUARE_DISTANCE; c->obs_mode = PIME_WT_OBS_INTEGRATOR; c->num_stack = 0;
    c->z1 = 1.0; c->distance_threshold = 0.05; c->integral_max = 25.0; c->integral_punish = 0.0; c->noise_scale = 0.01;
    c->a1_lo = 0.0015; c->a1_hi = 0.0024; c->a2_lo = 0.0015; c->a2_hi = 0.0024; c->Kp_lo = 0.07; c->Kp_hi = 0.17;
    c->h_lo = 0.0; c->h_hi = 10.0; c->r_lo = 0.0; c->r_hi = 10.0;
}

void pime_ph_default_config(pime_ph_config *c) {
    if (!c) return;
    *c = pime_ph_config{};
    c->reward_type = PIME_REWARD_SQUARE_DISTANCE; c->integrator_mode = PIME_PH_INTEGRATOR; c->max_episode_steps = 50;
    c->table_len = 100000; c->act_low = 0.0; c->act_high = 1.5; c->sample_t = 20.0; c->mhcl_step = 1e-5;
    c->distance_threshold = 0.05; c->integral_max = 25.0; c->integral_punish = 0.0; c->action_punishment = 0.0;
    c->kw = 1e-14; c->kchem = 5.6e-10; c->ka = 0.5e-5; c->MNaOH = 0.01; c->MHA = 0.005; c->MNH3 = 0.01;
    c->qww_lo = 0.005; c->qww_hi = 0.015; c->qc_lo = 0.0015; c->qc_hi = 0.0025;
    c->x_lo = 0.0; c->x_hi = 50.0; c->r_lo = 3.0; c->r_hi = 11.0;
}

int pime_wt_reset_f32(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, uint64_t seed, uint64_t env_offset,
                      int resample_params, const uint8_t *mask, float *obs_out, void *stream) {
    return wt_reset_impl<float>(cfg, n, st, seed, env_offset, resample_params, mask, obs_out, stream);
}
int pime_wt_reset_f64(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, uint64_t seed, uint64_t env_offset,
                      int resample_params, const uint8_t *mask, double *obs_out, void *stream) {
    return wt_reset_impl<double>(cfg, n, st, seed, env_offset, resample_params, mask, obs_out, stream);
}
int pime_wt_step_f32(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const float *action, const float *noise1,
                     const float *noise2, uint64_t seed, uint64_t env_offset, uint32_t tick, float *obs_out, float *reward,
                     uint8_t *done, void *stream) {
    return wt_step_impl<float>(cfg, n, st, action, noise1, noise2, seed, env_offset, tick, obs_out, reward, done, stream);
}
int pime_wt_step_f64(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const double *action, const double *noise1,
                     const double *noise2, uint64_t seed, uint64_t env_offset, uint32_t tick, double *obs_out, double *reward,
                     uint8_t *done, void *stream) {
    return wt_step_impl<double>(cfg, n, st, action, noise1, noise2, seed, env_offset, tick, obs_out, reward, done, stream);
}

int pime_ph_table_build(const pime_ph_config *cfg, double *table_f64, float *table_f32, void *stream) {
    PIME_REQUIRE(cfg && table_f64, "null config/table");
    PIME_REQUIRE(cfg->table_len > 1, "table_len");
    if (int rc = require_device()) return rc;
    int grid = (cfg->table_len + kBlock - 1) / kBlock;
    ph_table_kernel<<<grid, kBlock, 0, (cudaStream_t)stream>>>(cfg->table_len, cfg->mhcl_step, cfg->kw, cfg->kchem, cfg->ka,
                                                              cfg->MNaOH, cfg->MHA, cfg->MNH3, table_f64, table_f32);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

int pime_ph_update_system_f32(const pime_ph_config *cfg, int64_t n, const pime_ph_state *st, void *stream) {
    return ph_update_impl<float>(cfg, n, st, stream);
}
int pime_ph_update_system_f64(const pime_ph_config *cfg, int64_t n, const pime_ph_state *st, void *stream) {
    return ph_update_impl<double>(cfg, n, st, stream);
}
int pime_ph_reset_f32(const pime_ph_config *cfg, const float *table, int64_t n, const pime_ph_state *st, uint64_t seed,
                      uint64_t env_offset, int resample_params, const uint8_t *mask, float *obs_out, int32_t *status,
                      void *stream) {
    return ph_reset_impl<float>(cfg, table, n, st, seed, env_offset, resample_params, mask, obs_out, status, stream);
}
int pime_ph_reset_f64(const pime_ph_config *cfg, const double *table, int64_t n, const pime_ph_state *st, uint64_t seed,
                      uint64_t env_offset, int resample_params, const uint8_t *mask, double *obs_out, int32_t *status,
                      void *stream) {
    return ph_reset_impl<double>(cfg, table, n, st, seed, env_offset, resample_params, mask, obs_out, status, stream);
}
int pime_ph_step_f32(const pime_ph_config *cfg, const float *table, int64_t n, const pime_ph_state *st, const float *action,
                     float *obs_out, float *reward, uint8_t *done, int32_t *status, void *stream) {
    return ph_step_impl<float>(cfg, table, n, st, action, obs_out, reward, done, status, stream);
}
int pime_ph_step_f64(const pime_ph_config *cfg, const double *table, int64_t n, const pime_ph_state *st, const double *action,
                     double *obs_out, double *reward, uint8_t *done, int32_t *status, void *stream) {
    return ph_step_impl<double>(cfg, table, n, st, action, obs_out, reward, done, status, stream);
}

int pime_prior_action_f32(int64_t n, int32_t S, const float *obs, const double *K_host, int clip, float *out, void *stream) {
    return prior_impl<float>(n, S, obs, K_host, clip, out, stream);
}
int pime_prior_action_f64(int64_t n, int32_t S, const double *obs, const double *K_host, int clip, double *out, void *stream) {
    return prior_impl<double>(n, S, obs, K_host, clip, out, stream);
}

int pime_gae_scan(int64_t n, int32_t T, const float *reward, const float *mask, int32_t stride, const float *value,
                  float lambda_gae, float *r_sum, float *adv, void *stream) {
    PIME_REQUIRE(reward && mask && value && r_sum && adv, "null pointer");
    PIME_REQUIRE(T >= 1 && stride >= 1, "T/stride");
    if (int rc = require_device()) return rc;
    if (n <= 0) return PIME_OK;
    gae_kernel<<<grid_for(n, kBlock), kBlock, 0, (cudaStream_t)stream>>>(n, T, reward, mask, stride, value, lambda_gae, r_sum, adv);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

int pime_reduce_episode_stats_f32(int64_t n, const float *ep_return, double *stats, void *stream) {
    PIME_REQUIRE(ep_return && stats, "null pointer");
    if (int rc = require_device()) return rc;
    if (n <= 0) return PIME_OK;
    stats_kernel<float><<<grid_for(n, kBlock, 4), kBlock, 0, (cudaStream_t)stream>>>(n, ep_return, stats);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}
int pime_reduce_episode_stats_f64(int64_t n, const double *ep_return, double *stats, void *stream) {
    PIME_REQUIRE(ep_return && stats, "null pointer");
    if (int rc = require_device()) return rc;
    if (n <= 0) return PIME_OK;
    stats_kernel<double><<<grid_for(n, kBlock, 4), kBlock, 0, (cudaStream_t)stream>>>(n, ep_return, stats);
    PIME_LAUNCH_CHECK();
    return PIME_OK;
}

int pime_philox_probe(uint64_t seed, uint64_t index, uint32_t tick, uint32_t stream_id, uint32_t *out_host) {
    PIME_REQUIRE(out_host, "null pointer");
    if (int rc = require_device()) return rc;
    uint32_t *d = nullptr;
    PIME_CUDA(cudaMalloc(&d, 16));
    philox_probe_kernel<<<1, 1>>>(seed, index, tick, stream_id, d);
    cudaError_t e = cudaMemcpy(out_host, d, 16, cudaMemcpyDeviceToHost);
    cudaFree(d);
    PIME_CUDA(e);
    return PIME_OK;
}

}  // extern "C"
