// plants.cuh -- per-env device arithmetic of the two gym_control plants (one thread = one env, state in registers), the
// typed view of each plant's SoA state arrays and the argument checks of its entry points.
// Used by the stand-alone step/reset kernels (step.cu) and by the fused rollout kernels (rollout_impl.cuh).
#pragma once

#include "pime_common.cuh"

namespace pime {

// ============================================================================================== water tank
template <typename T> struct WtConst {
    T twoG, A1, A2, dt, Pmax, z1, thr, Imax, Ipunish, noise_scale;
    // f32 fast path: sqrt(2G)*dt/A folded once per launch
    T sq2G_dt_over_A1, sq2G_dt_over_A2, dt_over_A1, halfP;
    T a1_lo, a1_w, a2_lo, a2_w, Kp_lo, Kp_w, h_lo, h_w, r_lo, r_w;
    int n_discrete, max_step, reward_type, obs_mode, num_stack, from_last;
};

template <typename T> inline WtConst<T> make_wt_const(const pime_wt_config &c) {
    WtConst<T> k;
    k.twoG = (T)(2 * c.G);
    k.A1 = (T)c.A1; k.A2 = (T)c.A2;
    k.dt = (T)(c.sample_t / (double)c.n_discrete);  // delta_t (nonlinear_watertank.py:151)
    k.Pmax = (T)c.P_max_action;
    k.z1 = (T)c.z1; k.thr = (T)c.distance_threshold; k.Imax = (T)c.integral_max; k.Ipunish = (T)c.integral_punish;
    k.noise_scale = (T)c.noise_scale;
    double dt = c.sample_t / (double)c.n_discrete;
    k.sq2G_dt_over_A1 = (T)(sqrt(2 * c.G) * dt / c.A1);
    k.sq2G_dt_over_A2 = (T)(sqrt(2 * c.G) * dt / c.A2);
    k.dt_over_A1 = (T)(dt / c.A1);
    k.halfP = (T)(c.P_max_action / 2);
    k.a1_lo = (T)c.a1_lo; k.a1_w = (T)(c.a1_hi - c.a1_lo);
    k.a2_lo = (T)c.a2_lo; k.a2_w = (T)(c.a2_hi - c.a2_lo);
    k.Kp_lo = (T)c.Kp_lo; k.Kp_w = (T)(c.Kp_hi - c.Kp_lo);
    k.h_lo = (T)c.h_lo; k.h_w = (T)(c.h_hi - c.h_lo);
    k.r_lo = (T)c.r_lo; k.r_w = (T)(c.r_hi - c.r_lo);
    k.n_discrete = c.n_discrete; k.max_step = c.max_step; k.reward_type = c.reward_type;
    k.obs_mode = c.obs_mode; k.num_stack = c.num_stack; k.from_last = c.reset_from_last_state;
    return k;
}

template <typename T> struct WtEnv {
    T h1, h2, r, I, a1, a2, Kp;
    int t;
};

// The per-env arrays of pime_wt_state with their element types.  The loaders and storers are small on purpose: each
// kernel reads and writes only the arrays it needs (HBM traffic is the cost of the stand-alone kernels).
template <typename T> struct WtPtrs {
    T *h1, *h2, *r, *I, *a1, *a2, *Kp, *ep_return, *frames, *last_h1, *last_h2;
    int32_t *t;
    uint32_t *episode;

    WtPtrs() = default;
    explicit WtPtrs(const pime_wt_state &s)
        : h1((T *)s.h1), h2((T *)s.h2), r((T *)s.r), I((T *)s.I), a1((T *)s.a1), a2((T *)s.a2), Kp((T *)s.Kp),
          ep_return((T *)s.ep_return), frames((T *)s.frames), last_h1((T *)s.last_h1), last_h2((T *)s.last_h2), t(s.t),
          episode(s.episode) {}

    // the arrays of envs [off, ...).  frames ([3 num_stack][n], row stride n) is not shifted: a range of envs would need
    // every row shifted and the stride kept, so the stacking observation always runs as a single slice.
    WtPtrs shifted(int64_t off) const {
        auto adv = [off](auto *q) { return q ? q + off : q; };
        WtPtrs p;
        p.h1 = adv(h1); p.h2 = adv(h2); p.r = adv(r); p.I = adv(I);
        p.a1 = adv(a1); p.a2 = adv(a2); p.Kp = adv(Kp);
        p.ep_return = adv(ep_return); p.frames = frames; p.last_h1 = adv(last_h1); p.last_h2 = adv(last_h2);
        p.t = adv(t); p.episode = adv(episode);
        return p;
    }

    // what env.step() reads; I only when the observation carries the integrator (the array may be NULL otherwise)
    __device__ __forceinline__ void load(WtEnv<T> &e, int64_t i, bool integ) const {
        e.h1 = h1[i]; e.h2 = h2[i]; e.r = r[i];
        e.I = integ ? I[i] : (T)0;
        load_params(e, i);
        e.t = t[i];
    }
    __device__ __forceinline__ void load_params(WtEnv<T> &e, int64_t i) const { e.a1 = a1[i]; e.a2 = a2[i]; e.Kp = Kp[i]; }
    // what env.step() changes (the set-point and the ensemble parameters stay)
    __device__ __forceinline__ void store_step(const WtEnv<T> &e, int64_t i, bool integ) const {
        h1[i] = e.h1; h2[i] = e.h2;
        if (integ) I[i] = e.I;
        t[i] = e.t;
    }
    // everything load() reads
    __device__ __forceinline__ void store(const WtEnv<T> &e, int64_t i, bool integ) const {
        h1[i] = e.h1; h2[i] = e.h2; r[i] = e.r;
        if (integ) I[i] = e.I;
        a1[i] = e.a1; a2[i] = e.a2; Kp[i] = e.Kp;
        t[i] = e.t;
    }
};

// width of the observation vector
inline int wt_obs_dim(const pime_wt_config &c) {
    return c.obs_mode == PIME_WT_OBS_GOAL ? 3 : (c.obs_mode == PIME_WT_OBS_INTEGRATOR ? 4 : 3 * c.num_stack);
}

// The argument checks of every water-tank entry point (step, reset, rollout, host-buffer rollout).  They need no device, so
// the entries run them before require_device().
inline int validate_wt(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st) {
    PIME_REQUIRE(cfg && st, "null config/state");
    PIME_REQUIRE(n >= 0, "negative n");
    PIME_REQUIRE(st->h1 && st->h2 && st->r && st->a1 && st->a2 && st->Kp && st->t && st->episode, "null state array");
    PIME_REQUIRE(cfg->obs_mode >= 0 && cfg->obs_mode <= 2, "obs_mode");
    PIME_REQUIRE(cfg->obs_mode != PIME_WT_OBS_INTEGRATOR || st->I, "integrator array missing");
    PIME_REQUIRE(cfg->obs_mode != PIME_WT_OBS_STACKING || (st->frames && cfg->num_stack >= 1 && cfg->num_stack <= 10),
                 "stacking needs frames and 1 <= num_stack <= 10");
    PIME_REQUIRE(cfg->n_discrete >= 1 && cfg->reward_type >= 0 && cfg->reward_type <= 2, "n_discrete/reward_type");
    PIME_REQUIRE(!cfg->reset_from_last_state || (st->last_h1 && st->last_h2), "reset_from_last_state needs last_h1/last_h2");
    return PIME_OK;
}

// 20 Euler sub-steps (nonlinear_watertank.py:805-809).  f64: the reference's operation order, no contraction.
__device__ __forceinline__ void wt_integrate(const WtConst<double> &c, double a1, double a2, double Kp, double u, double &x1,
                                             double &x2) {
    using N = Num<double>;
    const double na1 = N::div(-a1, c.A1), pa1 = N::div(a1, c.A2), pa2 = N::div(a2, c.A2);
    const double kpu = N::mul(N::div(Kp, c.A1), u);
    for (int k = 0; k < c.n_discrete; ++k) {
        double s1 = N::sqrt(N::mul(c.twoG, x1));
        double s2 = N::sqrt(N::mul(c.twoG, x2));
        double n1 = N::add(x1, N::mul(N::add(N::mul(na1, s1), kpu), c.dt));
        double n2 = N::add(x2, N::mul(N::sub(N::mul(pa1, s1), N::mul(pa2, s2)), c.dt));
        x1 = clip_lo0(n1);
        x2 = clip_lo0(n2);
    }
}

// f32: same recurrence with the constants folded (sqrt(2G h) = sqrt(2G) sqrt(h)) -> 2 MUFU + 4 FMA + 2 FMNMX per sub-step.
__device__ __forceinline__ void wt_integrate(const WtConst<float> &c, float a1, float a2, float Kp, float u, float &x1, float &x2) {
    const float k1 = -a1 * c.sq2G_dt_over_A1;  // coefficient of sqrt(h1) in h1'
    const float k2a = a1 * c.sq2G_dt_over_A2;  // coefficient of sqrt(h1) in h2'
    const float k2b = -a2 * c.sq2G_dt_over_A2; // coefficient of sqrt(h2) in h2'
    const float b1 = Kp * u * c.dt_over_A1;    // pump inflow per sub-step
#pragma unroll 4
    for (int k = 0; k < c.n_discrete; ++k) {
        float s1 = Num<float>::sqrt(x1);
        float s2 = Num<float>::sqrt(x2);
        float n1 = fmaf(k1, s1, x1 + b1);
        float n2 = fmaf(k2a, s1, fmaf(k2b, s2, x2));
        x1 = fmaxf(n1, 0.0f);
        x2 = fmaxf(n2, 0.0f);
    }
}

// f32: u = a*P/2 + P/2 as one FMA (shared by the scalar, the 4-env and the fused kernels, so that an env steps
// identically whichever kernel it lands in)
__device__ __forceinline__ float wt_u(const WtConst<float> &c, float action) { return fmaf(action, c.halfP, c.halfP); }
__device__ __forceinline__ double wt_u(const WtConst<double> &c, double action) { return action * c.halfP + c.halfP; }

// One env.step(): NonLinearWaterTankUniformGoalIntegrator.step (:800-826) / base step (:274-297).
template <typename T>
__device__ __forceinline__ void wt_advance(const WtConst<T> &c, WtEnv<T> &e, T action, T nz1, T nz2, T &reward, bool &done) {
    using N = Num<T>;
    e.t += 1;                                                                                   // :801
    T u;                                                                                        // :260 (no clip)
    if constexpr (sizeof(T) == 4) u = wt_u(c, action);
    else u = N::add(N::div(N::mul(action, c.Pmax), (T)2), N::div(c.Pmax, (T)2));
    T x1 = e.h1, x2 = e.h2;
    wt_integrate(c, e.a1, e.a2, e.Kp, u, x1, x2);
    x1 = clip_lo0(N::add(x1, nz1));                                                             // :810-813
    x2 = clip_lo0(N::add(x2, nz2));
    T rew = reward_of<T>(c.reward_type, N::abs(N::sub(x2, e.r)), c.z1, c.thr);                  // :815
    done = e.t >= c.max_step;                                                                   // :816-821
    if (c.obs_mode == PIME_WT_OBS_INTEGRATOR) {
        T integ = N::add(e.I, N::sub(e.r, x2));                                                 // :822-823
        rew = N::add(rew, N::mul(-c.Ipunish, N::abs(integ)));                                   // :824
        e.I = clampT(integ, -c.Imax, c.Imax);                                                   // :825
    }
    e.h1 = x1;
    e.h2 = x2;
    reward = rew;
}

// low + (high - low) u of numpy's uniform(low, high), product and sum rounded separately: left to itself nvcc contracts
// the expression into one DFMA, and the f64 parameters would no longer be the ones numpy's arithmetic gives
__device__ __forceinline__ double uniform_in(double lo, double w, double u) { return __dadd_rn(lo, __dmul_rn(w, u)); }

// reset_all()/reset_r() (:902-939): u[] are the six uniforms of reset_uniforms().
template <typename T> __device__ __forceinline__ void wt_reset(const WtConst<T> &c, WtEnv<T> &e, const double u[6], bool resample) {
    if (resample) {  // sample_parameters (:890-894): low + (high-low)*u
        e.a1 = (T)uniform_in((double)c.a1_lo, (double)c.a1_w, u[0]);
        e.a2 = (T)uniform_in((double)c.a2_lo, (double)c.a2_w, u[1]);
        e.Kp = (T)uniform_in((double)c.Kp_lo, (double)c.Kp_w, u[2]);
    }
    e.h1 = (T)uniform_in((double)c.h_lo, (double)c.h_w, u[3]);  // :912
    e.h2 = (T)uniform_in((double)c.h_lo, (double)c.h_w, u[4]);
    e.r = (T)uniform_in((double)c.r_lo, (double)c.r_w, u[5]);   // :913
    e.t = 0;
    e.I = (T)0;
}

// reset_from_last_state=True (:904-910): the levels of the last finished episode, or |N(0,1)|*0.1 before the first one
// (last1 is NaN = None).  The two normals are the Box-Muller pair of the uniforms that would have drawn h1, h2.
template <typename T> __device__ __forceinline__ void wt_reset_levels_from_last(WtEnv<T> &e, const double u[6], T last1, T last2) {
    if (last1 == last1) {
        e.h1 = last1;
        e.h2 = last2;
    } else {
        double rad = sqrt(-2.0 * log1p(-u[3])), sn, cs;
        sincospi(2.0 * u[4], &sn, &cs);
        e.h1 = (T)(fabs(rad * cs) * 0.1);
        e.h2 = (T)(fabs(rad * sn) * 0.1);
    }
}

// ============================================================================================== pH
// Mixed precision of the float flavour: the reaction invariant x, the discretised system (A, B) and the three-operation
// table index rint(C x 1e5) are fp64 in BOTH flavours (arrays x, last_x, A, B are double even for *_f32).  y is a staircase
// in x, so an fp32 x (one ulp = 0.008 index units at C x 1e5 = 7.5e4) lands on the neighbouring table entry in 1-2 % of the
// steps; with these four quantities in fp64 the float kernels pick the SAME entry as the double kernels on identical
// (x, A, B, C, action).  Everything else of the float flavour (y, r, I, C = qc_V, reward, table values) is fp32.
template <typename T> struct PhConst {
    T thr, Imax, Ipunish, act_punish;
    double act_low, act_w, sample_t;
    double qww_lo, qww_w, qc_lo, qc_w, x_lo, x_w, r_lo, r_w;
    int reward_type, integrator_mode, max_episode_steps, table_len, from_last;
};

template <typename T> inline PhConst<T> make_ph_const(const pime_ph_config &c) {
    PhConst<T> k;
    k.act_low = c.act_low; k.act_w = c.act_high - c.act_low;
    k.thr = (T)c.distance_threshold; k.Imax = (T)c.integral_max; k.Ipunish = (T)c.integral_punish;
    k.act_punish = (T)c.action_punishment; k.sample_t = c.sample_t;
    k.qww_lo = c.qww_lo; k.qww_w = c.qww_hi - c.qww_lo;
    k.qc_lo = c.qc_lo; k.qc_w = c.qc_hi - c.qc_lo;
    k.x_lo = c.x_lo; k.x_w = c.x_hi - c.x_lo;
    k.r_lo = c.r_lo; k.r_w = c.r_hi - c.r_lo;
    k.reward_type = c.reward_type; k.integrator_mode = c.integrator_mode;
    k.max_episode_steps = c.max_episode_steps; k.table_len = c.table_len; k.from_last = c.reset_from_last_state;
    return k;
}

template <typename T> struct PhEnv {
    double x, A, B;   // fp64 in both flavours (see above)
    T y, r, I, C;
    int t;
};

// The per-env arrays of pime_ph_state with their element types (x, A, B, last_x fp64 in both flavours, see above).
template <typename T> struct PhPtrs {
    double *x, *A, *B, *last_x;
    T *y, *r, *I, *C, *qww, *qc, *ep_return;
    int32_t *t;
    uint32_t *episode;

    PhPtrs() = default;
    explicit PhPtrs(const pime_ph_state &s)
        : x((double *)s.x), A((double *)s.A), B((double *)s.B), last_x((double *)s.last_x), y((T *)s.y), r((T *)s.r),
          I((T *)s.I), C((T *)s.C), qww((T *)s.qww_V), qc((T *)s.qc_V), ep_return((T *)s.ep_return), t(s.t),
          episode(s.episode) {}

    // the arrays of envs [off, ...)
    PhPtrs shifted(int64_t off) const {
        auto adv = [off](auto *q) { return q ? q + off : q; };
        PhPtrs p;
        p.x = adv(x); p.A = adv(A); p.B = adv(B); p.last_x = adv(last_x);
        p.y = adv(y); p.r = adv(r); p.I = adv(I); p.C = adv(C); p.qww = adv(qww); p.qc = adv(qc); p.ep_return = adv(ep_return);
        p.t = adv(t); p.episode = adv(episode);
        return p;
    }

    // what env.step() reads; I only when the plant integrates (the array may be NULL otherwise).  y is an output of the step:
    // with_y also loads it, for a caller that observes the env before stepping it.
    __device__ __forceinline__ void load(PhEnv<T> &e, int64_t i, bool integ, bool with_y = false) const {
        e.x = x[i];
        if (with_y) e.y = y[i];
        e.r = r[i];
        e.I = integ ? I[i] : (T)0;
        load_system(e, i);
        e.t = t[i];
    }
    __device__ __forceinline__ void load_system(PhEnv<T> &e, int64_t i) const { e.A = A[i]; e.B = B[i]; e.C = C[i]; }
    __device__ __forceinline__ void store_system(const PhEnv<T> &e, int64_t i) const { A[i] = e.A; B[i] = e.B; C[i] = e.C; }
    // what env.step() changes
    __device__ __forceinline__ void store_step(const PhEnv<T> &e, int64_t i, bool integ) const {
        x[i] = e.x; y[i] = e.y;
        if (integ) I[i] = e.I;
        t[i] = e.t;
    }
    // the whole PhEnv
    __device__ __forceinline__ void store(const PhEnv<T> &e, int64_t i, bool integ) const {
        x[i] = e.x; y[i] = e.y; r[i] = e.r;
        if (integ) I[i] = e.I;
        store_system(e, i);
        t[i] = e.t;
    }
};

inline int ph_obs_dim(const pime_ph_config &c) { return c.integrator_mode == PIME_PH_NO_INTEGRATOR ? 2 : 3; }

// The argument checks of every pH entry point (step, reset, update_system, rollout, host-buffer rollout), run before
// require_device().  table_len > 1 also keeps ph_lookup's clamp to the last entry inside the table.
inline int validate_ph(const pime_ph_config *cfg, int64_t n, const pime_ph_state *st) {
    PIME_REQUIRE(cfg && st, "null config/state");
    PIME_REQUIRE(n >= 0, "negative n");
    PIME_REQUIRE(st->x && st->y && st->r && st->A && st->B && st->C && st->qww_V && st->qc_V && st->t && st->episode,
                 "null state array");
    PIME_REQUIRE(cfg->integrator_mode >= 0 && cfg->integrator_mode <= 2, "integrator_mode");
    PIME_REQUIRE(cfg->integrator_mode == PIME_PH_NO_INTEGRATOR || st->I, "integrator array missing");
    PIME_REQUIRE(cfg->table_len > 1 && cfg->reward_type >= 0 && cfg->reward_type <= 2, "table_len/reward_type");
    PIME_REQUIRE(!cfg->reset_from_last_state || st->last_x, "reset_from_last_state needs last_x");
    return PIME_OK;
}

// observe_state (ph.py:187-189): first i with MHCl[i] >= around(C*x,5)  ==  rint(C*x*1e5)  (MHCl[i] = i*1e-5;
// equivalence checked on the reference in tests/golden/ph.npz).  The index is computed in fp64 for both table types.
// Returns false when past the table (IndexError).
template <typename T>
__device__ __forceinline__ bool ph_lookup(const T *__restrict__ table, int table_len, double C, double x, T &y) {
    double k = rint(__dmul_rn(__dmul_rn(C, x), 1e5));
    long long i = (long long)k;
    if (i < 0) i = 0;
    if (i >= table_len) { y = table[table_len - 1]; return false; }
    y = __ldg(table + i);
    return true;
}

// PH1DUniformGoalIntegrator.step (ph.py:320-348) / _NoBound.step (:449-478) + TimeLimit.
template <typename T>
__device__ __forceinline__ bool ph_advance(const PhConst<T> &c, const T *__restrict__ table, PhEnv<T> &e, T action, T &reward,
                                           bool &done) {
    using N = Num<T>;
    T a = clampT(action, (T)-1, (T)1);                                                          // :321
    e.t += 1;                                                                                   // :325
    // :155-159  low + (high-low) * ((a - (-1)) / 2); the halving is exact, so * 0.5 rounds like / 2
    const double u = __dadd_rn(c.act_low, __dmul_rn(c.act_w, __dmul_rn(__dsub_rn((double)a, -1.0), 0.5)));
    const double xn = __dadd_rn(__dmul_rn(e.A, e.x), __dmul_rn(e.B, u));                        // :330 (never contracted)
    T y;
    bool ok = ph_lookup(table, c.table_len, (double)e.C, xn, y);                                // :188
    T rew = reward_of<T>(c.reward_type, N::abs(N::sub(y, e.r)), (T)1, c.thr);                   // :334
    rew = N::sub(rew, N::mul(c.act_punish, N::abs((T)u)));                                      // :336
    if (c.integrator_mode != PIME_PH_NO_INTEGRATOR) {
        T integ = N::add(e.I, N::sub(e.r, y));                                                  // :339-340
        rew = N::add(rew, N::mul(-c.Ipunish, N::abs(integ)));                                   // :343
        e.I = c.integrator_mode == PIME_PH_INTEGRATOR ? clampT(integ, -c.Imax, c.Imax) : integ; // :341 / :470
    }
    e.x = xn;
    e.y = y;
    reward = rew;
    done = e.t >= c.max_episode_steps;  // gym TimeLimit (gym_control/__init__.py:6)
    return ok;
}

// update_system (ph.py:114-121): closed form of the ZOH discretisation of qc_V/(s+qww_V).
template <typename T> __device__ __forceinline__ void ph_update_system(double sample_t, T qww, T qc, double &A, double &B, T &C) {
    double a = exp(-(double)qww * sample_t);
    A = a;
    B = (1.0 - a) / (double)qww;
    C = qc;
}

// last_x: the state kept by reset_from_last_state=True (:417-418, :430-431); NaN = None / flag off.
template <typename T>
__device__ __forceinline__ bool ph_reset(const PhConst<T> &c, const T *__restrict__ table, PhEnv<T> &e, T &qww, T &qc,
                                         const double u[6], bool resample, double last_x) {
    if (resample) {  // sample_parameters (:409-410) + update_system (:414)
        qww = (T)uniform_in(c.qww_lo, c.qww_w, u[0]);
        qc = (T)uniform_in(c.qc_lo, c.qc_w, u[1]);
        ph_update_system<T>(c.sample_t, qww, qc, e.A, e.B, e.C);
    }
    e.x = last_x == last_x ? last_x : uniform_in(c.x_lo, c.x_w, u[2]);              // :417-420
    bool ok = ph_lookup(table, c.table_len, (double)e.C, e.x, e.y); // :422
    e.t = 0;
    e.r = (T)uniform_in(c.r_lo, c.r_w, u[3]);           // :424
    e.I = (T)0;
    return ok;
}

}  // namespace pime
