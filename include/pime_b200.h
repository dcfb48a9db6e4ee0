/*
 * pime_b200.h -- C ABI of libpime_b200.so: the B200-native (sm_100a) implementation of PIME's batched
 * plant step + P/PI prior + integrated-error observation + residual-actor forward.
 *
 * The reference (ruoqizzz/PIME-Robust-Non-linear-Set-point-control-with-Reinforcement-Learning) is pure
 * Python and has no FFI of its own; the seam it offers is its duck-typed gym / ElegantRL interface.  Each
 * entry point below therefore names the reference symbol (file:line into the reference checkout) whose
 * arithmetic it replaces; INTEGRATION.md shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer unless the name ends in _host;
 *   - per-env data are structure-of-arrays, one array of n elements per field (coalesced);
 *   - *_f32 works on float state (throughput), *_f64 on double state (parity with the numpy reference);
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); calls are asynchronous;
 *   - nothing persistent is allocated by the library; scratch lives in caller-provided buffers;
 *   - return value: 0 on success, negative PIME_E* otherwise; pime_last_error() gives the message
 *     (thread-local).  No exception crosses the ABI and there is no CPU fallback: without a CUDA device
 *     every compute entry point returns PIME_ENODEV.
 */
#ifndef PIME_B200_H_
#define PIME_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PIME_B200_ABI_VERSION 5

enum {
    PIME_OK = 0,
    PIME_EINVAL = -1,   /* bad argument (null pointer, unsupported dimension, ...)                         */
    PIME_ENODEV = -2,   /* no CUDA device / not an sm_100 device                                            */
    PIME_ECUDA = -3,    /* a CUDA runtime call failed; see pime_last_error()                                */
    PIME_ERANGE = -4,   /* pH table lookup ran past the table (reference: IndexError, ph.py:188)            */
    PIME_ESTATE = -5    /* env not reset ("Please reset the env first", nonlinear_watertank.py:794)         */
};

enum { PIME_REWARD_DISTANCE = 0, PIME_REWARD_SQUARE_DISTANCE = 1, PIME_REWARD_SPARSE = 2 };

/* observation layouts of the water-tank family */
enum {
    PIME_WT_OBS_GOAL = 0,       /* [h1,h2,r]            NonLinearWaterTankChangingParamUniformGoal        (:942-1053) */
    PIME_WT_OBS_INTEGRATOR = 1, /* [h1,h2,r,I]          ...ChangingParamUniformGoalIntegrator             (:793-797)  */
    PIME_WT_OBS_STACKING = 2    /* k x [h1,h2,r], oldest first   ...ChangingParamUniformGoalStacking        (:1164-1166) */
};

/* integrator handling of the pH family */
enum {
    PIME_PH_NO_INTEGRATOR = 0,  /* obs [y,r]      PH1DChangingParamUniformGoal            (ph.py:479-485) */
    PIME_PH_INTEGRATOR = 1,     /* obs [y,r,I]    PH1DChangingParamUniformGoalIntegrator  (ph.py:320-348) */
    PIME_PH_INTEGRATOR_NOBOUND = 2 /* unclipped I  ..._NoBound                             (ph.py:449-478) */
};

/* ---------------------------------------------------------------------------------------------------------
 * Water tank.  Constructor arguments of NonLinearWaterTank (nonlinear_watertank.py:84-186) at the values
 * registered in gym_control/__init__.py:29-142.
 * ------------------------------------------------------------------------------------------------------- */
typedef struct pime_wt_config {
    double A1, A2, G;            /* 1, 1, 980                                                     */
    double sample_t;             /* 2.0                                                           */
    int32_t n_discrete;          /* 20 Euler sub-steps per env step (:805-809)                    */
    int32_t max_step;            /* 200; done = (t >= max_step) (:816-821)                        */
    double P_max_action;         /* 10.0; u = a*P/2 + P/2, NOT clipped (:258-260)                 */
    int32_t reward_type;         /* PIME_REWARD_*  (:486-514)                                     */
    int32_t obs_mode;            /* PIME_WT_OBS_*                                                 */
    int32_t num_stack;           /* frames in PIME_WT_OBS_STACKING (1, 4, 10), else ignored       */
    int32_t reset_from_last_state; /* 1: reset() restarts from the levels of the last finished episode
                                    (|N(0,1)|*0.1 before the first one) instead of U(h_lo,h_hi) (:904-912);
                                    needs state.last_h1/last_h2.  0 at every registered id.       */
    double z1;                   /* 1.0                                                           */
    double distance_threshold;   /* 0.05 (sparse reward)                                          */
    double integral_max;         /* 25.0 (:731-733)                                               */
    double integral_punish;      /* 0.0                                                           */
    double noise_scale;          /* 0.01 process noise sigma (:95,:271-272); 0 with --env_zero_noise */
    double a1_lo, a1_hi, a2_lo, a2_hi, Kp_lo, Kp_hi; /* ensemble ranges (sample_parameters :890-894) */
    double h_lo, h_hi;           /* reset: h1,h2 ~ U(0,10) (:912)                                 */
    double r_lo, r_hi;           /* reset: r ~ U(0,10) (:913)                                     */
} pime_wt_config;

/* Per-env state, structure of arrays.  Element type of the void* arrays is float (_f32) or double (_f64). */
typedef struct pime_wt_state {
    void *h1, *h2;        /* tank levels                                                                 */
    void *r;              /* set-point                                                                   */
    void *I;              /* integrated error (PIME_WT_OBS_INTEGRATOR), may be NULL otherwise            */
    void *a1, *a2, *Kp;   /* ensemble parameters of this env (get/reset_changable_parameters :896-900)   */
    int32_t *t;           /* _episode_steps; a negative value marks "not reset yet"                      */
    uint32_t *episode;    /* number of resets so far (RNG tick)                                          */
    void *ep_return;      /* running sum of rewards of the current episode                               */
    void *frames;         /* PIME_WT_OBS_STACKING: [3*num_stack][n] (component-major), else NULL         */
    void *last_h1, *last_h2; /* levels at the last `done` (:819-821); NaN = None.  Required when
                                cfg.reset_from_last_state, else may be NULL                              */
} pime_wt_state;

void pime_wt_default_config(pime_wt_config *cfg); /* registered ...Integrator-SquareDistance-v2 values */

/* reset() -> reset_all() / reset_r()  (nonlinear_watertank.py:902-939, stacking :1168-1208).
 * Draws come from Philox4x32-10 keyed by (seed, env_offset+i, episode[i]); resample_params=1 is
 * if_reset_all=True.  mask (uint8[n], may be NULL = all) selects the envs to reset.
 * obs_out: [S][n] component-major observation after reset, may be NULL. */
int pime_wt_reset_f32(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, uint64_t seed, uint64_t env_offset,
                      int resample_params, const uint8_t *mask, float *obs_out, void *stream);
int pime_wt_reset_f64(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, uint64_t seed, uint64_t env_offset,
                      int resample_params, const uint8_t *mask, double *obs_out, void *stream);

/* env.step(action) for n envs  (NonLinearWaterTankUniformGoalIntegrator.step :800-826, base :274-297,
 * stacking :1122-1149; action_P :258-260; compute_reward :486-514).
 * action[n]; noise1/noise2[n]: the two get_noise() draws (:810-811) -- when NULL and cfg->noise_scale > 0 the
 * kernel draws N(0, noise_scale) from Philox keyed by (seed, env_offset+i, tick); when NULL and noise_scale == 0
 * no noise.  Outputs: state updated in place, obs_out [S][n] (may be NULL), reward[n], done[n]. */
int pime_wt_step_f32(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const float *action,
                     const float *noise1, const float *noise2, uint64_t seed, uint64_t env_offset, uint32_t tick,
                     float *obs_out, float *reward, uint8_t *done, void *stream);
int pime_wt_step_f64(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const double *action,
                     const double *noise1, const double *noise2, uint64_t seed, uint64_t env_offset, uint32_t tick,
                     double *obs_out, double *reward, uint8_t *done, void *stream);

/* ---------------------------------------------------------------------------------------------------------
 * pH neutralisation (gym_control/envs/ph.py).
 * ------------------------------------------------------------------------------------------------------- */
typedef struct pime_ph_config {
    int32_t reward_type;        /* 'square_distance' at the registered ids (gym_control/__init__.py:10)  */
    int32_t integrator_mode;    /* PIME_PH_*                                                             */
    int32_t max_episode_steps;  /* 50, gym TimeLimit (gym_control/__init__.py:6)                         */
    int32_t table_len;          /* len(MHCl) = 100000 (gym_control/__init__.py:12)                       */
    int32_t reset_from_last_state; /* 1: reset() keeps the state of the last finished episode (ph.py:417-420,
                                    :345-346); needs state.last_x.  0 at every registered id.            */
    int32_t reserved0;
    double act_low, act_high;   /* 0.0, 1.5 (ph.py:146-147)                                              */
    double sample_t;            /* 20 (ph.py:40)                                                         */
    double mhcl_step;           /* 1e-5, the only step accepted (the table index is rint(C*x*1e5))      */
    double distance_threshold, integral_max, integral_punish, action_punishment;
    double kw, kchem, ka, MNaOH, MHA, MNH3; /* chemistry (ph.py:31-36); shared by every env              */
    double qww_lo, qww_hi, qc_lo, qc_hi;    /* ensemble ranges (ph.py:357-358)                           */
    double x_lo, x_hi, r_lo, r_hi;          /* reset: x ~ U(0,50), r ~ U(3,11) (ph.py:420-424)           */
} pime_ph_config;

/* Precision of the float flavour: x, last_x, A and B are DOUBLE arrays in both flavours.  y is a staircase in x
 * (100 000-entry table), so the reaction invariant, the discretised system and the three-operation index
 * rint(C*x*1e5) are kept in fp64 -- the *_f32 entry points then pick the same table entry as the *_f64 ones on identical
 * (x, A, B, C, action); every other array of the float flavour (y, r, I, C = qc_V, qww_V, qc_V, ep_return) is float. */
typedef struct pime_ph_state {
    void *x;              /* reaction-invariant state; double[n] in BOTH flavours                        */
    void *y;              /* pH                                                                          */
    void *r, *I;
    void *A, *B, *C;      /* discretised system dsys.A/B/C (update_system ph.py:114-121); A, B: double[n] in
                             BOTH flavours, C: state dtype                                               */
    void *qww_V, *qc_V;   /* ensemble parameters (get_changable_parameters ph.py:268-270)                */
    int32_t *t;
    uint32_t *episode;
    void *ep_return;
    void *last_x;         /* state at the last time-limit step (ph.py:345-346); double[n], NaN = None.  Required
                             when cfg.reset_from_last_state, else may be NULL                            */
} pime_ph_state;

void pime_ph_default_config(pime_ph_config *cfg); /* registered PH1D...Integrator-SqaureDistance-v35 values */

/* PH1D.__init__ titration table (ph.py:72-84).  table_f64[table_len] (required) and table_f32 (may be NULL)
 * are written on the device.  The table is the reference's chain itself (5 abs-Newton steps per grid point,
 * warm-started from the previous one), computed on the host and copied; the call returns when the copies are
 * done.  PIME_EINVAL unless mhcl_step == 1e-5 (every pH entry point checks it: the table index is rint(C*x*1e5)). */
int pime_ph_table_build(const pime_ph_config *cfg, double *table_f64, float *table_f32, void *stream);

/* update_system (ph.py:114-121): A = exp(-qww_V*T), B = (1-A)/qww_V, C = qc_V for every env. */
int pime_ph_update_system_f32(const pime_ph_config *cfg, int64_t n, const pime_ph_state *st, void *stream);
int pime_ph_update_system_f64(const pime_ph_config *cfg, int64_t n, const pime_ph_state *st, void *stream);

/* reset() -> reset_all()/reset_r() (ph.py:412-445).  status (int32[1], device) is set to PIME_ERANGE by a
 * lookup past the table. */
int pime_ph_reset_f32(const pime_ph_config *cfg, const float *table, int64_t n, const pime_ph_state *st, uint64_t seed,
                      uint64_t env_offset, int resample_params, const uint8_t *mask, float *obs_out, int32_t *status,
                      void *stream);
int pime_ph_reset_f64(const pime_ph_config *cfg, const double *table, int64_t n, const pime_ph_state *st, uint64_t seed,
                      uint64_t env_offset, int resample_params, const uint8_t *mask, double *obs_out, int32_t *status,
                      void *stream);

/* env.step(action): PH1DUniformGoalIntegrator.step (ph.py:320-348), _NoBound.step (:449-478), observe_state
 * (:187-189, index = rint(C*x*1e5)), compute_reward (:202-225) and the TimeLimit done flag. */
int pime_ph_step_f32(const pime_ph_config *cfg, const float *table, int64_t n, const pime_ph_state *st,
                     const float *action, float *obs_out, float *reward, uint8_t *done, int32_t *status, void *stream);
int pime_ph_step_f64(const pime_ph_config *cfg, const double *table, int64_t n, const pime_ph_state *st,
                     const double *action, double *obs_out, double *reward, uint8_t *done, int32_t *status, void *stream);

/* get_P_action / get_linear_action (nonlinear_watertank.py:755-759, ph.py:227-231): out[i] = -obs[:,i].K,
 * optionally clipped to [-1,1].  obs is [S][n] component-major; K_host[S] doubles on the HOST. */
int pime_prior_action_f32(int64_t n, int32_t S, const float *obs, const double *K_host, int clip, float *out, void *stream);
int pime_prior_action_f64(int64_t n, int32_t S, const double *obs, const double *K_host, int clip, double *out, void *stream);

/* ---------------------------------------------------------------------------------------------------------
 * Residual actor (elegantrl/net_residual.py) on tcgen05 tensor cores.
 * ------------------------------------------------------------------------------------------------------- */
enum {
    PIME_ACTOR_PLAIN = 0,   /* ActorResidualPPO                  S->H->H->H->1, tanh   (net_residual.py:6-66)    */
    PIME_ACTOR_MODULAR = 1, /* ActorResidualIntegratorModularPPO                        (net_residual.py:138-205) */
    PIME_CRITIC_ADV = 2     /* CriticAdv                         S->H->H->H->1, ReLU   (net.py:274-277)          */
};

/* Arithmetic of the network forward (chosen per call; one packed image serves both):
 *   PIME_PRECISION_TC    throughput: tcgen05 tensor cores, fp16 hidden operands, fp32 accumulation, tanh.approx
 *                        (|a_avg - fp32 torch| <= 4e-3, measured 7e-4 .. 1.6e-3);
 *   PIME_PRECISION_FP32  fidelity: every layer in fp32 on the CUDA cores, tanhf (|a_avg - fp32 torch| <= 2e-5): the
 *                        reference's own arithmetic type, for parity runs and for the critic values of the learner. */
enum { PIME_PRECISION_TC = 0, PIME_PRECISION_FP32 = 1 };

typedef struct pime_actor_config {
    int32_t kind;           /* PIME_ACTOR_* / PIME_CRITIC_ADV                                   */
    int32_t state_dim;      /* S: 3, 4, 12, 30                                                  */
    int32_t mid_dim;        /* H: 32, 64, 128 or 256 (net_dim)                                  */
    int32_t integrator_dim; /* modular: 1                                                       */
    int32_t precision;      /* PIME_PRECISION_*                                                 */
} pime_actor_config;

/* number of fp32 parameters expected in `params` (state_dict order, see INTEGRATION.md) and size in bytes
 * of the packed device image produced by pime_actor_pack. */
int64_t pime_actor_param_count(const pime_actor_config *cfg);
int64_t pime_actor_pack_bytes(const pime_actor_config *cfg);

/* Host-only introspection of the packed image: the list of streamed weight blocks in consumption order, four int32 per
 * block (MMA N, number of K=16 slices, first TMEM column, bytes).  Returns the number of blocks (<= max_blocks are
 * written) or -1 for unsupported dimensions.  Used by the tests to check the kernel's static MMA program against the
 * pack layout without a GPU. */
int32_t pime_actor_block_list(const pime_actor_config *cfg, int32_t *out, int32_t max_blocks);

/* Re-pack fp32 torch-layout parameters (device, state_dict order) into the kernel image: a 4-KB header (the list of
 * weight blocks in consumption order, the fp32 output layer, for the modular actor the fp32 first layer of the
 * integrator branch) followed by the fp16 weight blocks (<= 16 KB each) pre-tiled in the tcgen05 shared-memory operand
 * layout, so that one cp.async.bulk (TMA) copy brings a ready-to-use B operand.  First layers are stored as hi + lo
 * fp16 parts ([W_hi | W_hi | W_lo | b_hi b_lo] against [in_hi | in_lo | in_hi | 1 1]): fp32-grade products on the
 * tensor core; hidden-layer biases as [b_hi b_lo 0 ...] blocks against a constant ones operand.  The fp32 parameters
 * themselves follow the fp16 blocks (the PIME_PRECISION_FP32 forward reads them). */
int pime_actor_pack(const pime_actor_config *cfg, const float *params, void *pack, void *stream);

/* a_avg[i] = net(obs[i,:])  (pre-tanh, pre-prior; get_action_noise net_residual.py:172-175 / :51-53).
 * obs row-major [n][S] fp32. */
int pime_actor_forward(const pime_actor_config *cfg, const void *pack, int64_t n, const float *obs, float *a_avg,
                       void *stream);

/* ---------------------------------------------------------------------------------------------------------
 * Fused rollout: T env steps of plant + prior + observation + actor for n envs in ONE launch, plant state and
 * integrator in registers.  Replaces the loops AgentResidualPPO.explore_env (agent_residual.py:52-69; with
 * deterministic=0) and get_episode_return (run.py:600-619; deterministic=1).
 *
 *   obs32   = float32(obs)                                   elegantrl/env.py:46,72
 *   a_raw   = net(obs32) + eps*exp(a_std_log)                net_residual.py:172-180   (deterministic: eps=0)
 *   action  = tanh(a_raw) + obs32 . priorK                   agent_residual.py:61 / net_residual.py:167-170
 *   env.step(action)                                         as pime_*_step_*
 *   row     = obs32[S], reward*reward_scale, (done?0:gamma), a_raw, eps      agent_residual.py:64-65, replay.py:278
 *
 * The config and state are checked as by the step entries (PIME_EINVAL, also without a device and for n = 0).
 * ------------------------------------------------------------------------------------------------------- */
typedef struct pime_rollout_args {
    const pime_actor_config *actor; /* NULL: prior-only policy (a_avg = 0)                                   */
    const void *actor_pack;
    float a_std_log;                /* act.a_std_log (net_residual.py:162)                                   */
    int32_t deterministic;
    const double *priorK_host;      /* [S] HOST doubles: priorK = -K (agent_residual.py:16-21)               */
    int32_t T;                      /* steps in this launch                                                  */
    int32_t auto_reset;             /* 1: reset (resampling ensemble params) inside the kernel when done     */
    double reward_scale, gamma;
    uint64_t seed, env_offset;
    uint32_t tick0;                 /* RNG tick of the first step (global step counter)                      */
    uint32_t keep_params;           /* 1: the in-kernel reset keeps the ensemble parameters (if_reset_all=False ->
                                       reset_r, nonlinear_watertank.py:935-939 / ph.py:441-445); 0: reset_all          */
    const float *eps;               /* [T][n] exploration noise; NULL: Philox N(0,1) (0 when deterministic)  */
    const void *pnoise1, *pnoise2;  /* [T][n] process noise (state dtype); NULL: Philox or none (see step)   */
    float *buf_state;               /* [T][n][S] float32 replay states, may be NULL                          */
    float *buf_other;               /* [T][n][4] float32 (reward*scale, mask, a_raw, eps), may be NULL       */
    void *env_action;               /* [T][n] action fed to the plant (state dtype), may be NULL (tests)     */
    double *stats;                  /* device double[8], accumulated: sum(ret), sum(ret^2), n_episodes,
                                       sum|r-y_final|, sum(reward), n_steps, -, -; may be NULL               */
    int32_t *status;                /* device int32[1], set to PIME_E* on a device-side fault; may be NULL   */
    int64_t ld;                     /* row length of the per-step buffers (eps, pnoise*, buf_*, env_action: element [t][i]
                                       lives at t * ld + i); 0 = n.  ld > n lets a call work on a slice of a wider env
                                       range whose buffers were allocated for the full range (pointers pre-offset)      */
} pime_rollout_args;

int pime_wt_rollout_f32(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const pime_rollout_args *args, void *stream);
int pime_wt_rollout_f64(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const pime_rollout_args *args, void *stream);
int pime_ph_rollout_f32(const pime_ph_config *cfg, const float *table, int64_t n, const pime_ph_state *st, const pime_rollout_args *args, void *stream);
int pime_ph_rollout_f64(const pime_ph_config *cfg, const double *table, int64_t n, const pime_ph_state *st, const pime_rollout_args *args, void *stream);

/* ---------------------------------------------------------------------------------------------------------
 * Scheduled rollout: the set-point staircase (utils/test.py:70-347, :1369-1407) as one fused launch.  args->T = K L
 * steps run as K segments of L steps; segment k tracks setpoints_host[k].  Each segment begins (right after an env is
 * loaded, and after step k L - 1) with
 *
 *   keep the plant state (h1, h2 / x); reset() keyed as pime_*_reset (episode counter, reset_all when resample_params
 *   is 1, reset_r when 0; reset_from_last_state; t = 0, I = 0, ep_return = 0; stacking frames from the reset's state);
 *   restore the kept state (pH: y = table lookup under the new C, PIME_ERANGE past the table); r = setpoints_host[k].
 *
 * Per env and segment, in fp64, with y the controlled output after a step (h2 / y) and e = r - y:
 *   metrics[0][k][i] = sum of rewards (unscaled)     metrics[1][k][i] = sum of |e| over the segment's steps
 *   metrics[2][k][i] = |e| after the last step       metrics[3][k][i] = max(0, max of d (y - r)),  d = +1 if r >= y at
 *                                                                         the segment begin, else -1
 * The replay rows, env_action, stats and status keep their meaning; args->auto_reset must be 0.  The schedule is checked
 * with the config, state and argument block (PIME_EINVAL, also without a device and for n = 0).
 * ------------------------------------------------------------------------------------------------------- */
#define PIME_MAX_SEGMENTS 16
typedef struct pime_schedule {
    int32_t num_segments;           /* K, 1 .. PIME_MAX_SEGMENTS                                             */
    int32_t segment_steps;          /* L >= 1; args->T must equal K * L                                      */
    int32_t resample_params;        /* segment begin = reset_all (1) / reset_r (0)                           */
    int32_t reserved0;
    const double *setpoints_host;   /* [K] HOST doubles                                                      */
    double *metrics;                /* device double[4][K][n] (ret, iae, final_err, overshoot); may be NULL  */
} pime_schedule;

int pime_wt_rollout_schedule_f32(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const pime_rollout_args *args,
                                 const pime_schedule *sched, void *stream);
int pime_wt_rollout_schedule_f64(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const pime_rollout_args *args,
                                 const pime_schedule *sched, void *stream);
int pime_ph_rollout_schedule_f32(const pime_ph_config *cfg, const float *table, int64_t n, const pime_ph_state *st,
                                 const pime_rollout_args *args, const pime_schedule *sched, void *stream);
int pime_ph_rollout_schedule_f64(const pime_ph_config *cfg, const double *table, int64_t n, const pime_ph_state *st,
                                 const pime_rollout_args *args, const pime_schedule *sched, void *stream);

/* Scheduled rollout with an extension block: per-env set-points and the choice of policy, in the same launch.
 *
 *   setpoints_dev   segment k of env i tracks setpoints_dev[k * n + i] (DEVICE doubles, [K][n]; i is the env's index in
 *                   this call, not env_offset + i); sched->setpoints_host must then be NULL.  NULL: setpoints_host as above.
 *   policy          PIME_POLICY_ACTOR: the policy of the entries above (args->actor's residual policy, or the prior term
 *                   alone when it is NULL).  PIME_POLICY_LINEAR: get_linear_action (utils/test.py:1056-1067), the action
 *                   -(state . K) with K = -priorK_host, computed in the state dtype from the observation before float32
 *                   (h1, h2, r, I / the frame history / y, r, I), summed in k order as pime_prior_action_* sums it,
 *                   clipped to [-1, 1] for the water tank (get_P_action, nonlinear_watertank.py:755-759) and not for pH
 *                   (ph.py:227-231).  Needs args->actor == NULL and args->deterministic != 0.  Replay rows keep their
 *                   layout: float32(obs), (reward*scale, mask, a_raw = 0, eps = 0); env_action holds the clipped action.
 *
 * Besides everything the entries above reject, these reject (PIME_EINVAL, also without a device and for n = 0) a NULL
 * ext, a policy outside PIME_POLICY_*, reserved0 != 0, set-points given as neither or both of setpoints_host /
 * setpoints_dev, and PIME_POLICY_LINEAR with an actor or with deterministic == 0.
 */
#define PIME_POLICY_ACTOR 0
#define PIME_POLICY_LINEAR 1
typedef struct pime_schedule_ext {
    const double *setpoints_dev;    /* DEVICE double[K][n], or NULL: sched->setpoints_host                    */
    int32_t policy;                 /* PIME_POLICY_*                                                         */
    int32_t reserved0;              /* must be 0                                                             */
} pime_schedule_ext;

int pime_wt_rollout_schedule_ext_f32(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const pime_rollout_args *args,
                                     const pime_schedule *sched, const pime_schedule_ext *ext, void *stream);
int pime_wt_rollout_schedule_ext_f64(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const pime_rollout_args *args,
                                     const pime_schedule *sched, const pime_schedule_ext *ext, void *stream);
int pime_ph_rollout_schedule_ext_f32(const pime_ph_config *cfg, const float *table, int64_t n, const pime_ph_state *st,
                                     const pime_rollout_args *args, const pime_schedule *sched, const pime_schedule_ext *ext,
                                     void *stream);
int pime_ph_rollout_schedule_ext_f64(const pime_ph_config *cfg, const double *table, int64_t n, const pime_ph_state *st,
                                     const pime_rollout_args *args, const pime_schedule *sched, const pime_schedule_ext *ext,
                                     void *stream);

/* Scheduled rollout with the step response: the launch of the _ext entries (ext may be NULL: shared set-points and
 * PIME_POLICY_ACTOR), which also stores per env and segment, in fp64, with j = 0 .. L-1 the step inside the segment, y_j
 * the output after step j, e_j = r - y_j, u_j the action fed to the plant at step j (what env_action records), y_b the
 * output at the segment begin (after the restore), D = |r - y_b| and d = +1 if r >= y_b, else -1:
 *
 *   response[0][k][i]  settle       0 if |e_j| <= settle_band * D for every j, else 1 + the largest j with |e_j| > that
 *                                   band (L: not settled at the segment end)
 *   response[1][k][i]  rise         1 + the smallest j with d (y_j - y_b) >= 0.9 D; -1 if no step reaches it; 0 if D = 0
 *   response[2][k][i]  effort       sum over j = 1 .. L-1 of |u_j - u_{j-1}|, in j order
 *   response[3][k][i]  peak_action  max over j of |u_j|
 *
 * Dead tail rows store nothing.  Besides everything the _ext entries reject, these reject (PIME_EINVAL, also without a
 * device and for n = 0) a NULL resp or response, settle_band outside (0, 1) or NaN, and segment_steps > 65535.
 */
typedef struct pime_step_response {
    double *response;               /* device double[4][K][n] (settle, rise, effort, peak_action)             */
    double settle_band;             /* settling band relative to D, in (0, 1); 0.02 is the usual choice       */
} pime_step_response;

int pime_wt_rollout_schedule_response_f32(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st,
                                          const pime_rollout_args *args, const pime_schedule *sched,
                                          const pime_schedule_ext *ext, const pime_step_response *resp, void *stream);
int pime_wt_rollout_schedule_response_f64(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st,
                                          const pime_rollout_args *args, const pime_schedule *sched,
                                          const pime_schedule_ext *ext, const pime_step_response *resp, void *stream);
int pime_ph_rollout_schedule_response_f32(const pime_ph_config *cfg, const float *table, int64_t n, const pime_ph_state *st,
                                          const pime_rollout_args *args, const pime_schedule *sched,
                                          const pime_schedule_ext *ext, const pime_step_response *resp, void *stream);
int pime_ph_rollout_schedule_response_f64(const pime_ph_config *cfg, const double *table, int64_t n, const pime_ph_state *st,
                                          const pime_rollout_args *args, const pime_schedule *sched,
                                          const pime_schedule_ext *ext, const pime_step_response *resp, void *stream);

/* Scheduled rollout with the step response and per-env controller gains: the launch of the _response entries (ext may be
 * NULL), with env i's priorK (= -K, S entries, S the observation dimension) taken from column i of a DEVICE matrix instead
 * of args->priorK_host, for the agent's prior term and for the linear policy:
 *
 *   priorK of env i  =  priorK_dev[k * n + i],  k = 0 .. S-1   (i is the env's index in this call, not env_offset + i)
 *
 * Each env computes exactly what the _response entries compute from priorK_host equal to its column: a launch whose
 * columns are all equal is bit-identical to that one.  A gain x plant robustness map is one launch with one column per
 * (gain, plant) pair.  Besides everything the _response entries reject, these reject (PIME_EINVAL, also without a device
 * and for n = 0) a NULL gains or priorK_dev, args->priorK_host != NULL (the gains are given exactly once), and the water
 * tank's PIME_WT_OBS_STACKING (its K spans the frame history, which no gain map tunes).
 */
typedef struct pime_schedule_gains {
    const double *priorK_dev;       /* DEVICE double[S][n]: env i's priorK (= -K) is priorK_dev[k * n + i]    */
} pime_schedule_gains;

int pime_wt_rollout_schedule_gains_f32(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st,
                                       const pime_rollout_args *args, const pime_schedule *sched, const pime_schedule_ext *ext,
                                       const pime_step_response *resp, const pime_schedule_gains *gains, void *stream);
int pime_wt_rollout_schedule_gains_f64(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st,
                                       const pime_rollout_args *args, const pime_schedule *sched, const pime_schedule_ext *ext,
                                       const pime_step_response *resp, const pime_schedule_gains *gains, void *stream);
int pime_ph_rollout_schedule_gains_f32(const pime_ph_config *cfg, const float *table, int64_t n, const pime_ph_state *st,
                                       const pime_rollout_args *args, const pime_schedule *sched, const pime_schedule_ext *ext,
                                       const pime_step_response *resp, const pime_schedule_gains *gains, void *stream);
int pime_ph_rollout_schedule_gains_f64(const pime_ph_config *cfg, const double *table, int64_t n, const pime_ph_state *st,
                                       const pime_rollout_args *args, const pime_schedule *sched, const pime_schedule_ext *ext,
                                       const pime_step_response *resp, const pime_schedule_gains *gains, void *stream);

/* Per-env GAE / reward-to-go reverse scan over a time-major replay (AgentPPO.compute_reward_gae
 * agent.py:685-708 without the final normalisation): reward, mask, value are [T][n] with element stride
 * `stride` floats (4 for buf_other columns, 1 for dense); r_sum, adv are dense [T][n]. */
int pime_gae_scan(int64_t n, int32_t T, const float *reward, const float *mask, int32_t stride, const float *value,
                  float lambda_gae, float *r_sum, float *adv, void *stream);

/* Episode statistics (Evaluator.get_r_avg_std_s_avg_std run.py:593-597): stats[0..2] += sum, sum of squares,
 * count of ep_return[n] (warp-shuffle + one atomic per block). */
int pime_reduce_episode_stats_f32(int64_t n, const float *ep_return, double *stats, void *stream);
int pime_reduce_episode_stats_f64(int64_t n, const double *ep_return, double *stats, void *stream);

/* ---------------------------------------------------------------------------------------------------------
 * Host-buffer convenience entry (what an unmodified gym-style caller with numpy arrays uses): copies the
 * per-env state from pinned/pageable HOST arrays to the device scratch `st_dev`, runs the fused rollout and
 * copies ep_return[n] (and the final state) back.  All host<->device traffic is inside the call, which returns after
 * the last byte has arrived.  Large env ranges (>= 8 waves of SM count x 256 envs, no stacking frames) are cut into up to 8 slices of whole waves and pipelined: the copy-in of slice k+1 and the copy-out
 * of slice k-1 run on two internal streams under the rollout of slice k.  An env's random stream is keyed by its global
 * id, so the result does not depend on the slicing; pime_set_host_slices(c) forces c slices of whole 256-env tiles
 * (tests / tuning; 0 = automatic).
 * ------------------------------------------------------------------------------------------------------- */
int pime_wt_rollout_host_f32(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st_host, const pime_wt_state *st_dev,
                             const pime_rollout_args *args, float *ep_return_host, void *stream);
/* pH flavour: st_host holds x, A, B as double[n] and y, r, I, C, qww_V, qc_V as float[n] (t, episode int32 / uint32);
 * x, y, r, I of the final state are copied back.  `table` is the DEVICE table of pime_ph_table_build. */
int pime_ph_rollout_host_f32(const pime_ph_config *cfg, const float *table, int64_t n, const pime_ph_state *st_host,
                             const pime_ph_state *st_dev, const pime_rollout_args *args, float *ep_return_host, void *stream);
int pime_set_host_slices(int32_t slices);
int pime_host_slice_plan(int64_t n, int32_t single, int64_t *out2); /* {slices, envs per slice} the entries would use */

/* ---------------------------------------------------------------------------------------------------------
 * PPO learner: one minibatch step of AgentPPO.update_net (elegantrl/agent.py:635-658) on the GPU-resident replay
 * in two launches (rows kernel: gather + actor / critic forward + objectives + data gradients; weight-gradient
 * kernel with the Adam update fused in).  fp32 throughout, torch.optim.Adam arithmetic.
 *
 *   new_logprob = compute_logprob(state, action)                       net_residual.py:62-66
 *   ratio       = exp(new_logprob - logprob)
 *   obj_actor   = -mean(min(adv*ratio, adv*clamp(ratio, 1-clip, 1+clip))) + lambda_entropy * mean(exp(lp)*lp)
 *   obj_critic  = SmoothL1(critic(state), r_sum)
 *   obj_united  = obj_actor + obj_critic / (r_sum.std() + 1e-5);  Adam step on actor, critic and a_std_log
 *
 * theta = [actor parameters | pad | critic parameters | a_std_log], each net in state_dict order (pime_actor_param_count
 * floats; the critic is CriticAdv with the actor's S and H; its offset, a multiple of 4 floats, the offset of
 * a_std_log and the total come from pime_ppo_theta_layout); theta_t holds every weight matrix transposed
 * (pime_ppo_transpose; kept up to date by the step).  state: device int32[1024], zero-initialised, owned by the
 * library between steps (Adam step count, a ticket, the a_std_log and output-layer gradient accumulators).  loss_ring: device
 * float[ring_len][4], zero-initialised; step t (0-based count before the call) adds the means of (obj_united,
 * obj_actor, obj_critic, obj_entropy) to row t % ring_len and clears the next row.
 * ------------------------------------------------------------------------------------------------------- */
typedef struct pime_ppo_args {
    const pime_actor_config *actor;   /* PIME_ACTOR_PLAIN or PIME_ACTOR_MODULAR                               */
    float *theta, *theta_t;           /* [pime_ppo_theta_count]                                                */
    float *adam_m, *adam_v;           /* Adam moments, same layout; may be NULL when grad_out is given         */
    float *grad_out;                  /* not NULL: write the gradient of obj_united here and leave theta alone */
    const float *buf_state;           /* [buf_len][S]                                                          */
    const float *buf_action, *buf_r_sum, *buf_logprob, *buf_advantage; /* [buf_len]                            */
    const int64_t *idx;               /* [batch] rows of this minibatch (torch.randint, agent.py:636)          */
    int32_t batch;
    float ratio_clip, lambda_entropy;
    float lr, beta1, beta2, eps;      /* torch.optim.Adam                                                      */
    int32_t *state;
    float *work;                      /* scratch: pime_ppo_work_floats(actor, batch) floats                    */
    float *loss_ring;
    int32_t ring_len;
} pime_ppo_args;

int64_t pime_ppo_theta_count(const pime_actor_config *actor);
int pime_ppo_theta_layout(const pime_actor_config *actor, int64_t *out3); /* critic offset, a_std_log offset, total */
int64_t pime_ppo_work_floats(const pime_actor_config *actor, int32_t batch);
int pime_ppo_transpose(const pime_actor_config *actor, const float *theta, float *theta_t, void *stream);
int pime_ppo_step(const pime_ppo_args *args, void *stream);
/* Data-parallel training (BASELINE configs[4]): every rank runs pime_ppo_step with grad_out set (the gradient of obj_united
 * over ITS minibatch rows, flat, theta's layout), the caller all-reduces that buffer (NCCL), then this entry applies
 * torch.optim.Adam's arithmetic to theta / theta_t / the moments with grad * scale (scale = 1 / world size for the mean).
 * It must follow the pime_ppo_step of the same step on the same stream: the step count and the bias corrections are
 * the ones that call left in `state`. */
int pime_ppo_apply_grad(const pime_ppo_args *args, const float *grad, float scale, void *stream);

/* Large minibatches (BASELINE configs[4]: 131 072 rows) on the tcgen05 tensor cores (csrc/learner_tc.cu): the batch is cut
 * into 128-row tiles, every layer of the forward pass, of the data-gradient chain and every weight gradient is a GEMM whose
 * operands are fp16 hi + lo pairs (three MMAs per product: fp32-grade sums) streamed by TMA, accumulated in TMEM.
 *   pime_ppo_grad_tc     gradient of obj_united over the rows args->idx into grad[pime_ppo_theta_count] (theta's layout;
 *                        zeroed first), the loss-ring row and the Adam bias corrections of the step; theta is NOT touched.
 *                        work_tc: pime_ppo_tc_work_bytes(actor, batch) bytes of device scratch, 256-byte aligned.
 *                        mid_dim 128 or 256, plain or modular actor, 2 <= batch <= 2^20.  args->theta_t / adam_* / work unused.
 *   pime_ppo_apply_grad  (above) applies Adam; all-reduce grad in between when the job is data parallel.
 *   pime_ppo_close_step  increments the step count and clears the next loss-ring row (the small-batch pime_ppo_step does
 *                        this itself); call it last.
 *   pime_ppo_tc_layout   byte offset / unit count of the intermediate matrices inside work_tc (X, activations, pre-activation
 *                        gradients; 17 pairs) -- lets the tests compare every stage with torch. */
int64_t pime_ppo_tc_work_bytes(const pime_actor_config *actor, int32_t batch);
int pime_ppo_tc_layout(const pime_actor_config *actor, int32_t batch, int64_t *out34);
int pime_ppo_grad_tc(const pime_ppo_args *args, void *work_tc, float *grad, void *stream);
int pime_ppo_close_step(const pime_ppo_args *args, void *stream);

/* misc */
int pime_abi_version(void);
const char *pime_last_error(void);
int pime_device_info(int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor); /* PIME_ENODEV without a GPU */
/* Philox4x32-10 block for (seed, index, tick, stream) computed on the device -> out_host[4]; used by tests to
 * check the device stream against the oracle bit for bit. */
int pime_philox_probe(uint64_t seed, uint64_t index, uint32_t tick, uint32_t stream_id, uint32_t *out_host);

#ifdef __cplusplus
}
#endif
#endif /* PIME_B200_H_ */
