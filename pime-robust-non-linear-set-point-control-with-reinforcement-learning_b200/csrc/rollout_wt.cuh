// rollout_wt.cuh -- water-tank instantiation of the fused rollout (included by rollout_wt_f32.cu / rollout_wt_f64.cu).
#pragma once
#include "rollout_impl.cuh"

namespace pime {

// The rollout of n envs whose config and state passed validate_wt; p is the state of these n envs.  sg: the schedule of a
// scheduled launch (fill_seg_params), NULL for a plain one.  TRACK: the scheduled launch with the step response tr.  GAIN:
// that launch with the per-env gains gn (args->priorK_host is NULL).
template <typename T, bool TRACK = false, bool GAIN = false>
int wt_rollout_launch(const pime_wt_config *cfg, int64_t n, const WtPtrs<T> &p, const pime_rollout_args *args, void *stream,
                      const SegParams *sg = nullptr, const TrackParams *tr = nullptr, const GainParams *gn = nullptr) {
    RolloutParams rp;
    tc::PackLayout L;
    if (int rc = fill_rollout_params(args, n, wt_obs_dim(*cfg), rp, L, GAIN)) return rc;
    if (int rc = require_device()) return rc;
    if (n == 0) return PIME_OK;
    cudaStream_t s = (cudaStream_t)stream;
    if constexpr (!GAIN) {   // the gain entries reject the stacking observation before this
        if (cfg->obs_mode == PIME_WT_OBS_STACKING) {   // observation history: plain actor only (the modular one needs the integrator)
            PIME_REQUIRE(!rp.has_actor || args->actor->kind == PIME_ACTOR_PLAIN, "the stacking observation goes with the plain actor");
            return launch_rollout_glue<false, TRACK>(WtGlue<T, true>{make_wt_const<T>(*cfg), p}, sg, rp, L, args, s, tr);
        }
    }
    PIME_REQUIRE(!rp.has_actor || args->actor->kind != PIME_ACTOR_MODULAR || cfg->obs_mode == PIME_WT_OBS_INTEGRATOR,
                 "the modular actor needs the integrator observation");
    return launch_rollout_glue<true, TRACK, GAIN>(WtGlue<T, false>{make_wt_const<T>(*cfg), p}, sg, rp, L, args, s, tr, gn);
}

template <typename T>
int wt_rollout_impl(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const pime_rollout_args *args, void *stream) {
    if (int rc = validate_wt(cfg, n, st)) return rc;
    return wt_rollout_launch<T>(cfg, n, WtPtrs<T>(*st), args, stream);
}

template <typename T>
int wt_rollout_schedule_impl(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const pime_rollout_args *args,
                             const pime_schedule *sched, const pime_schedule_ext *ext, void *stream) {
    if (int rc = validate_wt(cfg, n, st)) return rc;
    SegParams sg;
    if (int rc = fill_seg_params(sched, ext, args, sg)) return rc;
    return wt_rollout_launch<T>(cfg, n, WtPtrs<T>(*st), args, stream, &sg);
}

// the scheduled launch with the step response (instantiated in rollout_track_wt_*.cu only)
template <typename T>
int wt_rollout_response_impl(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const pime_rollout_args *args,
                             const pime_schedule *sched, const pime_schedule_ext *ext, const pime_step_response *resp,
                             void *stream) {
    if (int rc = validate_wt(cfg, n, st)) return rc;
    SegParams sg;
    if (int rc = fill_seg_params(sched, ext, args, sg)) return rc;
    TrackParams tr;
    if (int rc = fill_track_params(resp, sg, tr)) return rc;
    return wt_rollout_launch<T, true>(cfg, n, WtPtrs<T>(*st), args, stream, &sg, &tr);
}

// the scheduled launch with the step response and per-env gains (instantiated in rollout_gain_wt_*.cu only)
template <typename T>
int wt_rollout_gains_impl(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const pime_rollout_args *args,
                          const pime_schedule *sched, const pime_schedule_ext *ext, const pime_step_response *resp,
                          const pime_schedule_gains *gains, void *stream) {
    if (int rc = validate_wt(cfg, n, st)) return rc;
    SegParams sg;
    if (int rc = fill_seg_params(sched, ext, args, sg)) return rc;
    TrackParams tr;
    if (int rc = fill_track_params(resp, sg, tr)) return rc;
    GainParams gn;
    if (int rc = fill_gain_params(gains, gn)) return rc;
    PIME_REQUIRE(cfg->obs_mode != PIME_WT_OBS_STACKING, "per-env gains do not take the stacking observation");
    return wt_rollout_launch<T, true, true>(cfg, n, WtPtrs<T>(*st), args, stream, &sg, &tr, &gn);
}

}  // namespace pime
