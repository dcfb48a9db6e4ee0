// rollout_ph.cuh -- pH instantiation of the fused rollout.
#pragma once
#include "rollout_impl.cuh"

namespace pime {

// The rollout of n envs whose config and state passed validate_ph; p is the state of these n envs.  sg: the schedule of a
// scheduled launch (fill_seg_params), NULL for a plain one.  TRACK: the scheduled launch with the step response tr.  GAIN:
// that launch with the per-env gains gn (args->priorK_host is NULL).
template <typename T, bool TRACK = false, bool GAIN = false>
int ph_rollout_launch(const pime_ph_config *cfg, const T *table, int64_t n, const PhPtrs<T> &p, const pime_rollout_args *args,
                      void *stream, const SegParams *sg = nullptr, const TrackParams *tr = nullptr,
                      const GainParams *gn = nullptr) {
    RolloutParams rp;
    tc::PackLayout L;
    if (int rc = fill_rollout_params(args, n, ph_obs_dim(*cfg), rp, L, GAIN)) return rc;
    if (int rc = require_device()) return rc;
    if (n == 0) return PIME_OK;
    PIME_REQUIRE(!rp.has_actor || args->actor->kind != PIME_ACTOR_MODULAR || cfg->integrator_mode != PIME_PH_NO_INTEGRATOR,
                 "the modular actor needs the integrator observation");
    return launch_rollout_glue<true, TRACK, GAIN>(PhGlue<T>{make_ph_const<T>(*cfg), table, p}, sg, rp, L, args,
                                                  (cudaStream_t)stream, tr, gn);
}

template <typename T>
int ph_rollout_impl(const pime_ph_config *cfg, const T *table, int64_t n, const pime_ph_state *st, const pime_rollout_args *args,
                    void *stream) {
    if (int rc = validate_ph(cfg, n, st)) return rc;
    PIME_REQUIRE(table, "null table");
    return ph_rollout_launch<T>(cfg, table, n, PhPtrs<T>(*st), args, stream);
}

template <typename T>
int ph_rollout_schedule_impl(const pime_ph_config *cfg, const T *table, int64_t n, const pime_ph_state *st,
                             const pime_rollout_args *args, const pime_schedule *sched, const pime_schedule_ext *ext, void *stream) {
    if (int rc = validate_ph(cfg, n, st)) return rc;
    PIME_REQUIRE(table, "null table");
    SegParams sg;
    if (int rc = fill_seg_params(sched, ext, args, sg)) return rc;
    return ph_rollout_launch<T>(cfg, table, n, PhPtrs<T>(*st), args, stream, &sg);
}

// the scheduled launch with the step response (instantiated in rollout_track_ph_*.cu only)
template <typename T>
int ph_rollout_response_impl(const pime_ph_config *cfg, const T *table, int64_t n, const pime_ph_state *st,
                             const pime_rollout_args *args, const pime_schedule *sched, const pime_schedule_ext *ext,
                             const pime_step_response *resp, void *stream) {
    if (int rc = validate_ph(cfg, n, st)) return rc;
    PIME_REQUIRE(table, "null table");
    SegParams sg;
    if (int rc = fill_seg_params(sched, ext, args, sg)) return rc;
    TrackParams tr;
    if (int rc = fill_track_params(resp, sg, tr)) return rc;
    return ph_rollout_launch<T, true>(cfg, table, n, PhPtrs<T>(*st), args, stream, &sg, &tr);
}

// the scheduled launch with the step response and per-env gains (instantiated in rollout_gain_ph_*.cu only)
template <typename T>
int ph_rollout_gains_impl(const pime_ph_config *cfg, const T *table, int64_t n, const pime_ph_state *st,
                          const pime_rollout_args *args, const pime_schedule *sched, const pime_schedule_ext *ext,
                          const pime_step_response *resp, const pime_schedule_gains *gains, void *stream) {
    if (int rc = validate_ph(cfg, n, st)) return rc;
    PIME_REQUIRE(table, "null table");
    SegParams sg;
    if (int rc = fill_seg_params(sched, ext, args, sg)) return rc;
    TrackParams tr;
    if (int rc = fill_track_params(resp, sg, tr)) return rc;
    GainParams gn;
    if (int rc = fill_gain_params(gains, gn)) return rc;
    return ph_rollout_launch<T, true, true>(cfg, table, n, PhPtrs<T>(*st), args, stream, &sg, &tr, &gn);
}

}  // namespace pime
