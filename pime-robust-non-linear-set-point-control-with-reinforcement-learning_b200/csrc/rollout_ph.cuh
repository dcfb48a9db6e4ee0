// rollout_ph.cuh -- pH instantiation of the fused rollout.
#pragma once
#include "rollout_impl.cuh"

namespace pime {

// The rollout of n envs whose config and state passed validate_ph; p is the state of these n envs.  sg: the schedule of a
// scheduled launch (fill_seg_params), NULL for a plain one.
template <typename T>
int ph_rollout_launch(const pime_ph_config *cfg, const T *table, int64_t n, const PhPtrs<T> &p, const pime_rollout_args *args,
                      void *stream, const SegParams *sg = nullptr) {
    RolloutParams rp;
    tc::PackLayout L;
    if (int rc = fill_rollout_params(args, n, ph_obs_dim(*cfg), rp, L)) return rc;
    if (int rc = require_device()) return rc;
    if (n == 0) return PIME_OK;
    PIME_REQUIRE(!rp.has_actor || args->actor->kind != PIME_ACTOR_MODULAR || cfg->integrator_mode != PIME_PH_NO_INTEGRATOR,
                 "the modular actor needs the integrator observation");
    return launch_rollout_glue<true>(PhGlue<T>{make_ph_const<T>(*cfg), table, p}, sg, rp, L, args, (cudaStream_t)stream);
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
                             const pime_rollout_args *args, const pime_schedule *sched, void *stream) {
    if (int rc = validate_ph(cfg, n, st)) return rc;
    PIME_REQUIRE(table, "null table");
    SegParams sg;
    if (int rc = fill_seg_params(sched, args, sg)) return rc;
    return ph_rollout_launch<T>(cfg, table, n, PhPtrs<T>(*st), args, stream, &sg);
}

}  // namespace pime
