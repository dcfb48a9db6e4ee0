// rollout_wt.cuh -- water-tank instantiation of the fused rollout (included by rollout_wt_f32.cu / rollout_wt_f64.cu).
#pragma once
#include "rollout_impl.cuh"

namespace pime {

// The rollout of n envs whose config and state passed validate_wt; p is the state of these n envs.  sg: the schedule of a
// scheduled launch (fill_seg_params), NULL for a plain one.
template <typename T>
int wt_rollout_launch(const pime_wt_config *cfg, int64_t n, const WtPtrs<T> &p, const pime_rollout_args *args, void *stream,
                      const SegParams *sg = nullptr) {
    RolloutParams rp;
    tc::PackLayout L;
    if (int rc = fill_rollout_params(args, n, wt_obs_dim(*cfg), rp, L)) return rc;
    if (int rc = require_device()) return rc;
    if (n == 0) return PIME_OK;
    cudaStream_t s = (cudaStream_t)stream;
    if (cfg->obs_mode == PIME_WT_OBS_STACKING) {   // observation history: plain actor only (the modular one needs the integrator)
        PIME_REQUIRE(!rp.has_actor || args->actor->kind == PIME_ACTOR_PLAIN, "the stacking observation goes with the plain actor");
        return launch_rollout_glue<false>(WtGlue<T, true>{make_wt_const<T>(*cfg), p}, sg, rp, L, args, s);
    }
    PIME_REQUIRE(!rp.has_actor || args->actor->kind != PIME_ACTOR_MODULAR || cfg->obs_mode == PIME_WT_OBS_INTEGRATOR,
                 "the modular actor needs the integrator observation");
    return launch_rollout_glue<true>(WtGlue<T, false>{make_wt_const<T>(*cfg), p}, sg, rp, L, args, s);
}

template <typename T>
int wt_rollout_impl(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const pime_rollout_args *args, void *stream) {
    if (int rc = validate_wt(cfg, n, st)) return rc;
    return wt_rollout_launch<T>(cfg, n, WtPtrs<T>(*st), args, stream);
}

template <typename T>
int wt_rollout_schedule_impl(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const pime_rollout_args *args,
                             const pime_schedule *sched, void *stream) {
    if (int rc = validate_wt(cfg, n, st)) return rc;
    SegParams sg;
    if (int rc = fill_seg_params(sched, args, sg)) return rc;
    return wt_rollout_launch<T>(cfg, n, WtPtrs<T>(*st), args, stream, &sg);
}

}  // namespace pime
