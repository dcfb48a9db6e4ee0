// rollout_wt.cuh -- water-tank instantiation of the fused rollout (included by rollout_wt_f32.cu / rollout_wt_f64.cu).
#pragma once
#include "rollout_impl.cuh"

namespace pime {

// The rollout of n envs whose config and state passed validate_wt; p is the state of these n envs.
template <typename T>
int wt_rollout_launch(const pime_wt_config *cfg, int64_t n, const WtPtrs<T> &p, const pime_rollout_args *args, void *stream) {
    RolloutParams rp;
    tc::PackLayout L;
    if (int rc = fill_rollout_params(args, n, wt_obs_dim(*cfg), rp, L)) return rc;
    if (int rc = require_device()) return rc;
    if (n == 0) return PIME_OK;
    cudaStream_t s = (cudaStream_t)stream;
    if (cfg->obs_mode == PIME_WT_OBS_STACKING) {   // observation history: plain actor only (the modular one needs the integrator)
        const WtGlue<T, true> g{make_wt_const<T>(*cfg), p};
        if (!rp.has_actor) return launch_rollout_prior<WtGlue<T, true>>(g, rp, s);
        PIME_REQUIRE(args->actor->kind == PIME_ACTOR_PLAIN, "the stacking observation goes with the plain actor");
        if (args->actor->precision == PIME_PRECISION_FP32) return launch_rollout_fp32<WtGlue<T, true>>(g, L, args->actor_pack, rp, s);
        return launch_rollout_k<WtGlue<T, true>, PIME_ACTOR_PLAIN>(g, &L, args->actor_pack, rp, L.H, s);
    }
    const WtGlue<T, false> g{make_wt_const<T>(*cfg), p};
    if (!rp.has_actor) return launch_rollout_prior<WtGlue<T, false>>(g, rp, s);
    PIME_REQUIRE(args->actor->kind != PIME_ACTOR_MODULAR || cfg->obs_mode == PIME_WT_OBS_INTEGRATOR,
                 "the modular actor needs the integrator observation");
    if (args->actor->precision == PIME_PRECISION_FP32) return launch_rollout_fp32<WtGlue<T, false>>(g, L, args->actor_pack, rp, s);
    if (args->actor->kind == PIME_ACTOR_MODULAR) {
        return launch_rollout_k<WtGlue<T, false>, PIME_ACTOR_MODULAR>(g, &L, args->actor_pack, rp, L.H, s);
    }
    return launch_rollout_k<WtGlue<T, false>, PIME_ACTOR_PLAIN>(g, &L, args->actor_pack, rp, L.H, s);
}

template <typename T>
int wt_rollout_impl(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const pime_rollout_args *args, void *stream) {
    if (int rc = validate_wt(cfg, n, st)) return rc;
    return wt_rollout_launch<T>(cfg, n, WtPtrs<T>(*st), args, stream);
}

}  // namespace pime
