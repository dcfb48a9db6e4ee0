// rollout_ph.cuh -- pH instantiation of the fused rollout.
#pragma once
#include "rollout_impl.cuh"

namespace pime {

// The rollout of n envs whose config and state passed validate_ph; p is the state of these n envs.
template <typename T>
int ph_rollout_launch(const pime_ph_config *cfg, const T *table, int64_t n, const PhPtrs<T> &p, const pime_rollout_args *args,
                      void *stream) {
    RolloutParams rp;
    tc::PackLayout L;
    if (int rc = fill_rollout_params(args, n, ph_obs_dim(*cfg), rp, L)) return rc;
    if (int rc = require_device()) return rc;
    if (n == 0) return PIME_OK;
    const PhGlue<T> g{make_ph_const<T>(*cfg), table, p};
    cudaStream_t s = (cudaStream_t)stream;
    if (!rp.has_actor) return launch_rollout_prior<PhGlue<T>>(g, rp, s);
    PIME_REQUIRE(args->actor->kind != PIME_ACTOR_MODULAR || cfg->integrator_mode != PIME_PH_NO_INTEGRATOR,
                 "the modular actor needs the integrator observation");
    if (args->actor->precision == PIME_PRECISION_FP32) return launch_rollout_fp32<PhGlue<T>>(g, L, args->actor_pack, rp, s);
    if (args->actor->kind == PIME_ACTOR_MODULAR) {
        return launch_rollout_k<PhGlue<T>, PIME_ACTOR_MODULAR>(g, &L, args->actor_pack, rp, L.H, s);
    }
    return launch_rollout_k<PhGlue<T>, PIME_ACTOR_PLAIN>(g, &L, args->actor_pack, rp, L.H, s);
}

template <typename T>
int ph_rollout_impl(const pime_ph_config *cfg, const T *table, int64_t n, const pime_ph_state *st, const pime_rollout_args *args,
                    void *stream) {
    if (int rc = validate_ph(cfg, n, st)) return rc;
    PIME_REQUIRE(table, "null table");
    return ph_rollout_launch<T>(cfg, table, n, PhPtrs<T>(*st), args, stream);
}

}  // namespace pime
