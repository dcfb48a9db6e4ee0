#include "rollout_ph.cuh"
#include "host_pipe.cuh"
using namespace pime;
extern "C" int pime_ph_rollout_f32(const pime_ph_config *cfg, const float *table, int64_t n, const pime_ph_state *st,
                                   const pime_rollout_args *args, void *stream) {
    return ph_rollout_impl<float>(cfg, table, n, st, args, stream);
}
extern "C" int pime_ph_rollout_schedule_f32(const pime_ph_config *cfg, const float *table, int64_t n, const pime_ph_state *st,
                                            const pime_rollout_args *args, const pime_schedule *sched, void *stream) {
    return ph_rollout_schedule_impl<float>(cfg, table, n, st, args, sched, nullptr, stream);
}
extern "C" int pime_ph_rollout_schedule_ext_f32(const pime_ph_config *cfg, const float *table, int64_t n,
                                                const pime_ph_state *st, const pime_rollout_args *args,
                                                const pime_schedule *sched, const pime_schedule_ext *ext, void *stream) {
    PIME_REQUIRE(ext, "null schedule extension");
    return ph_rollout_schedule_impl<float>(cfg, table, n, st, args, sched, ext, stream);
}

// Host-buffer entry (configs[3] end to end): H2D of the per-env state, fused rollout, D2H of ep_return + the final state,
// pipelined over env slices (host_pipe.cuh).  x, A, B are double arrays in the float flavour (include/pime_b200.h),
// everything else float / int32.
extern "C" int pime_ph_rollout_host_f32(const pime_ph_config *cfg, const float *table, int64_t n, const pime_ph_state *h,
                                        const pime_ph_state *d, const pime_rollout_args *args, float *ep_return_host, void *stream) {
    PIME_REQUIRE(cfg && table && h && d && args, "null pointer");
    if (int rc = validate_ph(cfg, n, d)) return rc;
    PIME_REQUIRE(d->ep_return, "device ep_return scratch is required");
    const int S = ph_obs_dim(*cfg);
    {   // the argument block is checked before anything is enqueued; each slice fills its own RolloutParams
        RolloutParams rp;
        tc::PackLayout L;
        if (int rc = fill_rollout_params(args, n, S, rp, L)) return rc;
    }
    if (int rc = require_device()) return rc;
    const PhPtrs<float> hp(*h), dp(*d);
    const HostArr arr[11] = {host_arr(hp.x, dp.x, true), host_arr(hp.y, dp.y, true), host_arr(hp.r, dp.r, true),
                             host_arr(hp.I, dp.I, true), host_arr(hp.A, dp.A, false), host_arr(hp.B, dp.B, false),
                             host_arr(hp.C, dp.C, false), host_arr(hp.qww, dp.qww, false), host_arr(hp.qc, dp.qc, false),
                             host_arr(hp.t, dp.t, false), host_arr(hp.episode, dp.episode, false)};
    auto launch = [&](int64_t off, int64_t cnt, const pime_rollout_args &a) {
        pime_rollout_args b = a;
        shift_step_buffers(b, off, S, sizeof(float));
        return ph_rollout_launch<float>(cfg, table, cnt, dp.shifted(off), &b, stream);
    };
    return host_pipelined_rollout(n, arr, 11, dp.ep_return, ep_return_host, args, (cudaStream_t)stream, launch, false);
}

#ifdef PIME_PROFILE_WORKER
extern "C" int pime_debug_worker_prof_ph(double *out16) {
    return cudaMemcpyFromSymbol(out16, pime::tc::g_worker_prof, 16 * sizeof(double)) == cudaSuccess ? 0 : -3;
}
#endif
