#include "rollout_wt.cuh"
#include "host_pipe.cuh"
using namespace pime;
extern "C" int pime_wt_rollout_f32(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const pime_rollout_args *args,
                                   void *stream) {
    return wt_rollout_impl<float>(cfg, n, st, args, stream);
}
extern "C" int pime_wt_rollout_schedule_f32(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st,
                                            const pime_rollout_args *args, const pime_schedule *sched, void *stream) {
    return wt_rollout_schedule_impl<float>(cfg, n, st, args, sched, stream);
}

// Host-buffer entry: H2D of the per-env state, fused rollout, D2H of ep_return (+ final state), pipelined over env slices
// (host_pipe.cuh).  The stacking observation keeps its frames [3 num_stack][n] with stride n: one slice.
extern "C" int pime_wt_rollout_host_f32(const pime_wt_config *cfg, int64_t n, const pime_wt_state *h, const pime_wt_state *d,
                                        const pime_rollout_args *args, float *ep_return_host, void *stream) {
    PIME_REQUIRE(cfg && h && d && args, "null pointer");
    if (int rc = validate_wt(cfg, n, d)) return rc;
    PIME_REQUIRE(d->ep_return, "device ep_return scratch is required");
    const int S = wt_obs_dim(*cfg);
    {   // the argument block is checked before anything is enqueued; each slice fills its own RolloutParams
        RolloutParams rp;
        tc::PackLayout L;
        if (int rc = fill_rollout_params(args, n, S, rp, L)) return rc;
    }
    if (int rc = require_device()) return rc;
    const WtPtrs<float> hp(*h), dp(*d);
    const HostArr arr[9] = {host_arr(hp.h1, dp.h1, true), host_arr(hp.h2, dp.h2, true), host_arr(hp.r, dp.r, true),
                            host_arr(hp.I, dp.I, true), host_arr(hp.a1, dp.a1, false), host_arr(hp.a2, dp.a2, false),
                            host_arr(hp.Kp, dp.Kp, false), host_arr(hp.t, dp.t, false), host_arr(hp.episode, dp.episode, false)};
    const bool single = cfg->obs_mode == PIME_WT_OBS_STACKING;
    auto launch = [&](int64_t off, int64_t cnt, const pime_rollout_args &a) {
        pime_rollout_args b = a;
        shift_step_buffers(b, off, S, sizeof(float));   // (stacking: one slice, off = 0)
        return wt_rollout_launch<float>(cfg, cnt, dp.shifted(off), &b, stream);
    };
    return host_pipelined_rollout(n, arr, 9, dp.ep_return, ep_return_host, args, (cudaStream_t)stream, launch, single);
}

// the slicing the host-buffer entries would use for n envs on the current device (148 SMs assumed when there is none):
// out2 = {number of slices, envs per slice}.  Host arithmetic only.
extern "C" int pime_host_slice_plan(int64_t n, int32_t single, int64_t *out2) {
    PIME_REQUIRE(out2 && n >= 0, "null output / negative n");
    const int slices = n == 0 ? 1 : host_slice_count(n, single != 0);
    out2[0] = slices;
    out2[1] = host_slice_len(n, slices);
    return PIME_OK;
}

// tests / tuning: force the number of env slices of the host-buffer entries (0 = automatic)
extern "C" int pime_set_host_slices(int32_t slices) {
    PIME_REQUIRE(slices >= 0 && slices <= kMaxSlices, "0 <= slices <= 8");
    host_slices_override() = slices;
    return PIME_OK;
}

#ifdef PIME_PROFILE_WORKER
extern "C" int pime_debug_worker_prof(double *out16) {
    return cudaMemcpyFromSymbol(out16, pime::tc::g_worker_prof, 16 * sizeof(double)) == cudaSuccess ? 0 : -3;
}
#endif
