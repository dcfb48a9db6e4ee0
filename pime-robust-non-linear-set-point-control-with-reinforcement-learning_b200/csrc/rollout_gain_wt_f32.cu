// Water-tank scheduled rollout with the step response and per-env gains: the Gained kernels, in an object of their own.
#include "rollout_wt.cuh"
using namespace pime;
extern "C" int pime_wt_rollout_schedule_gains_f32(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st,
                                                  const pime_rollout_args *args, const pime_schedule *sched,
                                                  const pime_schedule_ext *ext, const pime_step_response *resp,
                                                  const pime_schedule_gains *gains, void *stream) {
    return wt_rollout_gains_impl<float>(cfg, n, st, args, sched, ext, resp, gains, stream);
}
