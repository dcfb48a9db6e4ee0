// Water-tank scheduled rollout with the step response: the Tracked kernels, in an object of their own.
#include "rollout_wt.cuh"
using namespace pime;
extern "C" int pime_wt_rollout_schedule_response_f32(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st,
                                                    const pime_rollout_args *args, const pime_schedule *sched,
                                                    const pime_schedule_ext *ext, const pime_step_response *resp,
                                                    void *stream) {
    return wt_rollout_response_impl<float>(cfg, n, st, args, sched, ext, resp, stream);
}
