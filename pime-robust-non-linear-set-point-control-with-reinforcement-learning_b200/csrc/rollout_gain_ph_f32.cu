// pH scheduled rollout with the step response and per-env gains: the Gained kernels, in an object of their own.
#include "rollout_ph.cuh"
using namespace pime;
extern "C" int pime_ph_rollout_schedule_gains_f32(const pime_ph_config *cfg, const float *table, int64_t n,
                                                  const pime_ph_state *st, const pime_rollout_args *args,
                                                  const pime_schedule *sched, const pime_schedule_ext *ext,
                                                  const pime_step_response *resp, const pime_schedule_gains *gains,
                                                  void *stream) {
    return ph_rollout_gains_impl<float>(cfg, table, n, st, args, sched, ext, resp, gains, stream);
}
