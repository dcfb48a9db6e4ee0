#include "rollout_wt.cuh"
using namespace pime;
extern "C" int pime_wt_rollout_f64(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st, const pime_rollout_args *args,
                                   void *stream) {
    return wt_rollout_impl<double>(cfg, n, st, args, stream);
}
extern "C" int pime_wt_rollout_schedule_f64(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st,
                                            const pime_rollout_args *args, const pime_schedule *sched, void *stream) {
    return wt_rollout_schedule_impl<double>(cfg, n, st, args, sched, nullptr, stream);
}
extern "C" int pime_wt_rollout_schedule_ext_f64(const pime_wt_config *cfg, int64_t n, const pime_wt_state *st,
                                                const pime_rollout_args *args, const pime_schedule *sched,
                                                const pime_schedule_ext *ext, void *stream) {
    PIME_REQUIRE(ext, "null schedule extension");
    return wt_rollout_schedule_impl<double>(cfg, n, st, args, sched, ext, stream);
}
