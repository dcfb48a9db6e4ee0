#include "rollout_ph.cuh"
using namespace pime;
extern "C" int pime_ph_rollout_f64(const pime_ph_config *cfg, const double *table, int64_t n, const pime_ph_state *st,
                                   const pime_rollout_args *args, void *stream) {
    return ph_rollout_impl<double>(cfg, table, n, st, args, stream);
}
extern "C" int pime_ph_rollout_schedule_f64(const pime_ph_config *cfg, const double *table, int64_t n, const pime_ph_state *st,
                                            const pime_rollout_args *args, const pime_schedule *sched, void *stream) {
    return ph_rollout_schedule_impl<double>(cfg, table, n, st, args, sched, nullptr, stream);
}
extern "C" int pime_ph_rollout_schedule_ext_f64(const pime_ph_config *cfg, const double *table, int64_t n,
                                                const pime_ph_state *st, const pime_rollout_args *args,
                                                const pime_schedule *sched, const pime_schedule_ext *ext, void *stream) {
    PIME_REQUIRE(ext, "null schedule extension");
    return ph_rollout_schedule_impl<double>(cfg, table, n, st, args, sched, ext, stream);
}
