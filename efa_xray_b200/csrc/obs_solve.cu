// Obs-space serial solve (piece 2 + the obs-row half of piece 4 of the north star): the entry points and the choice
// between the two solvers, each the only one that runs on its inputs.
//
//   obs_solve_dag.cu         dependency-driven solve: the serial chain shrinks to the longest dependency path.  Used
//                            with localisation; it declines (EXB_ERR_UNSUPPORTED) a dependency graph more than half
//                            dense, where walking predecessor lists costs more than the panels save.
//   obs_solve_persistent.cu  one cooperative kernel walking panels of 64 obs.  Used without localisation, where every
//                            ob depends on every earlier one, and for the graphs the dependency-driven solve declines.
//
// EXB_OBS_IMPL = dag | persistent picks one regardless of the inputs (tests compare the two); dag then also runs on a
// dense graph.
#include "common.cuh"
#include <cstring>
#include <cstdlib>

template <typename T>
int exb_obs_solve_dag(T *Ym, T *Yp, const double *ob_value, const double *ob_error, const uint8_t *ob_assim,
                      const double *ob_thr, const double *geo, int64_t nobs, int nens, int loc_mode, double *rec,
                      unsigned long long *counters, cudaStream_t st, bool force, void *plan);
template <typename T>
int exb_obs_solve_persistent(T *Ym, T *Yp, const double *ob_value, const double *ob_error, const uint8_t *ob_assim,
                             const double *ob_thr, const double *geo, int64_t nobs, int nens, int loc_mode, double *rec,
                             unsigned long long *counters, cudaStream_t st);

// ob_thr: outlier threshold per ob (device array), or NULL for no check (DESIGN.md section 4.7)
template <typename T>
static int obs_solve_impl(T *Ym, T *Yp, const double *ob_value, const double *ob_error, const uint8_t *ob_assim,
                          const double *ob_thr, const double *geo, int64_t nobs, int nens, int loc_mode, double *rec,
                          unsigned long long *counters, void *stream, void *plan = nullptr) {
    EXB_REQUIRE(Ym && Yp && ob_value && ob_error && ob_assim && geo && rec, "null pointer");
    EXB_REQUIRE(nobs > 0 && nens >= 2, "need nobs > 0 and nens >= 2");
    EXB_REQUIRE(loc_mode == EXB_LOC_NONE || loc_mode == EXB_LOC_GC, "bad loc_mode");
    if (nens > EXB_MAX_NENS) {
        exb_set_error("exb_obs_solve: nens=%d exceeds EXB_MAX_NENS=%d", nens, EXB_MAX_NENS);
        return EXB_ERR_UNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const char *impl = getenv("EXB_OBS_IMPL");
    const bool dag = impl && strcmp(impl, "dag") == 0;
    if (impl && !dag && strcmp(impl, "persistent") != 0) {
        exb_set_error("exb_obs_solve: EXB_OBS_IMPL=%s; the accepted values are dag and persistent", impl);
        return EXB_ERR_ARG;
    }
    if (dag || (!impl && loc_mode == EXB_LOC_GC)) {
        const int rc = exb_obs_solve_dag<T>(Ym, Yp, ob_value, ob_error, ob_assim, ob_thr, geo, nobs, nens, loc_mode, rec,
                                            counters, st, dag, plan);
        if (rc != EXB_ERR_UNSUPPORTED) return rc;
    }
    return exb_obs_solve_persistent<T>(Ym, Yp, ob_value, ob_error, ob_assim, ob_thr, geo, nobs, nens, loc_mode, rec, counters,
                                       st);
}

extern "C" int exb_obs_solve_f64(double *Ym, double *Yp, const double *ob_value, const double *ob_error,
                                 const uint8_t *ob_assim, const double *obgeo, int64_t nobs, int nens,
                                 int loc_mode, double *rec, unsigned long long *counters, void *stream) {
    return obs_solve_impl<double>(Ym, Yp, ob_value, ob_error, ob_assim, nullptr, obgeo, nobs, nens, loc_mode, rec, counters,
                                  stream);
}
extern "C" int exb_obs_solve_f32(float *Ym, float *Yp, const double *ob_value, const double *ob_error,
                                 const uint8_t *ob_assim, const double *obgeo, int64_t nobs, int nens,
                                 int loc_mode, double *rec, unsigned long long *counters, void *stream) {
    return obs_solve_impl<float>(Ym, Yp, ob_value, ob_error, ob_assim, nullptr, obgeo, nobs, nens, loc_mode, rec, counters,
                                 stream);
}

// Same with a plan built earlier (exb_obs_plan_create), e.g. on a side stream while the ob priors were computed.
extern "C" int exb_obs_solve_planned_f64(void *plan, double *Ym, double *Yp, const double *ob_value, const double *ob_error,
                                         const uint8_t *ob_assim, const double *obgeo, int64_t nobs, int nens, int loc_mode,
                                         double *rec, unsigned long long *counters, void *stream) {
    return obs_solve_impl<double>(Ym, Yp, ob_value, ob_error, ob_assim, nullptr, obgeo, nobs, nens, loc_mode, rec, counters,
                                  stream, plan);
}
extern "C" int exb_obs_solve_planned_f32(void *plan, float *Ym, float *Yp, const double *ob_value, const double *ob_error,
                                         const uint8_t *ob_assim, const double *obgeo, int64_t nobs, int nens, int loc_mode,
                                         double *rec, unsigned long long *counters, void *stream) {
    return obs_solve_impl<float>(Ym, Yp, ob_value, ob_error, ob_assim, nullptr, obgeo, nobs, nens, loc_mode, rec, counters,
                                 stream, plan);
}

// With the outlier check: ob_threshold is a device array of one threshold per ob (NULL: no check).
extern "C" int exb_obs_solve_qc_f64(double *Ym, double *Yp, const double *ob_value, const double *ob_error,
                                    const uint8_t *ob_assim, const double *ob_threshold, const double *obgeo, int64_t nobs,
                                    int nens, int loc_mode, double *rec, unsigned long long *counters, void *stream) {
    return obs_solve_impl<double>(Ym, Yp, ob_value, ob_error, ob_assim, ob_threshold, obgeo, nobs, nens, loc_mode, rec,
                                  counters, stream);
}
extern "C" int exb_obs_solve_qc_f32(float *Ym, float *Yp, const double *ob_value, const double *ob_error,
                                    const uint8_t *ob_assim, const double *ob_threshold, const double *obgeo, int64_t nobs,
                                    int nens, int loc_mode, double *rec, unsigned long long *counters, void *stream) {
    return obs_solve_impl<float>(Ym, Yp, ob_value, ob_error, ob_assim, ob_threshold, obgeo, nobs, nens, loc_mode, rec,
                                 counters, stream);
}
extern "C" int exb_obs_solve_planned_qc_f64(void *plan, double *Ym, double *Yp, const double *ob_value,
                                            const double *ob_error, const uint8_t *ob_assim, const double *ob_threshold,
                                            const double *obgeo, int64_t nobs, int nens, int loc_mode, double *rec,
                                            unsigned long long *counters, void *stream) {
    return obs_solve_impl<double>(Ym, Yp, ob_value, ob_error, ob_assim, ob_threshold, obgeo, nobs, nens, loc_mode, rec,
                                  counters, stream, plan);
}
extern "C" int exb_obs_solve_planned_qc_f32(void *plan, float *Ym, float *Yp, const double *ob_value,
                                            const double *ob_error, const uint8_t *ob_assim, const double *ob_threshold,
                                            const double *obgeo, int64_t nobs, int nens, int loc_mode, double *rec,
                                            unsigned long long *counters, void *stream) {
    return obs_solve_impl<float>(Ym, Yp, ob_value, ob_error, ob_assim, ob_threshold, obgeo, nobs, nens, loc_mode, rec,
                                 counters, stream, plan);
}
