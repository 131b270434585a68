/*
 * efa_xray_b200 -- C ABI of the B200 (sm_100a) serial-EnSRF analysis step.
 *
 * Drop-in boundary for the hot path of lmadaus/efa_xray: EnSRF(state, obs, loc='GC').update()
 * (efa_xray/assimilation/ensrf.py:33-151).  The reference has no FFI of its own (it is pure Python
 * on numpy), so these are the entry points a ctypes binding placed under its Python API calls; see
 * INTEGRATION.md for the stub.  Citations below are file:line under /root/reference/efa_xray/.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++ or torch types.
 *   - Every function returns 0 on success or a negative EXB_ERR_* code; exb_last_error() gives the
 *     message for the calling thread.  Nothing throws across the boundary.
 *   - Functions WITHOUT the _host suffix take DEVICE pointers (caller owns the memory, e.g. torch
 *     tensors) and a cudaStream_t passed as void*; they only enqueue work on that stream.
 *   - Functions WITH the _host suffix take HOST pointers, do their own H2D/D2H and synchronise.
 *   - _f64 / _f32 select the storage+arithmetic type T of means and perturbations.  Per-observation
 *     scalars (variance, innovation, gain denominator, beta) and all geometry are always double.
 *   - State matrix layout is the reference's to_vect() layout (state/ensemble.py:110-114):
 *     X[row][member], row = ((var*nt + t)*ny + y)*nx + x, member contiguous.  "nlev" = nvar*nt.
 *   - Observation geometry "obgeo" is an SoA block double[8][nobs] made by exb_obs_prepare:
 *     0..2 unit vector, 3 1/|halfwidth|, 4 haversine-a cutoff, 5 cos(theta), 6 sin(theta), 7 theta,
 *     theta = support radius (2*|halfwidth|) as an angle, clamped to pi.
 *   - Per-observation records "rec" are an SoA block double[8][nobs] written by exb_obs_solve_*:
 *     0 prior_mean, 1 prior_var, 2 post_mean, 3 post_var (NaN if skipped), 4 innovation,
 *     5 1/((Nens-1)*kdenom), 6 beta, 7 assimilated (1.0 / 0.0).
 */
#ifndef EFA_XRAY_B200_H
#define EFA_XRAY_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EXB_OK 0
#define EXB_ERR_ARG (-1)        /* bad argument (null pointer, size out of range)            */
#define EXB_ERR_CUDA (-2)       /* a CUDA runtime call or kernel launch failed               */
#define EXB_ERR_UNSUPPORTED (-3)/* e.g. ensemble size above EXB_MAX_NENS                     */
#define EXB_ERR_NODEVICE (-4)   /* no CUDA device / not an sm_100 device                     */

#define EXB_MAX_NENS 256
#define EXB_LOC_NONE 0          /* loc in (None, False): no localisation, ensrf.py:99        */
#define EXB_LOC_GC 1            /* loc == 'GC': Gaspari-Cohn, observation.py:117-130          */
#define EXB_REC_FIELDS 8
#define EXB_GEO_FIELDS 8

/* ---- library ---------------------------------------------------------------------------- */
int exb_version(void);                       /* 100*major + minor                             */
const char *exb_last_error(void);            /* message of the last failure on this thread    */
int exb_device_check(void);                  /* 0 if the current device can run the kernels   */
int64_t exb_launch_count(void);              /* kernels launched by this library so far        */
/* Work buffers are allocated stream-ordered from a memory pool owned by this library (one per device; other users of
 * cudaMallocAsync are unaffected).  Freed blocks stay cached up to EXB_POOL_KEEP_GB (environment, default 32 GiB);
 * exb_pool_trim returns cached blocks of the current device to the driver, keeping at most keep_bytes. */
int exb_pool_trim(uint64_t keep_bytes);

/* ---- geometry --------------------------------------------------------------------------- */
/* Unit vectors of grid points from lat/lon in degrees; out is SoA double[3][npts].
 * Feeds the on-the-fly great-circle distance that replaces EnsembleState.distance_to_point
 * (state/ensemble.py:254-267). */
int exb_grid_unitvec(const double *lat_deg, const double *lon_deg, int64_t npts, double *grid_u,
                     void *stream);

/* Per-observation geometry (see "obgeo" above) from lat/lon in degrees and the Gaspari-Cohn
 * half-width in km (Observation.localize_radius, observation.py:62; abs() as observation.py:120).
 * With loc_mode == EXB_LOC_NONE every weight is 1 and halfwidth may be NULL. */
int exb_obs_prepare(const double *ob_lat_deg, const double *ob_lon_deg, const double *ob_halfwidth_km,
                    int64_t nobs, int loc_mode, double *obgeo, void *stream);

/* sin(radians(lat)) and cos(radians(lon)) of the obs: the ob-side tables exb_stencil_search* take.  (An exact tie
 * between two grid points of the pseudo-metric is a symmetry of the GRID tables and does not depend on these.) */
int exb_obs_trig(const double *ob_lat_deg, const double *ob_lon_deg, int64_t nobs, double *ob_sinlat, double *ob_coslon,
                 void *stream);

/* Distances (km) and localisation weights from ONE observation to n points given as unit vectors
 * (SoA double[3][n], from exb_grid_unitvec): Observation.distance_to_state / Observation.localize for a
 * state or a list of obs (observation/observation.py:53-87).  Either output may be NULL. */
int exb_localization_weights(const double *u, int64_t n, double ob_lat_deg, double ob_lon_deg,
                             double halfwidth_km, int loc_mode, double *dist_km, double *weights, void *stream);

/* gaspari_cohn(distances, halfwidth), elementwise (observation/observation.py:117-130). */
int exb_gaspari_cohn(const double *dist_km, int64_t n, double halfwidth_km, double *weights, void *stream);

/* ---- forward operator: EnsembleState.nearest_points + interpolate ------------------------ */
/* For every ob the 4 grid points with the smallest pseudo-distance
 *   hypot(sin(lat_g) - sin(lat_ob), cos(lon_g) - cos(lon_ob))        (state/ensemble.py:160-165)
 * ordered by (distance, flat index), then true haversine distances to them and inverse-distance
 * weights (state/ensemble.py:181-200).  sinlat_g / coslon_g / ob_sinlat / ob_coslon are the caller's
 * tables of sin(radians(lat)) and cos(radians(lon)) so that ties fall exactly where they do on the
 * host.  idx4 is int64[nobs][4] (flat y*nx+x), w4 double[nobs][4].
 * n_exact (device int32[1], may be NULL) counts obs with a selected point closer than 1 km, where the
 * reference raises IndexError (state/ensemble.py:195-196); for those obs w4 is 1 at the nearest point
 * and 0 elsewhere (what that branch was meant to do). */
int exb_stencil_search(const double *sinlat_g, const double *coslon_g, const double *lat_g_deg,
                       const double *lon_g_deg, int64_t npts, const double *ob_sinlat,
                       const double *ob_coslon, const double *ob_lat_deg, const double *ob_lon_deg,
                       int64_t nobs, int64_t *idx4, double *w4, int32_t *n_exact, void *stream);

/* Squared pseudo-distance (same roundings as exb_stencil_search) of one observation to all npts grid points: the
 * sort key of nearest_points(npt) for any npt (state/ensemble.py:160-165). */
int exb_pseudo_distance(const double *sinlat_g, const double *coslon_g, int64_t npts, double ob_sinlat,
                        double ob_coslon, double *d2, void *stream);

/* Same search for RECTILINEAR grids (lat a function of y only, lon of x only -- every regular lat-lon
 * grid): the squared pseudo-distance separates into A[y] + B[x], so the search costs O(ny + nx) per ob
 * instead of O(ny * nx).  Tables are per row / per column; results are bit-identical to
 * exb_stencil_search on the expanded 2-D tables. */
int exb_stencil_search_rect(const double *sinlat_y, const double *coslon_x, const double *lat_y_deg,
                            const double *lon_x_deg, int64_t ny, int64_t nx, const double *ob_sinlat,
                            const double *ob_coslon, const double *ob_lat_deg, const double *ob_lon_deg,
                            int64_t nobs, int64_t *idx4, double *w4, int32_t *n_exact, void *stream);

/* Bilinear forward operator (DESIGN.md section 4.8), the opt-in alternative to exb_stencil_search*: for every ob the
 * 4 corners of the grid cell that contains it, in the order (j,i), (j,i+1), (j+1,i), (j+1,i+1), with the weights
 * (1-s)(1-t), s(1-t), (1-s)t, st.  idx4 is int64[nobs][4] (flat y*nx+x), w4 double[nobs][4], as
 * exb_stencil_combine consumes them.  An ob outside the grid gets idx 0 / weight 0 and is counted in n_outside
 * (device int32[1], required; zeroed on the stream first).
 *
 * RECTILINEAR grids: lat_y_deg[ny] strictly monotone (either direction); lon_x_unwrapped[nx] strictly increasing
 * with a span below 360 degrees.  The ob longitude is taken to L0 + ((lon - L0) mod 360), L0 = lon_x_unwrapped[0].
 * periodic = 1 adds the closing cell between column nx-1 and column 0 (right edge L0 + 360).  One thread per ob,
 * binary search on each axis; s and t are linear in degrees. */
int exb_stencil_bilinear_rect(const double *lat_y_deg, const double *lon_x_unwrapped, int64_t ny, int64_t nx,
                              int periodic, const double *ob_lat_deg, const double *ob_lon_deg, int64_t nobs,
                              int64_t *idx4, double *w4, int32_t *n_outside, void *stream);

/* CURVILINEAR grids (2-D lat/lon, e.g. rotated-pole or Lambert-conformal regional grids): the nearest grid point p*
 * by great-circle distance (largest dot product with grid_u[3][ny*nx] of exb_grid_unitvec; ties: lowest flat index),
 * then the cells that have p* as a corner, then the rest of the 4x4-cell block around p*, row-major by lower-left
 * index.  A cell contains the ob when its inverse bilinear coordinates, computed in the (lat, lon) plane with corner
 * longitudes unwrapped to within 180 degrees of the ob's, lie in [-1e-10, 1 + 1e-10]; they are clamped to [0, 1].
 * The grid never wraps; cells that contain a pole are not supported. */
int exb_stencil_bilinear_curv(const double *grid_u, const double *lat_g_deg, const double *lon_g_deg, int64_t ny,
                              int64_t nx, const double *ob_lat_deg, const double *ob_lon_deg, int64_t nobs,
                              int64_t *idx4, double *w4, int32_t *n_outside, void *stream);

/* 8-point stencils of the full forward operator: the 4 space points at the two bracketing time levels with the
 * products of space and time weights (state/ensemble.py:202-237).  row0/row1 = first state row of the ob's variable
 * at its lower / upper time level, tw0/tw1 the time weights.  idx8 are row indices into a shard that holds grid rows
 * [y_begin, y_end) of every level (0, ny: the full state); stencil points outside the band get weight 0, so that the
 * ranks of a latitude-band decomposition produce partial sums that add up to H.x.  diag != 0: idx4 holds indices n
 * into a 1-D point list (states with 1-D lat/lon) and the stencil point is (y, x) = (n, n), as the reference's 1-D
 * branch reads the state (state/ensemble.py:185-187, :226). */
int exb_stencil_combine(const int64_t *idx4, const double *w4, const int64_t *row0, const int64_t *row1,
                        const double *tw0, const double *tw1, int64_t nobs, int64_t ny, int64_t nx, int64_t y_begin,
                        int64_t y_end, int diag, int64_t *idx8, double *w8, void *stream);

/* Y[k][m] = sum_p w[k][p] * X[idx[k][p]][m], p < K (K <= 8): the gather + weighted sums of
 * interpolate (state/ensemble.py:226-237) for all obs at once (compute_ob_priors,
 * assimilation/assimilation.py:36-49).  idx are ROW indices into X. */
int exb_gather_f64(const double *X, int64_t nrows, int nens, const int64_t *idx, const double *w, int K,
                   int64_t nobs, double *Y, void *stream);
int exb_gather_f32(const float *X, int64_t nrows, int nens, const int64_t *idx, const double *w, int K,
                   int64_t nobs, float *Y, void *stream);

/* In place: xm[r] = mean_m X[r][m]; X[r][m] -= xm[r]   (assimilation/assimilation.py:146-147 for the
 * state, :47-48 for the ob priors). */
int exb_split_mean_pert_f64(double *X, double *xm, int64_t nrows, int nens, void *stream);
int exb_split_mean_pert_f32(float *X, float *xm, int64_t nrows, int nens, void *stream);

/* In place multiplicative inflation about the ensemble mean, X = (X - mean)*factor + mean, the float
 * path of inflate_state (assimilation/assimilation.py:62-69).  factor is per row block:
 * rows [i*rows_per_factor, (i+1)*rows_per_factor) use factor[i] (host array of nfactor doubles), which
 * covers both the single float and the per-variable dict (assimilation.py:103-114). */
int exb_inflate_f64(double *X, int64_t nrows, int nens, const double *factor_host, int64_t nfactor,
                    int64_t rows_per_factor, void *stream);
int exb_inflate_f32(float *X, int64_t nrows, int nens, const double *factor_host, int64_t nfactor,
                    int64_t rows_per_factor, void *stream);

/* In place X[r][m] += xm[r]: the recombination in format_posterior_state
 * (assimilation/assimilation.py:168). */
int exb_recombine_f64(double *X, const double *xm, int64_t nrows, int nens, void *stream);
int exb_recombine_f32(float *X, const float *xm, int64_t nrows, int nens, void *stream);

/* ---- posterior relaxation of the state rows after the serial loop (DESIGN.md section 4.6) -------------
 * The rows are those of levels lev < nlev, points [p_begin, p_end) of a shard X[nlev*npts][nens]: rows
 * lev*npts + p, so one call covers a latitude band of every level.  nens >= 2 (EXB_ERR_ARG otherwise).
 * Arithmetic is float64; float storage is rounded once on write.  alpha_dev is a DEVICE array of nlev values. */
/* sigma_out[lev*npts + p] = ensemble standard deviation (ddof = 1) of that row; other entries are untouched. */
int exb_row_spread_f64(const double *X, int64_t nlev, int64_t npts, int64_t p_begin, int64_t p_end, int nens,
                       double *sigma_out, void *stream);
int exb_row_spread_f32(const float *X, int64_t nlev, int64_t npts, int64_t p_begin, int64_t p_end, int nens,
                       double *sigma_out, void *stream);
/* RTPS, relaxation to prior spread: x = m_a + x'_a (1 + alpha (sigma_b - sigma_a) / sigma_a), with sigma_b from
 * exb_row_spread_* on the prior.  A row is not written when alpha = 0, sigma_a = 0, or sigma_a == sigma_b. */
int exb_relax_rtps_f64(double *X, const double *sigma_b, const double *alpha_dev, int64_t nlev, int64_t npts,
                       int64_t p_begin, int64_t p_end, int nens, void *stream);
int exb_relax_rtps_f32(float *X, const double *sigma_b, const double *alpha_dev, int64_t nlev, int64_t npts,
                       int64_t p_begin, int64_t p_end, int nens, void *stream);
/* RTPP, relaxation to prior perturbations: x = m_a + (1 - alpha) x'_a + alpha x'_b, with Xb the prior laid out as X.
 * A row is not written when alpha = 0, sigma_a = 0, or every member equals the prior's. */
int exb_relax_rtpp_f64(double *X, const double *Xb, const double *alpha_dev, int64_t nlev, int64_t npts,
                       int64_t p_begin, int64_t p_end, int nens, void *stream);
int exb_relax_rtpp_f32(float *X, const float *Xb, const double *alpha_dev, int64_t nlev, int64_t npts,
                       int64_t p_begin, int64_t p_end, int nens, void *stream);

/* ---- the serial loop, split in two (SURVEY.md section 0: the obs rows are a closed subsystem) --- */
/* Obs-space serial solve: the rows Nstate..Nstate+Nobs-1 of the reference's augmented state evolved
 * through the whole loop ensrf.py:50-149 in the given (serial) order.
 *   in : Ym[nobs], Yp[nobs][nens]  ob-prior means and perturbations (assimilation.py:149-150)
 *   out: Yp[k][:] = ye_k, the ensemble of ob k as read when ob k is processed (ensrf.py:64);
 *        Ym[k]    = mye_k (ensrf.py:63);  rec = per-ob records (see top).
 * counters (device uint64[2], may be NULL): [0] += number of (ob k, obs row j >= k) pairs with
 * non-zero localisation weight = sum_k |F_o(k)| of SURVEY.md section 8d.
 * Two implementations with identical results up to summation order (environment EXB_OBS_IMPL = dag |
 * persistent; default: dag with localisation unless its dependency graph is more than half dense, persistent
 * otherwise; any other value is EXB_ERR_ARG): see DESIGN.md section 4.2. */
int exb_obs_solve_f64(double *Ym, double *Yp, const double *ob_value, const double *ob_error,
                      const uint8_t *ob_assimilate, const double *obgeo, int64_t nobs, int nens,
                      int loc_mode, double *rec, unsigned long long *counters, void *stream);
int exb_obs_solve_f32(float *Ym, float *Yp, const double *ob_value, const double *ob_error,
                      const uint8_t *ob_assimilate, const double *obgeo, int64_t nobs, int nens,
                      int loc_mode, double *rec, unsigned long long *counters, void *stream);

/* The part of exb_obs_solve_* that depends on the observation geometry only (the predecessor lists of the
 * dependency-driven solve) can be built ahead, on another stream, while the ob priors are still being computed:
 * exb_obs_plan_create only enqueues (packing, counting pass, prefix sum) on ITS stream and returns an opaque plan;
 * exb_obs_plan_finish synchronises that stream, sizes the lists and enqueues the fill pass (it is implied by the
 * first exb_obs_solve_planned_* if not called); exb_obs_solve_planned_* makes its stream wait for the plan; exb_obs_plan_destroy frees the plan (its buffers are
 * released in stream order after the last solve that used it).  A plan fits the (obgeo, ob_assimilate, nobs,
 * loc_mode) it was built from. */
int exb_obs_plan_create(const double *obgeo, const uint8_t *ob_assimilate, int64_t nobs, int loc_mode, void *stream,
                        void **plan);
/* lists of this rank's rows only: blocks of `block` consecutive obs are dealt round-robin to the ranks, rank r owns
 * the obs j with (j / block) % world == r (block = 1: plain round-robin) */
int exb_obs_plan_create_dist(const double *obgeo, const uint8_t *ob_assimilate, int64_t nobs, int loc_mode, int rank,
                             int world, int block, void *stream, void **plan);
int exb_obs_plan_finish(void *plan);
int exb_obs_plan_destroy(void *plan);
int exb_obs_solve_planned_f64(void *plan, double *Ym, double *Yp, const double *ob_value, const double *ob_error,
                              const uint8_t *ob_assimilate, const double *obgeo, int64_t nobs, int nens,
                              int loc_mode, double *rec, unsigned long long *counters, void *stream);
int exb_obs_solve_planned_f32(void *plan, float *Ym, float *Yp, const double *ob_value, const double *ob_error,
                              const uint8_t *ob_assimilate, const double *obgeo, int64_t nobs, int nens,
                              int loc_mode, double *rec, unsigned long long *counters, void *stream);

/* Obs-space solve distributed over the GPUs of one NVLink domain (<= 8): rank `rank` solves the obs rows its plan
 * (exb_obs_plan_create_dist) lists and publishes their records into the record buffers of EVERY rank over peer memory, so that the
 * dependency waits of all ranks resolve locally; the serial chain (longest dependency path) is unchanged, the work per
 * GPU is 1/world.  P_peers[q] / S_peers[q] are pointers, valid on this device, to rank q's buffers (e.g. torch symmetric
 * memory): P nobs*32*MC elements of T (MC = 4 up to 128 members, 8 above), S nobs*2 doubles.  Preconditions: every
 * buffer is filled with 0xFF bytes and the group has synchronised after that; every rank passes identical inputs and
 * its own plan from exb_obs_plan_create_dist (lists must fit one block).  Outputs (Ym, Yp, rec, counters[0]) are written for the rank's own rows
 * only: zero the others and sum over the group.  Returns EXB_ERR_UNSUPPORTED when the plan is dense or multi-block. */
int exb_obs_solve_dist_f64(void *plan, double *Ym, double *Yp, const double *ob_value, const double *ob_error,
                           const uint8_t *ob_assimilate, const double *obgeo, int64_t nobs, int nens, int loc_mode,
                           double *rec, unsigned long long *counters, int rank, int world, void *const *P_peers,
                           void *const *S_peers, void *stream);
int exb_obs_solve_dist_f32(void *plan, float *Ym, float *Yp, const double *ob_value, const double *ob_error,
                           const uint8_t *ob_assimilate, const double *obgeo, int64_t nobs, int nens, int loc_mode,
                           double *rec, unsigned long long *counters, int rank, int world, void *const *P_peers,
                           void *const *S_peers, void *stream);

/* Outlier quality control inside the serial loop (DESIGN.md section 4.7): the entries above with one more argument,
 * ob_threshold, a DEVICE array of one threshold t_k per ob (NULL: no check, exactly the entries above).  An ob k with
 * ob_assimilate[k] != 0 is rejected when |value_k - mye_k| > t_k * sqrt(varye_k + error_k), evaluated in float64 with
 * a correctly rounded sqrt on its prior INSIDE the loop (after obs 0..k-1); t_k = +inf never rejects.  A rejected ob
 * is left out exactly as if its flag were 0: rec 7 = 0.0, post_mean / post_var NaN, no obs row changes; prior_mean,
 * prior_var, innovation and beta are recorded as usual and rec 5 (1/((Nens-1)*kdenom)) is 0, so that a state sweep
 * given these records applies an exact zero update for it.  ob_assimilate itself is not modified: predecessor lists and
 * sweep plans keep being built from it.  The pair counter then counts the pairs the kernels visit, which includes the
 * pairs of a rejected ob with later obs wherever a kernel reaches them before its rejection is known (all of them in
 * the dependency-driven solve, those inside its panel in the persistent solve), so it depends on the implementation. */
int exb_obs_solve_qc_f64(double *Ym, double *Yp, const double *ob_value, const double *ob_error,
                         const uint8_t *ob_assimilate, const double *ob_threshold, const double *obgeo, int64_t nobs,
                         int nens, int loc_mode, double *rec, unsigned long long *counters, void *stream);
int exb_obs_solve_qc_f32(float *Ym, float *Yp, const double *ob_value, const double *ob_error,
                         const uint8_t *ob_assimilate, const double *ob_threshold, const double *obgeo, int64_t nobs,
                         int nens, int loc_mode, double *rec, unsigned long long *counters, void *stream);
int exb_obs_solve_planned_qc_f64(void *plan, double *Ym, double *Yp, const double *ob_value, const double *ob_error,
                                 const uint8_t *ob_assimilate, const double *ob_threshold, const double *obgeo, int64_t nobs,
                                 int nens, int loc_mode, double *rec, unsigned long long *counters, void *stream);
int exb_obs_solve_planned_qc_f32(void *plan, float *Ym, float *Yp, const double *ob_value, const double *ob_error,
                                 const uint8_t *ob_assimilate, const double *ob_threshold, const double *obgeo, int64_t nobs,
                                 int nens, int loc_mode, double *rec, unsigned long long *counters, void *stream);
int exb_obs_solve_dist_qc_f64(void *plan, double *Ym, double *Yp, const double *ob_value, const double *ob_error,
                              const uint8_t *ob_assimilate, const double *ob_threshold, const double *obgeo, int64_t nobs,
                              int nens, int loc_mode, double *rec, unsigned long long *counters, int rank, int world,
                              void *const *P_peers, void *const *S_peers, void *stream);
int exb_obs_solve_dist_qc_f32(void *plan, float *Ym, float *Yp, const double *ob_value, const double *ob_error,
                              const uint8_t *ob_assimilate, const double *ob_threshold, const double *obgeo, int64_t nobs,
                              int nens, int loc_mode, double *rec, unsigned long long *counters, int rank, int world,
                              void *const *P_peers, void *const *S_peers, void *stream);

/* exb_obs_solve_* only enqueues its kernels (the dependency-driven variant synchronises the stream once, to size
 * its work lists, before the solve itself is launched).  Its kernels wait on each other inside the launch; a
 * watchdog (wall clock, EXB_WATCHDOG_S seconds without progress, default 20 + 1e-4 nobs) ends a wait that can never be
 * satisfied (corrupted inputs) instead of hanging the device.  Every solve has its own verdict word; after
 * synchronising the stream, this returns EXB_OK, or EXB_ERR_CUDA if the watchdog fired during the last
 * exb_obs_solve_* issued by the CALLING THREAD (its outputs are then invalid; a state sweep launched from the same
 * thread after such a solve exits without touching the state). */
int exb_obs_solve_async_status(void);

/* State sweep over one latitude-band shard: applies obs [ob_begin, ob_end) in serial order to every
 * state row of the shard -- kcov, localisation, gain, mean update and square-root perturbation update
 * of ensrf.py:95-141 -- using the records of exb_obs_solve_*.
 *   xm[nlev][ny*nx], Xp[nlev][ny*nx][nens]   the shard (ny = rows of this band), updated in place
 *   grid_u double[3][ny*nx]                  unit vectors of the shard's grid points
 *   Yp, rec, obgeo                           as written by exb_obs_solve_* / exb_obs_prepare
 * counters (device uint64[2], may be NULL): [1] += number of (ob, grid point) pairs with non-zero
 * weight = sum_k |F_s(k)| / nlev of SURVEY.md section 8d.
 * Up to 103 members both types run on the two-phase FP64 tensor-core kernel (float32: float32 storage,
 * float64 arithmetic), which synchronises the stream once to size its candidate lists.  Float64 ensembles of 104 to
 * 255 members run on the blocked FP64 tensor-core kernel; float32 ensembles of 104 to 256 members and float64
 * ensembles of 256 run on the vector kernel, whose arithmetic is in the storage type (DESIGN.md section 4.3). */
int exb_state_update_f64(double *xm, double *Xp, int64_t nlev, int64_t ny, int64_t nx, int nens,
                         const double *grid_u, const double *Yp, const double *rec, const double *obgeo,
                         int64_t nobs, int64_t ob_begin, int64_t ob_end, int loc_mode,
                         unsigned long long *counters, void *stream);
int exb_state_update_f32(float *xm, float *Xp, int64_t nlev, int64_t ny, int64_t nx, int nens,
                         const double *grid_u, const float *Yp, const double *rec, const double *obgeo,
                         int64_t nobs, int64_t ob_begin, int64_t ob_end, int loc_mode,
                         unsigned long long *counters, void *stream);

/* Fused form of the state sweep for shards that still hold FULL ensemble values (no exb_split_mean_pert
 * before, no exb_recombine after): grid rows [y_begin, y_end) of the shard X[nlev][ny*nx][nens] are read once,
 * split into mean + perturbations in registers (assimilation/assimilation.py:146-147), updated by obs
 * [ob_begin, ob_end) in serial order (ensrf.py:95-141) and written back as mean + perturbations
 * (assimilation.py:168).  Rows no observation reaches are not written.  Bands of rows can be swept by separate
 * calls (e.g. to overlap the download of finished bands).  Synchronises the stream once (sizing of the candidate
 * lists).  Returns EXB_ERR_UNSUPPORTED for ensembles above 103 members (use the three-call form then).
 * _f32: float32 STORAGE of state and ye rows; the arithmetic is float64 in registers (FP64 tensor cores), so each
 * state value is rounded to float32 exactly once, when the analysis is written back. */
int exb_state_sweep_f64(double *X, int64_t nlev, int64_t ny, int64_t nx, int nens, const double *grid_u,
                        const double *Yp, const double *rec, const double *obgeo, int64_t nobs, int64_t ob_begin,
                        int64_t ob_end, int64_t y_begin, int64_t y_end, int loc_mode, unsigned long long *counters,
                        void *stream);
int exb_state_sweep_f32(float *X, int64_t nlev, int64_t ny, int64_t nx, int nens, const double *grid_u,
                        const float *Yp, const double *rec, const double *obgeo, int64_t nobs, int64_t ob_begin,
                        int64_t ob_end, int64_t y_begin, int64_t y_end, int loc_mode, unsigned long long *counters,
                        void *stream);

/* The part of exb_state_sweep_* that depends on the geometry only (fp32 scan records of the obs, candidate lists per
 * coarse tile of the grid) can be built ahead -- on another stream, while the ob priors and the obs-space solve are
 * computed: exb_sweep_plan_create enqueues it on ITS stream (synchronising that stream once, to size the lists) for grid
 * rows [y_begin, y_end) and obs [ob_begin, ob_end); exb_state_sweep_planned_* makes its stream wait for the plan and
 * sweeps any row sub-range of it; exb_sweep_plan_destroy frees it (in stream order after the last sweep that used it).
 * ob_assimilate must be the flags the obs-space solve is given. */
int exb_sweep_plan_create(const double *grid_u, int64_t nlev, int64_t ny, int64_t nx, const double *obgeo,
                          const uint8_t *ob_assimilate, int64_t nobs, int64_t ob_begin, int64_t ob_end, int64_t y_begin,
                          int64_t y_end, int loc_mode, void *stream, void **plan);
int exb_sweep_plan_destroy(void *plan);
int exb_state_sweep_planned_f64(void *plan, double *X, int64_t nlev, int64_t ny, int64_t nx, int nens, const double *grid_u,
                                const double *Yp, const double *rec, const double *obgeo, int64_t nobs, int64_t ob_begin,
                                int64_t ob_end, int64_t y_begin, int64_t y_end, int loc_mode, unsigned long long *counters,
                                void *stream);
int exb_state_sweep_planned_f32(void *plan, float *X, int64_t nlev, int64_t ny, int64_t nx, int nens, const double *grid_u,
                                const float *Yp, const double *rec, const double *obgeo, int64_t nobs, int64_t ob_begin,
                                int64_t ob_end, int64_t y_begin, int64_t y_end, int loc_mode, unsigned long long *counters,
                                void *stream);

/* Number of grid rows per patch row of exb_state_sweep_f64 for this shape (a small positive integer, not a status
 * code): row ranges whose edges are multiples of it are swept without splitting a patch between two calls. */
int exb_state_sweep_row_granularity(int64_t nlev, int64_t ny, int64_t nx);

/* ---- whole analysis with HOST buffers (one GPU) ------------------------------------------- */
/* EnSRF(...).update() for callers that hold plain host arrays: uploads X, computes the ob priors,
 * runs the serial analysis, downloads the analysis ensemble.  fp64 throughout.  Internally a three-stream pipeline:
 * the state is uploaded and downloaded in latitude bands that overlap the obs-space solve and the sweep of other
 * bands; when X_host is page-locked (cudaHostAlloc / cudaHostRegister / torch pin_memory) and inflation == 1 the ob
 * priors are gathered straight from host memory before the upload starts.
 *   X_host[nlev*ny*nx][nens]    in: prior ensemble; out: posterior ensemble (to_vect layout)
 *   lat/lon_deg[ny*nx]          2-D grid coordinates, row-major (y, x)
 *   ob_row0[nobs]               first state row of the ob's variable at its lower time level,
 *                               ((var*nt + t_lo)*ny*nx); ob_row1 same for the upper time level
 *   ob_tw0/ob_tw1[nobs]         time weights of those two levels (state/ensemble.py:202-224)
 *   ob_diag[4][nobs]            out: prior_mean, prior_var, post_mean, post_var (ensrf.py:66-70,144-147)
 *   inflation                   multiplicative factor applied first (1.0 = none)
 *   stats[8]                    out, may be NULL: [0] sum|F_s| pairs, [1] sum|F_o| pairs, [2] n obs
 *                               within 1 km of a grid point, [3..6] ms on the compute stream: geometry + stencils
 *                               (+ host-memory gather), wait for the state / ob-prior split, obs-space solve +
 *                               sweeps, download left exposed after the last sweep; [7] number of bands */
int exb_ensrf_host_f64(double *X_host, int64_t nlev, int64_t ny, int64_t nx, int nens,
                       const double *lat_deg, const double *lon_deg, int64_t nobs,
                       const double *ob_value, const double *ob_error, const double *ob_lat_deg,
                       const double *ob_lon_deg, const double *ob_halfwidth_km,
                       const uint8_t *ob_assimilate, const int64_t *ob_row0, const int64_t *ob_row1,
                       const double *ob_tw0, const double *ob_tw1, int loc_mode, double inflation,
                       double *ob_diag, double *stats);

/* ---- measurement helpers ----------------------------------------------------------------- */
/* Runs a dependent-free FP64 FMA loop on every SM and returns the achieved FMA rate in TFLOP/s
 * (2 flop per FMA) through *tflops: the roofline denominator of the state sweep, which is bound by
 * the FP64 pipe rather than by HBM (DESIGN.md). */
int exb_measure_fp64_peak(double *tflops, void *stream);

/* Same for the FP64 tensor-core path (mma.sync m8n8k4 f64, SASS DMMA) used by the blocked state sweep. */
int exb_measure_dmma_peak(double *tflops, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* EFA_XRAY_B200_H */
