// Shared device/host helpers for the efa_xray_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include "../../include/efa_xray_b200.h"

#define EXB_R_EARTH 6371.0            // km; state/ensemble.py:259, observation/observation.py:138
#define EXB_DEG2RAD 0.017453292519943295

// obgeo rows
#define GEO_UX 0
#define GEO_UY 1
#define GEO_UZ 2
#define GEO_INVHW 3
#define GEO_AMAX 4
#define GEO_COST 5
#define GEO_SINT 6
#define GEO_THETA 7
// rec rows
#define REC_PRIOR_MEAN 0
#define REC_PRIOR_VAR 1
#define REC_POST_MEAN 2
#define REC_POST_VAR 3
#define REC_INNOV 4
#define REC_C1 5
#define REC_BETA 6
#define REC_ASSIM 7

void exb_set_error(const char *fmt, ...);
int exb_check_launch(const char *what);
void exb_count_launches(int64_t n);   // bookkeeping for exb_launch_count()

// Stream-ordered work buffers come from a memory pool OWNED by this library (one per device), not from the device's
// default pool: freed blocks stay cached up to EXB_POOL_KEEP_GB (default 32 GiB; exb_pool_trim releases them) without
// changing the behaviour of anybody else's cudaMallocAsync.  Free with cudaFreeAsync.
cudaError_t exb_malloc_async(void **p, size_t bytes, cudaStream_t st);
template <typename U> static inline cudaError_t exb_malloc_async(U **p, size_t bytes, cudaStream_t st) {
    return exb_malloc_async(reinterpret_cast<void **>(p), bytes, st);
}
// Small page-locked, device-mapped words for results a kernel hands to the host without a copy (list totals,
// watchdog verdicts).  Every call gets its own: nothing is shared between concurrent analyses.
struct ExbHostWords { volatile long long *host; long long *dev; int slot; };      // 8 words
int exb_host_words_acquire(ExbHostWords *w);
void exb_host_words_release(const ExbHostWords &w);
// Watchdog word of an obs-space solve: a fresh slot per solve (ring of 1024), remembered per host thread so that
// exb_obs_solve_async_status() and the state sweep launched next from the same thread see THEIR solve's verdict.
int exb_status_slot_next(int **host, int **dev);
const int *exb_status_slot_last_dev();
// Page-locked staging buffers (cached; cudaHostAlloc is too slow to do per call)
int exb_pinned_acquire(size_t bytes, void **p);
void exb_pinned_release(void *p);

#define EXB_REQUIRE(cond, msg)                         \
    do {                                               \
        if (!(cond)) {                                 \
            exb_set_error("%s: %s", __func__, msg);    \
            return EXB_ERR_ARG;                        \
        }                                              \
    } while (0)

#define EXB_CUDA(call)                                                              \
    do {                                                                            \
        cudaError_t e__ = (call);                                                   \
        if (e__ != cudaSuccess) {                                                   \
            exb_set_error("%s: %s -> %s", __func__, #call, cudaGetErrorString(e__)); \
            return EXB_ERR_CUDA;                                                    \
        }                                                                           \
    } while (0)

// Haversine 'a' from two unit vectors: a = sin^2(d/2) = |u - v|^2 / 4.  Mathematically the same
// quantity as state/ensemble.py:264 and observation.py:144; computed from differences so it keeps
// full relative accuracy for nearby points.
__device__ __forceinline__ double hav_a(double ux, double uy, double uz, double vx, double vy, double vz) {
    const double dx = ux - vx, dy = uy - vy, dz = uz - vz;
    return 0.25 * (dx * dx + dy * dy + dz * dz);
}

// Great-circle angle c = 2*atan2(sqrt(a), sqrt(1-a))   (state/ensemble.py:266).
__device__ __forceinline__ double angle_from_a(double a) {
    a = fmin(fmax(a, 0.0), 1.0);
    if (a < 0.5) return 2.0 * asin(sqrt(a));            // same function, cheaper and exact to 1 ulp here
    return 2.0 * atan2(sqrt(a), sqrt(1.0 - a));
}

// Gaspari-Cohn weight of r = distance / |halfwidth|   (observation/observation.py:120-130).
__device__ __forceinline__ double gaspari_cohn_r(double r) {
    if (r <= 1.0) return ((((-0.25 * r + 0.5) * r + 0.625) * r - 5.0 / 3.0) * (r * r) + 1.0);
    if (r < 2.0)
        return (((((r / 12.0 - 0.5) * r + 0.625) * r + 5.0 / 3.0) * r - 5.0) * r + 4.0 - 2.0 / (3.0 * r));
    return 0.0;
}

// Localisation weight of a pair from its haversine a.  inv_hw = 1/|halfwidth| (0 when localisation
// is off, which makes r = 0 and the weight exactly 1); a_max is the value of a at r = 2.
__device__ __forceinline__ double loc_weight(double a, double inv_hw, double a_max) {
    if (a >= a_max) return 0.0;
    const double r = EXB_R_EARTH * angle_from_a(a) * inv_hw;
    return gaspari_cohn_r(r);
}

// ---- branch-free localisation weight for supports up to 5000 km -------------------------------------------
// Same function as loc_weight, written without data-dependent branches or libm slow paths so that several
// independent evaluations interleave in one thread (the libm asin/sqrt/division chain is latency-bound).
// Valid for a_max <= EXB_FAST_AMAX (support angle <= 45.6 degrees, 5070 km); callers fall back to loc_weight
// otherwise.  asin(sqrt(a)) = sqrt(a) * Q(a), Q(a) = sum_n c_n a^n, c_n = (2n)! / (4^n n!^2 (2n+1)); 20 terms
// leave a remainder below 1e-19 at a = 0.15.  Reciprocal and reciprocal square root start from the fp32
// special-function unit and take two Newton steps (relative error ~1e-28 before rounding).
#define EXB_FAST_AMAX 0.15
__device__ __forceinline__ double exb_asin_sqrt_over_sqrt(double a) {
    // Horner on two interleaved halves (even/odd powers) to halve the dependent chain
    const double a2 = a * a;
    double pe = 0.0035692053938259347, po = 0.003297059503473485;   // c18, c19
    pe = fma(pe, a2, 0.004240907093679363); po = fma(po, a2, 0.003880964558837669);   // c16, c17
    pe = fma(pe, a2, 0.005153309682319905); po = fma(po, a2, 0.004660143486915096);   // c14, c15
    pe = fma(pe, a2, 0.006447210311889649); po = fma(po, a2, 0.005740037670841924);   // c12, c13
    pe = fma(pe, a2, 0.008390335809616815); po = fma(po, a2, 0.0073125258735988454);   // c10, c11
    pe = fma(pe, a2, 0.011551800896139705); po = fma(po, a2, 0.009761609529194078);   // c8, c9
    pe = fma(pe, a2, 0.017352764423076924); po = fma(po, a2, 0.01396484375);   // c6, c7
    pe = fma(pe, a2, 0.030381944444444444); po = fma(po, a2, 0.022372159090909092);   // c4, c5
    pe = fma(pe, a2, 0.075); po = fma(po, a2, 0.044642857142857144);   // c2, c3
    pe = fma(pe, a2, 1.0); po = fma(po, a2, 0.16666666666666666);   // c0, c1
    return fma(po, a, pe);
}
// Same series cut after 10 terms: the remainder is c10 a^10 < 5e-18 for a <= EXB_SHORT_AMAX = 0.03 (support angle
// <= 20 degrees, 2200 km), i.e. below half an ulp of Q ~ 1.
#define EXB_SHORT_AMAX 0.03
__device__ __forceinline__ double exb_asin_sqrt_over_sqrt_short(double a) {
    const double a2 = a * a;
    double pe = 0.011551800896139705, po = 0.009761609529194078;   // c8, c9
    pe = fma(pe, a2, 0.017352764423076924); po = fma(po, a2, 0.01396484375);   // c6, c7
    pe = fma(pe, a2, 0.030381944444444444); po = fma(po, a2, 0.022372159090909092);   // c4, c5
    pe = fma(pe, a2, 0.075); po = fma(po, a2, 0.044642857142857144);   // c2, c3
    pe = fma(pe, a2, 1.0); po = fma(po, a2, 0.16666666666666666);   // c0, c1
    return fma(po, a, pe);
}
template <bool SHORT>
__device__ __forceinline__ double loc_weight_fast_t(double a, double inv_hw, double a_max) {
    const bool inside = a < a_max;
    a = fmin(fmax(a, 1e-30), SHORT ? EXB_SHORT_AMAX : EXB_FAST_AMAX);
    double y = (double)rsqrtf((float)a);                       // 1/sqrt(a) to ~1e-7
    y = y * fma(-0.5 * a, y * y, 1.5);
    y = y * fma(-0.5 * a, y * y, 1.5);
    const double s = a * y;                                    // sqrt(a)
    const double q = SHORT ? exb_asin_sqrt_over_sqrt_short(a) : exb_asin_sqrt_over_sqrt(a);
    const double r = (2.0 * EXB_R_EARTH) * inv_hw * s * q;
    const double rc = fmin(fmax(r, 1.0), 2.0);
    double ir = (double)__frcp_rn((float)rc);                  // 1/r on [1, 2]
    ir = ir * fma(-rc, ir, 2.0);
    ir = ir * fma(-rc, ir, 2.0);
    const double p1 = fma(fma(fma(fma(-0.25, r, 0.5), r, 0.625), r, -5.0 / 3.0), r * r, 1.0);
    const double p2 = fma(fma(fma(fma(fma(r, 1.0 / 12.0, -0.5), r, 0.625), r, 5.0 / 3.0), r, -5.0), r, 4.0) - (2.0 / 3.0) * ir;
    double w = (r <= 1.0) ? p1 : ((r < 2.0) ? p2 : 0.0);
    return inside ? w : 0.0;
}
// Lean form for warp-convergent callers (every lane of the warp must call it): the same arithmetic with the
// special-function seeds taken in double format (MUFU.RSQ64H / RCP64H: no conversions, no libm fix-up code), no
// clamps (values outside the support may become Inf/NaN on the way and are discarded by the final SELECT), and only
// the Gaspari-Cohn branch the warp needs when all of its lanes fall on the same side of r = 1.  The constants that are
// not exact in 32 bits come from a table in the kernel's parameter block (one uniform load each; as literals every
// use costs two moves): k.q = series coefficients c0..c19, k.g = {5/3, 1/12, 2/3, 2 R_earth}.
struct ExbLocConst { double q[20]; double g[4]; };
static inline ExbLocConst exb_loc_const() {
    ExbLocConst k;
    const double c[20] = {1.0, 0.16666666666666666, 0.075, 0.044642857142857144, 0.030381944444444444, 0.022372159090909092,
                          0.017352764423076924, 0.01396484375, 0.011551800896139705, 0.009761609529194078,
                          0.008390335809616815, 0.0073125258735988454, 0.006447210311889649, 0.005740037670841924,
                          0.005153309682319905, 0.004660143486915096, 0.004240907093679363, 0.003880964558837669,
                          0.0035692053938259347, 0.003297059503473485};
    for (int i = 0; i < 20; ++i) k.q[i] = c[i];
    k.g[0] = 5.0 / 3.0; k.g[1] = 1.0 / 12.0; k.g[2] = 2.0 / 3.0; k.g[3] = 2.0 * EXB_R_EARTH;
    return k;
}
template <bool SHORT>
__device__ __forceinline__ double loc_weight_lean(const ExbLocConst &k, double a, double inv_hw, double a_max) {
    const double ap = a + 1e-300;                              // a = 0 (ob on a grid point): r = 0, weight 1
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(ap));    // ~2^-22
    const double hm = -0.5 * ap;
    y = y * fma(hm, y * y, 1.5);
    y = y * fma(hm, y * y, 1.5);
    // asin(sqrt(a)) / sqrt(a) = sum c_n a^n, Horner on two interleaved halves (see exb_asin_sqrt_over_sqrt)
    const double a2 = a * a;
    constexpr int NQ = SHORT ? 10 : 20;
    double pe = k.q[NQ - 2], po = k.q[NQ - 1];
#pragma unroll
    for (int i = NQ - 4; i >= 0; i -= 2) { pe = fma(pe, a2, k.q[i]); po = fma(po, a2, k.q[i + 1]); }
    const double q = fma(po, a, pe);
    const double r = (k.g[3] * inv_hw) * ((ap * y) * q);
    const bool inner = r <= 1.0;
    double w;
    if (__all_sync(0xffffffffu, inner)) {
        w = fma(fma(fma(fma(-0.25, r, 0.5), r, 0.625), r, -k.g[0]), r * r, 1.0);
    } else {
        double ir;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(ir) : "d"(r));
        ir = ir * fma(-r, ir, 2.0);
        ir = ir * fma(-r, ir, 2.0);
        const double p2 = fma(fma(fma(fma(fma(r, k.g[1], -0.5), r, 0.625), r, k.g[0]), r, -5.0), r, 4.0) - k.g[2] * ir;
        w = (r < 2.0) ? p2 : 0.0;
        if (__any_sync(0xffffffffu, inner)) {
            const double p1 = fma(fma(fma(fma(-0.25, r, 0.5), r, 0.625), r, -k.g[0]), r * r, 1.0);
            w = inner ? p1 : w;
        }
    }
    return (a < a_max) ? w : 0.0;
}
__device__ __forceinline__ double loc_weight_fast(double a, double inv_hw, double a_max) {
    const bool inside = a < a_max;
    a = fmin(fmax(a, 1e-30), EXB_FAST_AMAX);
    double y = (double)rsqrtf((float)a);                       // 1/sqrt(a) to ~1e-7
    y = y * fma(-0.5 * a, y * y, 1.5);
    y = y * fma(-0.5 * a, y * y, 1.5);
    const double s = a * y;                                    // sqrt(a)
    const double r = (2.0 * EXB_R_EARTH) * inv_hw * s * exb_asin_sqrt_over_sqrt(a);
    const double rc = fmin(fmax(r, 1.0), 2.0);
    double ir = (double)__frcp_rn((float)rc);                  // 1/r on [1, 2]
    ir = ir * fma(-rc, ir, 2.0);
    ir = ir * fma(-rc, ir, 2.0);
    const double p1 = fma(fma(fma(fma(-0.25, r, 0.5), r, 0.625), r, -5.0 / 3.0), r * r, 1.0);
    const double p2 = fma(fma(fma(fma(fma(r, 1.0 / 12.0, -0.5), r, 0.625), r, 5.0 / 3.0), r, -5.0), r, 4.0) - (2.0 / 3.0) * ir;
    double w = (r <= 1.0) ? p1 : ((r < 2.0) ? p2 : 0.0);
    return inside ? w : 0.0;
}

// candidate lists per coarse tile of the state sweep (state_sweep_2p.cu)
#define SP_CT 4                       // coarse tile = SP_CT x SP_CT patches
struct SweepLists {
    float4 *caps = nullptr;
    int *cnt = nullptr;
    int64_t *off = nullptr;
    int *list = nullptr;
    const int64_t *tile_off = nullptr;    // off shifted so that it is indexed by absolute coarse-tile number
    int nctx = 1, eq_row = -1;
};
// Geometry-only part of a state sweep, built ahead of the obs-space solve (exb_sweep_plan_create): the fp32 scan
// records of the obs and the candidate lists per coarse tile for the patch shape of the two-phase kernel.
struct ExbSweepPlan {
    int64_t nlev = 0, ny = 0, nx = 0, nobs = 0, ob_begin = 0, ob_end = 0, y_begin = 0, y_end = 0;
    int loc_mode = 0;
    const double *grid_u = nullptr;       // identity of the inputs the plan was built from
    const double *obgeo = nullptr;
    float4 *scan = nullptr;
    bool have_lists = false;
    SweepLists lists;
    cudaStream_t st = nullptr;
    cudaEvent_t ready = nullptr, used = nullptr;
    bool was_used = false;
};

template <typename T> struct Vec2;
template <> struct Vec2<double> { typedef double2 type; };
template <> struct Vec2<float> { typedef float2 type; };

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
