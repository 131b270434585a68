// Posterior relaxation of the state rows after the serial loop (DESIGN.md section 4.6):
//   RTPS (relaxation to prior spread, Whitaker & Hamill 2012):
//       x <- m_a + x'_a * (1 + alpha (sigma_b - sigma_a) / sigma_a)
//   RTPP (relaxation to prior perturbations, Zhang et al. 2004):
//       x <- m_a + (1 - alpha) x'_a + alpha x'_b
// Rows are addressed as the band pipeline addresses them: for every level lev < nlev, points [p_begin, p_end) of a
// shard with npts points per level, i.e. rows lev*npts + p of X[nlev*npts][nens].  alpha is a device array with one
// value per level.  One warp per row, the row held in registers (NPL = 1, 2, 4 or 8 members per lane), a grid-stride
// loop over the points of a level and over the levels (grid y), so no row index needs a 64-bit division.  Float64
// arithmetic and float64 shuffle reductions in a fixed order: the same row always gives the same mean and sigma bit
// for bit (exb_row_spread before the sweep and the RTPS pass after it share the code, so a row the sweep did not change
// keeps sigma_a == sigma_b and is not written).
#include "common.cuh"

static constexpr int RX_WARPS = 8;            // warps (rows in flight) per 256-thread CTA

__device__ __forceinline__ double warp_sum(double s) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    return s;
}

// member i = lane + 32 j of the row in v[j] (0 past nens)
template <typename T, int NPL>
__device__ __forceinline__ void load_row(const T *__restrict__ row, int nens, int lane, double (&v)[NPL]) {
#pragma unroll
    for (int j = 0; j < NPL; ++j) {
        const int i = lane + 32 * j;
        v[j] = i < nens ? (double)row[i] : 0.0;
    }
}

template <int NPL>
__device__ __forceinline__ double row_mean(const double (&v)[NPL], int nens) {
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < NPL; ++j) s += v[j];
    return warp_sum(s) / (double)nens;
}

// Ensemble standard deviation, ddof = 1.  Exactly 0 when every member is equal: the rounded mean of equal values
// can differ from them, which would leave a sigma of rounding noise for RTPS to divide by.
template <int NPL>
__device__ __forceinline__ double row_sigma(const double (&v)[NPL], double mean, int nens, int lane) {
    const double v0 = __shfl_sync(0xffffffffu, v[0], 0);
    bool flat = true;
    double q = 0.0;
#pragma unroll
    for (int j = 0; j < NPL; ++j) {
        const bool in = lane + 32 * j < nens;
        flat &= !in || v[j] == v0;
        const double d = in ? v[j] - mean : 0.0;
        q += d * d;
    }
    q = warp_sum(q);
    return __all_sync(0xffffffffu, flat) ? 0.0 : sqrt(q / (double)(nens - 1));
}

// Rows lev * npts + p for lev < nlev, p in [p_begin, p_end): grid y strides over the levels, the warps of grid x over
// the points.
#define RX_ROWS_LOOP                                                                                        \
    const int lane = threadIdx.x % 32;                                                                      \
    const int64_t p0 = p_begin + blockIdx.x * (int64_t)RX_WARPS + threadIdx.x / 32;                          \
    const int64_t pstride = (int64_t)gridDim.x * RX_WARPS;                                                  \
    for (int lev = blockIdx.y; lev < nlev; lev += gridDim.y)                                                \
        for (int64_t g = (int64_t)lev * npts + p0, g_end = (int64_t)lev * npts + p_end; g < g_end; g += pstride)

template <typename T, int NPL>
__global__ void __launch_bounds__(32 * RX_WARPS)
row_spread_kernel(const T *__restrict__ X, int nlev, int64_t npts, int64_t p_begin, int64_t p_end, int nens,
                  double *__restrict__ sigma) {
    RX_ROWS_LOOP {
        double v[NPL];
        load_row<T, NPL>(X + g * nens, nens, lane, v);
        const double s = row_sigma<NPL>(v, row_mean<NPL>(v, nens), nens, lane);
        if (lane == 0) sigma[g] = s;
    }
}

template <typename T, int NPL>
__global__ void __launch_bounds__(32 * RX_WARPS)
relax_rtps_kernel(T *__restrict__ X, const double *__restrict__ sigma_b, const double *__restrict__ alpha, int nlev,
                  int64_t npts, int64_t p_begin, int64_t p_end, int nens) {
    RX_ROWS_LOOP {
        const double a = alpha[lev];
        if (a == 0.0) break;                       // alpha = 0: no row of this level is read or written
        T *row = X + g * nens;
        double v[NPL];
        load_row<T, NPL>(row, nens, lane, v);
        const double m = row_mean<NPL>(v, nens);
        const double sa = row_sigma<NPL>(v, m, nens, lane);
        const double sb = sigma_b[g];
        if (sa == 0.0 || sa == sb) continue;       // no spread to scale, or the analysis did not change the row
        const double f = 1.0 + a * (sb - sa) / sa;
#pragma unroll
        for (int j = 0; j < NPL; ++j) {
            const int i = lane + 32 * j;
            if (i < nens) row[i] = (T)(m + (v[j] - m) * f);
        }
    }
}

template <typename T, int NPL>
__global__ void __launch_bounds__(32 * RX_WARPS)
relax_rtpp_kernel(T *__restrict__ X, const T *__restrict__ Xb, const double *__restrict__ alpha, int nlev, int64_t npts,
                  int64_t p_begin, int64_t p_end, int nens) {
    RX_ROWS_LOOP {
        const double a = alpha[lev];
        if (a == 0.0) break;                       // alpha = 0: no row of this level is read or written
        T *row = X + g * nens;
        double v[NPL], w[NPL];
        load_row<T, NPL>(row, nens, lane, v);
        load_row<T, NPL>(Xb + g * nens, nens, lane, w);
        bool same = true;
#pragma unroll
        for (int j = 0; j < NPL; ++j) same &= v[j] == w[j];
        if (__all_sync(0xffffffffu, same)) continue;   // the analysis did not change the row
        const double ma = row_mean<NPL>(v, nens);
        if (row_sigma<NPL>(v, ma, nens, lane) == 0.0) continue;
        const double mb = row_mean<NPL>(w, nens);
#pragma unroll
        for (int j = 0; j < NPL; ++j) {
            const int i = lane + 32 * j;
            if (i < nens) row[i] = (T)(ma + (1.0 - a) * (v[j] - ma) + a * (w[j] - mb));
        }
    }
}

// Argument checks of the entry points; the message names the entry (`what`).
static int check_args(bool pointers, int64_t nlev, int64_t npts, int64_t p_begin, int64_t p_end, int nens,
                      const char *what) {
    if (!pointers) {
        exb_set_error("%s: null pointer", what);
        return EXB_ERR_ARG;
    }
    if (!(nlev > 0 && nlev <= 0x7fffffff && npts > 0 && 0 <= p_begin && p_begin < p_end && p_end <= npts)) {
        exb_set_error("%s: need 0 < nlev < 2^31 and 0 <= p_begin < p_end <= npts (nlev=%lld npts=%lld p=[%lld, %lld))",
                      what, (long long)nlev, (long long)npts, (long long)p_begin, (long long)p_end);
        return EXB_ERR_ARG;
    }
    if (nens < 2) {
        exb_set_error("%s: need nens >= 2 for an ensemble spread (nens=%d)", what, nens);
        return EXB_ERR_ARG;
    }
    if (nens > EXB_MAX_NENS) {
        exb_set_error("%s: nens=%d exceeds EXB_MAX_NENS=%d", what, nens, EXB_MAX_NENS);
        return EXB_ERR_UNSUPPORTED;
    }
    return EXB_OK;
}

// About 148 * 16 CTAs in all: levels on grid y (up to 65535), warps over the points of a level on grid x.
static dim3 grid_for(int64_t nlev, int64_t npts_range) {
    const int64_t gy = nlev < 65535 ? nlev : 65535;
    int64_t gx = ceil_div64(npts_range, RX_WARPS);
    const int64_t cap = (148 * 16 + gy - 1) / gy;
    if (gx > cap) gx = cap;
    return dim3((unsigned)gx, (unsigned)gy);
}

// Each entry instantiates its kernel for 1, 2, 4 or 8 members per lane (nens <= EXB_MAX_NENS = 256).
template <typename T>
static int row_spread_impl(const T *X, int64_t nlev, int64_t npts, int64_t p_begin, int64_t p_end, int nens,
                           double *sigma, void *stream) {
    const int rc = check_args(X && sigma, nlev, npts, p_begin, p_end, nens, "exb_row_spread");
    if (rc != EXB_OK) return rc;
    const dim3 grid = grid_for(nlev, p_end - p_begin);
    const int nl = (int)nlev;
    const cudaStream_t st = (cudaStream_t)stream;
    if (nens <= 32) row_spread_kernel<T, 1><<<grid, 32 * RX_WARPS, 0, st>>>(X, nl, npts, p_begin, p_end, nens, sigma);
    else if (nens <= 64) row_spread_kernel<T, 2><<<grid, 32 * RX_WARPS, 0, st>>>(
        X, nl, npts, p_begin, p_end, nens, sigma);
    else if (nens <= 128) row_spread_kernel<T, 4><<<grid, 32 * RX_WARPS, 0, st>>>(
        X, nl, npts, p_begin, p_end, nens, sigma);
    else row_spread_kernel<T, 8><<<grid, 32 * RX_WARPS, 0, st>>>(X, nl, npts, p_begin, p_end, nens, sigma);
    exb_count_launches(1);
    return exb_check_launch("row_spread_kernel");
}

template <typename T>
static int relax_rtps_impl(T *X, const double *sigma_b, const double *alpha, int64_t nlev, int64_t npts,
                           int64_t p_begin, int64_t p_end, int nens, void *stream) {
    const int rc = check_args(X && sigma_b && alpha, nlev, npts, p_begin, p_end, nens, "exb_relax_rtps");
    if (rc != EXB_OK) return rc;
    const dim3 grid = grid_for(nlev, p_end - p_begin);
    const int nl = (int)nlev;
    const cudaStream_t st = (cudaStream_t)stream;
    if (nens <= 32) relax_rtps_kernel<T, 1><<<grid, 32 * RX_WARPS, 0, st>>>(
        X, sigma_b, alpha, nl, npts, p_begin, p_end, nens);
    else if (nens <= 64) relax_rtps_kernel<T, 2><<<grid, 32 * RX_WARPS, 0, st>>>(
        X, sigma_b, alpha, nl, npts, p_begin, p_end, nens);
    else if (nens <= 128) relax_rtps_kernel<T, 4><<<grid, 32 * RX_WARPS, 0, st>>>(
        X, sigma_b, alpha, nl, npts, p_begin, p_end, nens);
    else relax_rtps_kernel<T, 8><<<grid, 32 * RX_WARPS, 0, st>>>(X, sigma_b, alpha, nl, npts, p_begin, p_end, nens);
    exb_count_launches(1);
    return exb_check_launch("relax_rtps_kernel");
}

template <typename T>
static int relax_rtpp_impl(T *X, const T *Xb, const double *alpha, int64_t nlev, int64_t npts, int64_t p_begin,
                           int64_t p_end, int nens, void *stream) {
    const int rc = check_args(X && Xb && alpha, nlev, npts, p_begin, p_end, nens, "exb_relax_rtpp");
    if (rc != EXB_OK) return rc;
    const dim3 grid = grid_for(nlev, p_end - p_begin);
    const int nl = (int)nlev;
    const cudaStream_t st = (cudaStream_t)stream;
    if (nens <= 32) relax_rtpp_kernel<T, 1><<<grid, 32 * RX_WARPS, 0, st>>>(
        X, Xb, alpha, nl, npts, p_begin, p_end, nens);
    else if (nens <= 64) relax_rtpp_kernel<T, 2><<<grid, 32 * RX_WARPS, 0, st>>>(
        X, Xb, alpha, nl, npts, p_begin, p_end, nens);
    else if (nens <= 128) relax_rtpp_kernel<T, 4><<<grid, 32 * RX_WARPS, 0, st>>>(
        X, Xb, alpha, nl, npts, p_begin, p_end, nens);
    else relax_rtpp_kernel<T, 8><<<grid, 32 * RX_WARPS, 0, st>>>(X, Xb, alpha, nl, npts, p_begin, p_end, nens);
    exb_count_launches(1);
    return exb_check_launch("relax_rtpp_kernel");
}

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
extern "C" int exb_row_spread_f64(const double *X, int64_t nlev, int64_t npts, int64_t p_begin, int64_t p_end, int nens,
                                  double *sigma_out, void *stream) {
    return row_spread_impl<double>(X, nlev, npts, p_begin, p_end, nens, sigma_out, stream);
}
extern "C" int exb_row_spread_f32(const float *X, int64_t nlev, int64_t npts, int64_t p_begin, int64_t p_end, int nens,
                                  double *sigma_out, void *stream) {
    return row_spread_impl<float>(X, nlev, npts, p_begin, p_end, nens, sigma_out, stream);
}
extern "C" int exb_relax_rtps_f64(double *X, const double *sigma_b, const double *alpha_dev, int64_t nlev, int64_t npts,
                                  int64_t p_begin, int64_t p_end, int nens, void *stream) {
    return relax_rtps_impl<double>(X, sigma_b, alpha_dev, nlev, npts, p_begin, p_end, nens, stream);
}
extern "C" int exb_relax_rtps_f32(float *X, const double *sigma_b, const double *alpha_dev, int64_t nlev, int64_t npts,
                                  int64_t p_begin, int64_t p_end, int nens, void *stream) {
    return relax_rtps_impl<float>(X, sigma_b, alpha_dev, nlev, npts, p_begin, p_end, nens, stream);
}
extern "C" int exb_relax_rtpp_f64(double *X, const double *Xb, const double *alpha_dev, int64_t nlev, int64_t npts,
                                  int64_t p_begin, int64_t p_end, int nens, void *stream) {
    return relax_rtpp_impl<double>(X, Xb, alpha_dev, nlev, npts, p_begin, p_end, nens, stream);
}
extern "C" int exb_relax_rtpp_f32(float *X, const float *Xb, const double *alpha_dev, int64_t nlev, int64_t npts,
                                  int64_t p_begin, int64_t p_end, int nens, void *stream) {
    return relax_rtpp_impl<float>(X, Xb, alpha_dev, nlev, npts, p_begin, p_end, nens, stream);
}
