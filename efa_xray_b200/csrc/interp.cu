// Bilinear forward operator (DESIGN.md section 4.8): for every ob the 4 corners of the grid cell that contains it
// and their bilinear weights, in the idx4 / w4 format exb_stencil_combine consumes.  An ob outside the grid gets
// idx 0 / w 0 and is counted in n_outside.
#include "common.cuh"

__device__ __forceinline__ void bilinear_store(int64_t k, int64_t p00, int64_t p01, int64_t p10, int64_t p11,
                                               double s, double t, int64_t *__restrict__ idx4,
                                               double *__restrict__ w4) {
    idx4[k * 4 + 0] = p00; idx4[k * 4 + 1] = p01; idx4[k * 4 + 2] = p10; idx4[k * 4 + 3] = p11;
    w4[k * 4 + 0] = (1.0 - s) * (1.0 - t);
    w4[k * 4 + 1] = s * (1.0 - t);
    w4[k * 4 + 2] = (1.0 - s) * t;
    w4[k * 4 + 3] = s * t;
}

__device__ __forceinline__ void bilinear_outside(int64_t k, int64_t *__restrict__ idx4, double *__restrict__ w4,
                                                 int32_t *__restrict__ n_outside) {
#pragma unroll
    for (int r = 0; r < 4; ++r) { idx4[k * 4 + r] = 0; w4[k * 4 + r] = 0.0; }
    atomicAdd(n_outside, 1);
}

// ------------------------------------------------------------------------------------------
// rectilinear grids: lat_y strictly monotone, lon_x strictly increasing after unwrapping (lon_u)
// ------------------------------------------------------------------------------------------
__global__ void bilinear_rect_kernel(const double *__restrict__ lat_y, const double *__restrict__ lon_u, int ny,
                                     int nx, int periodic, const double *__restrict__ ob_lat,
                                     const double *__restrict__ ob_lon, int64_t nobs, int64_t *__restrict__ idx4,
                                     double *__restrict__ w4, int32_t *__restrict__ n_outside) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= nobs) return;
    const double phi = ob_lat[k];
    const double L0 = lon_u[0], Llast = lon_u[nx - 1];
    // lambda' = L0 + ((lambda - L0) mod 360), with numpy's floating mod (the result takes the divisor's sign)
    double m = fmod(ob_lon[k] - L0, 360.0);
    if (m < 0.0) m += 360.0;
    const double lam = L0 + m;
    const bool asc = lat_y[ny - 1] > lat_y[0];
    const double lat_lo = asc ? lat_y[0] : lat_y[ny - 1], lat_hi = asc ? lat_y[ny - 1] : lat_y[0];
    if (!(phi >= lat_lo && phi <= lat_hi) || !(lam == lam) || (!periodic && !(lam <= Llast))) {
        bilinear_outside(k, idx4, w4, n_outside);
        return;
    }
    // column: the largest i <= nx-2 with L_i <= lambda' (L_0 <= lambda' always), or the closing cell nx-1 -> 0
    int i, i1;
    double xl, xr;
    if (lam > Llast) {
        i = nx - 1; i1 = 0; xl = Llast; xr = L0 + 360.0;
    } else {
        int lo = 0, hi = nx - 2;                       // invariant: lon_u[lo] <= lambda'
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (lon_u[mid] <= lam) lo = mid; else hi = mid - 1;
        }
        i = lo; i1 = lo + 1; xl = lon_u[i]; xr = lon_u[i1];
    }
    // row: the lowest j with phi between lat_y[j] and lat_y[j+1] inclusive = (first k >= 1 past phi) - 1
    int lo = 1, hi = ny - 1;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const double v = lat_y[mid];
        if (asc ? (v >= phi) : (v <= phi)) hi = mid; else lo = mid + 1;
    }
    const int j = lo - 1;
    const double s = (lam - xl) / (xr - xl);
    const double t = (phi - lat_y[j]) / (lat_y[j + 1] - lat_y[j]);
    const int64_t r0 = (int64_t)j * nx, r1 = r0 + nx;
    bilinear_store(k, r0 + i, r0 + i1, r1 + i, r1 + i1, s, t, idx4, w4);
}

// ------------------------------------------------------------------------------------------
// curvilinear grids: nearest grid point by great-circle distance, then inverse bilinear cell tests
// ------------------------------------------------------------------------------------------
// One CTA = BC_TX point-lanes x BC_OY groups of BC_OB obs, as nearest4_kernel, keeping the top 1 by dot product.
#define BC_TX 128
#define BC_OY 4
#define BC_OB 8
#define BC_OBS_PER_CTA (BC_OY * BC_OB)
#define BC_IN_TOL 1e-10

__device__ __forceinline__ bool dot_better(double da, int ia, double db, int ib) {
    return (da > db) || (da == db && ia < ib);
}

// longitude difference a - b wrapped into [-180, 180]
__device__ __forceinline__ double wrap180(double d) {
    d = fmod(d, 360.0);
    if (d > 180.0) d -= 360.0;
    else if (d < -180.0) d += 360.0;
    return d;
}

// Inverse bilinear coordinates (s, t) of the ob in the cell with corners A = (y, x), B = (y, x+1), C = (y+1, x),
// D = (y+1, x+1), in the (lon, lat) plane relative to the ob, corner longitudes unwrapped to within 180 degrees of
// the ob's.  P(s, t) = A + s e + t f + s t g with e = B - A, f = C - A, g = (A - B) - (C - D) (exactly 0 on a
// rectangle); P(s, t) = 0 is the quadratic k2 t^2 + k1 t + k0 = 0, solved in the form that stays accurate when k2 is
// small or 0.  Returns true when a root has both coordinates in [-tol, 1 + tol].
__device__ bool cell_contains(const double *__restrict__ lat, const double *__restrict__ lon, int nx, int y, int x,
                              double olat, double olon, double &s_out, double &t_out) {
    const int64_t a = (int64_t)y * nx + x, b = a + 1, c = a + nx, d = c + 1;
    const double ax = wrap180(lon[a] - olon), ay = lat[a] - olat;
    const double bx = wrap180(lon[b] - olon), by = lat[b] - olat;
    const double cx = wrap180(lon[c] - olon), cy = lat[c] - olat;
    const double dx = wrap180(lon[d] - olon), dy = lat[d] - olat;
    const double ex = bx - ax, ey = by - ay, fx = cx - ax, fy = cy - ay;
    const double gx = (ax - bx) - (cx - dx), gy = (ay - by) - (cy - dy);
    const double hx = -ax, hy = -ay;                   // ob - A
    const double k2 = gx * fy - gy * fx;
    const double k1 = (ex * fy - ey * fx) + (hx * gy - hy * gx);
    const double k0 = hx * ey - hy * ex;
    double roots[2];
    int nroot = 0;
    if (k2 == 0.0) {
        if (k1 != 0.0) roots[nroot++] = -k0 / k1;
    } else {
        const double disc = k1 * k1 - 4.0 * k0 * k2;
        if (disc < 0.0) return false;
        const double q = -0.5 * (k1 + copysign(sqrt(disc), k1));
        if (q != 0.0) roots[nroot++] = k0 / q;         // the root that tends to -k0/k1 as k2 -> 0
        roots[nroot++] = q / k2;
    }
    for (int r = 0; r < nroot; ++r) {
        const double t = roots[r];
        if (!(t >= -BC_IN_TOL && t <= 1.0 + BC_IN_TOL)) continue;
        const double denx = ex + gx * t, deny = ey + gy * t;
        double s;
        if (fabs(denx) >= fabs(deny)) {
            if (denx == 0.0) continue;
            s = (hx - fx * t) / denx;
        } else {
            s = (hy - fy * t) / deny;
        }
        if (!(s >= -BC_IN_TOL && s <= 1.0 + BC_IN_TOL)) continue;
        s_out = fmin(fmax(s, 0.0), 1.0);
        t_out = fmin(fmax(t, 0.0), 1.0);
        return true;
    }
    return false;
}

__global__ void __launch_bounds__(BC_TX *BC_OY)
bilinear_curv_kernel(const double *__restrict__ u, const double *__restrict__ lat, const double *__restrict__ lon,
                     int ny, int nx, const double *__restrict__ ob_lat, const double *__restrict__ ob_lon,
                     int64_t nobs, int64_t *__restrict__ idx4, double *__restrict__ w4,
                     int32_t *__restrict__ n_outside) {
    __shared__ double s_d[BC_OBS_PER_CTA][BC_TX / 32];
    __shared__ int s_i[BC_OBS_PER_CTA][BC_TX / 32];
    const int tx = threadIdx.x % BC_TX;
    const int oy = threadIdx.x / BC_TX;
    const int lane = threadIdx.x % 32;
    const int64_t ob0 = blockIdx.x * (int64_t)BC_OBS_PER_CTA + oy * BC_OB;
    const int npts = ny * nx;
    double ox[BC_OB], oyv[BC_OB], oz[BC_OB], bd[BC_OB];
    int bi[BC_OB];
#pragma unroll
    for (int o = 0; o < BC_OB; ++o) {
        const int64_t k = ob0 + o < nobs ? ob0 + o : nobs - 1;
        double sp, cp, sl, cl;                         // as grid_unitvec_kernel
        sincos(ob_lat[k] * EXB_DEG2RAD, &sp, &cp);
        sincos(ob_lon[k] * EXB_DEG2RAD, &sl, &cl);
        ox[o] = cp * cl; oyv[o] = cp * sl; oz[o] = sp;
        bd[o] = -INFINITY; bi[o] = 0x7fffffff;
    }
    // points in increasing index order, strict '>': each lane keeps the lowest index among equal dot products
    for (int p = tx; p < npts; p += BC_TX) {
        const double ux = u[p], uy = u[npts + p], uz = u[2 * (int64_t)npts + p];
#pragma unroll
        for (int o = 0; o < BC_OB; ++o) {
            const double v = ux * ox[o] + uy * oyv[o] + uz * oz[o];
            if (v > bd[o]) { bd[o] = v; bi[o] = p; }
        }
    }
#pragma unroll
    for (int o = 0; o < BC_OB; ++o) {
        double d = bd[o];
        int i = bi[o];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const double od = __shfl_xor_sync(0xffffffffu, d, off);
            const int oi = __shfl_xor_sync(0xffffffffu, i, off);
            if (dot_better(od, oi, d, i)) { d = od; i = oi; }
        }
        if (lane == 0) { s_d[oy * BC_OB + o][tx / 32] = d; s_i[oy * BC_OB + o][tx / 32] = i; }
    }
    __syncthreads();
    if (threadIdx.x >= BC_OBS_PER_CTA) return;
    const int o = threadIdx.x;
    const int64_t k = blockIdx.x * (int64_t)BC_OBS_PER_CTA + o;
    if (k >= nobs) return;
    double d = s_d[o][0];
    int best = s_i[o][0];
    for (int w = 1; w < BC_TX / 32; ++w)
        if (dot_better(s_d[o][w], s_i[o][w], d, best)) { d = s_d[o][w]; best = s_i[o][w]; }
    if (best >= npts) {                                // no comparable point (NaN ob coordinates)
        bilinear_outside(k, idx4, w4, n_outside);
        return;
    }
    const int py = best / nx, px = best - py * nx;
    const double olat = ob_lat[k], olon = ob_lon[k];
    // the up to 4 cells with p* as a corner first, then the rest of the 4x4-cell block around p*, row-major
    for (int pass = 0; pass < 2; ++pass) {
        for (int y = py - 2; y <= py + 1; ++y) {
            for (int x = px - 2; x <= px + 1; ++x) {
                const bool inner = (y == py - 1 || y == py) && (x == px - 1 || x == px);
                if (inner != (pass == 0) || y < 0 || y > ny - 2 || x < 0 || x > nx - 2) continue;
                double s, t;
                if (cell_contains(lat, lon, nx, y, x, olat, olon, s, t)) {
                    const int64_t r0 = (int64_t)y * nx, r1 = r0 + nx;
                    bilinear_store(k, r0 + x, r0 + x + 1, r1 + x, r1 + x + 1, s, t, idx4, w4);
                    return;
                }
            }
        }
    }
    bilinear_outside(k, idx4, w4, n_outside);
}

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
extern "C" int exb_stencil_bilinear_rect(const double *lat_y_deg, const double *lon_x_unwrapped, int64_t ny, int64_t nx,
                                         int periodic, const double *ob_lat_deg, const double *ob_lon_deg, int64_t nobs,
                                         int64_t *idx4, double *w4, int32_t *n_outside, void *stream) {
    EXB_REQUIRE(lat_y_deg && lon_x_unwrapped && ob_lat_deg && ob_lon_deg && idx4 && w4 && n_outside, "null pointer");
    EXB_REQUIRE(ny >= 2 && nx >= 2 && ny * nx < 0x7fffffff && nobs > 0, "need ny, nx >= 2, ny*nx < 2^31 and nobs > 0");
    EXB_REQUIRE(periodic == 0 || periodic == 1, "periodic must be 0 or 1");
    EXB_CUDA(cudaMemsetAsync(n_outside, 0, sizeof(int32_t), (cudaStream_t)stream));
    bilinear_rect_kernel<<<(unsigned)ceil_div64(nobs, 256), 256, 0, (cudaStream_t)stream>>>(
        lat_y_deg, lon_x_unwrapped, (int)ny, (int)nx, periodic, ob_lat_deg, ob_lon_deg, nobs, idx4, w4, n_outside);
    exb_count_launches(1);
    return exb_check_launch("bilinear_rect_kernel");
}

extern "C" int exb_stencil_bilinear_curv(const double *grid_u, const double *lat_g_deg, const double *lon_g_deg,
                                         int64_t ny, int64_t nx, const double *ob_lat_deg, const double *ob_lon_deg,
                                         int64_t nobs, int64_t *idx4, double *w4, int32_t *n_outside, void *stream) {
    EXB_REQUIRE(grid_u && lat_g_deg && lon_g_deg && ob_lat_deg && ob_lon_deg && idx4 && w4 && n_outside,
                "null pointer");
    EXB_REQUIRE(ny >= 2 && nx >= 2 && ny * nx < 0x7fffffff && nobs > 0, "need ny, nx >= 2, ny*nx < 2^31 and nobs > 0");
    EXB_CUDA(cudaMemsetAsync(n_outside, 0, sizeof(int32_t), (cudaStream_t)stream));
    bilinear_curv_kernel<<<(unsigned)ceil_div64(nobs, BC_OBS_PER_CTA), BC_TX * BC_OY, 0, (cudaStream_t)stream>>>(
        grid_u, lat_g_deg, lon_g_deg, (int)ny, (int)nx, ob_lat_deg, ob_lon_deg, nobs, idx4, w4, n_outside);
    exb_count_launches(1);
    return exb_check_launch("bilinear_curv_kernel");
}
