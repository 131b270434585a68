// State sweep, FP64 tensor-core version: the float64 path for ensembles of 104 to 255 members.
//
// Same tile-stationary organisation as state_update.cu -- a CTA keeps a patch of grid points (all of
// its levels, 64 state rows) in registers and walks the observations in serial order -- but the
// per-observation dot + axpy (assimilation/ensrf.py:95, :141) is evaluated for 8 consecutive candidate
// observations at a time in a blocked form that is algebraically identical to applying them one by one:
//
//   sequential (ensrf.py:95-141), for q = 0..7 :   d_q = y_q . x ;   x -= e_q y_q ,   e_q = omega_q d_q
//   blocked                                    :   g   = Y x0                        (8 dots at once)
//                                                  d_q = g_q - sum_{p<q} G_qp e_p    (G = Y Y^T, 8x8 Gram)
//                                                  x   = x0 - sum_q e_q y_q
//   omega_q = beta_q * loc_q(row) / ((Nens-1) kdenom_q) carries the localisation weight of the row's
//   grid point, so the short recurrence in the middle is per row; the two big steps are 8x8xNens matrix
//   products and run on the FP64 tensor cores (mma.sync.m8n8k4.f64 -> SASS DMMA, 37 TFLOP/s measured on
//   B200 vs 34 for a DFMA loop).  The point of the blocking is operand traffic: a y value read from shared
//   memory now feeds 8 FMAs instead of 2; the one-ob-at-a-time kernel was bound by the shared-memory pipe
//   (profiles/r01_state_update_v1.md), not by FP64.
//
// The ensemble mean of a row is carried as a pseudo-member: the LAST padded column (8*NT3-1) of the row
// holds xm, and the staged y_q holds -innov_q/beta_q there, so the rank-8 update also performs
// xam = xbm + kmat*innov (ensrf.py:130).  That column is masked out of the dot products.
//
// Fragment layout (m8n8k4, f64): A[8x4] lane l -> A[l/4][l%4]; B[4x8] lane l -> B[l%4][l/4];
// C[8x8] lane l -> C[l/4][2(l%4)], C[l/4][2(l%4)+1].  A warp owns 8 state rows (row = l/4); lane c = l%4 of a
// row keeps members {8t+2c, 8t+2c+1 : t < NT3} in x[2t], x[2t+1], which is simultaneously a valid A operand
// (k-step 2t uses members 8t+2c, k-step 2t+1 members 8t+2c+1) and a valid C operand (n-tile t).
#include "common.cuh"

#define SM_NT 256
#define SM_ROWS 64            // state rows per CTA (8 warps x 8)
#define SM_Q 64               // candidate obs staged per round (8 DMMA batches)

struct SmParams {
    double *xm;
    double *Xp;
    const double *Yp;
    const double *grid_u;
    const double *rec;
    const double *geo;
    const float4 *scan;
    unsigned long long *counters;
    int64_t npts, nobs, ob_begin, ob_end;
    int nlev, ny, nx, nens;
    int ty, tx, ntx;
    int G, Lc, nlc;
    int loc_mode;
};

__device__ __forceinline__ void dmma884(double &c0, double &c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
        : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

template <int NT3> __host__ __device__ constexpr int sm_yst() { return ((8 * NT3) % 16 == 8) ? 8 * NT3 : 8 * NT3 + 8; }
// shared-memory column of member m in staged row q: bit 2 of the column is flipped for rows 2,3,6,7 (mod 8)
// so that both access patterns (8 rows x 64 B and 4 rows x 32 B) are bank-conflict free
__device__ __forceinline__ int sm_swz(int q, int m) { return m ^ (((q >> 1) & 1) << 2); }

template <int NT3>
__global__ void __launch_bounds__(SM_NT, 1)
state_update_mma_kernel(const SmParams p) {
    constexpr int YST = sm_yst<NT3>();

    constexpr int PC = 8 * NT3 - 1;          // column of the pseudo-member (the mean)

    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *s_y = reinterpret_cast<double *>(smem_raw);                 // [SM_Q][YST]
    double *s_om = s_y + SM_Q * YST;                                    // [SM_ROWS grid slots][SM_Q]
    double *s_G = s_om + SM_ROWS * SM_Q;                                // [SM_Q/8][8][8]
    double *s_gu = s_G + (SM_Q / 8) * 64;                               // [3][SM_ROWS]
    double *s_ob = s_gu + 3 * SM_ROWS;                                  // [6][SM_Q] ux uy uz inv_hw a_max c1*beta
    int *s_cand = reinterpret_cast<int *>(s_ob + 6 * SM_Q);             // [SM_Q + SM_NT] queue of ob indices
    int *s_gvalid = s_cand + SM_Q + SM_NT;                              // [SM_ROWS]
    int *s_warp = s_gvalid + SM_ROWS;                                   // [SM_NT/32]
    __shared__ float s_bound[4];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int c = lane & 3, n = lane >> 2;
    const int G = p.G, Lc = p.Lc, nens = p.nens;

    const int lc = blockIdx.x % p.nlc;
    const int tile = blockIdx.x / p.nlc;
    const int y0 = (tile / p.ntx) * p.ty, x0 = (tile % p.ntx) * p.tx;
    const int l0 = lc * Lc;

    // ---- patch geometry -------------------------------------------------------------------
    if (tid < G) {
        const int gy = y0 + tid / p.tx, gx = x0 + tid % p.tx;
        const bool ok = gy < p.ny && gx < p.nx;
        const int64_t pt = ok ? (int64_t)gy * p.nx + gx : (int64_t)y0 * p.nx + x0;
        s_gu[tid] = p.grid_u[pt];
        s_gu[SM_ROWS + tid] = p.grid_u[p.npts + pt];
        s_gu[2 * SM_ROWS + tid] = p.grid_u[2 * p.npts + pt];
        s_gvalid[tid] = ok;
    }
    for (int i = tid; i < SM_Q * YST; i += SM_NT) s_y[i] = 0.0;          // padding columns stay zero
    __syncthreads();
    if (tid == 0) {
        double cx = 0, cy = 0, cz = 0;
        for (int g = 0; g < G; ++g) { cx += s_gu[g]; cy += s_gu[SM_ROWS + g]; cz += s_gu[2 * SM_ROWS + g]; }
        const double nn = sqrt(cx * cx + cy * cy + cz * cz);
        if (nn > 1e-12) { cx /= nn; cy /= nn; cz /= nn; } else { cx = s_gu[0]; cy = s_gu[SM_ROWS]; cz = s_gu[2 * SM_ROWS]; }
        double cmin = 1.0;
        for (int g = 0; g < G; ++g) cmin = fmin(cmin, cx * s_gu[g] + cy * s_gu[SM_ROWS + g] + cz * s_gu[2 * SM_ROWS + g]);
        s_bound[0] = (float)cx; s_bound[1] = (float)cy; s_bound[2] = (float)cz;
        s_bound[3] = (float)(acos(fmax(-1.0, fmin(1.0, cmin))) + 1e-6);
    }

    // ---- this lane's slice of its row ---------------------------------------------------------
    const int r = warp * 8 + n;               // row slot in the CTA
    const int g = r / Lc, l = r % Lc;
    bool active = false;
    int64_t row = 0;
    if (g < G && l0 + l < p.nlev) {
        const int gy = y0 + g / p.tx, gx = x0 + g % p.tx;
        if (gy < p.ny && gx < p.nx) {
            active = true;
            row = (int64_t)(l0 + l) * p.npts + (int64_t)gy * p.nx + gx;
        }
    }
    const int gslot = active ? g : 0;
    double x[2 * NT3];
#pragma unroll
    for (int t = 0; t < NT3; ++t) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int m = 8 * t + 2 * c + h;
            double v = 0.0;
            if (active) {
                if (m < nens) v = p.Xp[row * nens + m];
                else if (m == PC) v = p.xm[row];            // the mean rides along in the last column
            }
            x[2 * t + h] = v;
        }
    }
    const float inv_G = 1.0f / (float)G;
    unsigned long long npairs = 0;
    bool dirty = false;
    __syncthreads();
    const float bcx = s_bound[0], bcy = s_bound[1], bcz = s_bound[2], brho = s_bound[3];

    int qcount = 0;                           // candidates waiting in s_cand (uniform across the CTA)
    int64_t c0 = p.ob_begin;
    while (true) {
        // ---- fill the candidate queue (serial ob order is preserved by the ordered compaction) ----
        while (qcount < SM_Q && c0 < p.ob_end) {
            const int64_t k = c0 + tid;
            bool hit = false;
            if (k < p.ob_end) {
                const float4 sc = p.scan[k];
                if (sc.w >= 0.f) {
                    const float ang = sc.w + brho;
                    hit = (ang >= 3.1405f) || (sc.x * bcx + sc.y * bcy + sc.z * bcz >= __cosf(ang) - 4e-6f);
                }
            }
            const unsigned bal = __ballot_sync(0xffffffffu, hit);
            if (lane == 0) s_warp[warp] = __popc(bal);
            __syncthreads();
            int base = 0, total = 0;
#pragma unroll
            for (int w = 0; w < SM_NT / 32; ++w) {
                const int cnt = s_warp[w];
                if (w < warp) base += cnt;
                total += cnt;
            }
            if (hit) s_cand[qcount + base + __popc(bal & ((1u << lane) - 1u))] = (int)(k - p.ob_begin);
            __syncthreads();
            qcount += total;
            c0 += SM_NT;
        }
        const int nq = qcount < SM_Q ? qcount : SM_Q;
        if (nq == 0) break;
        const int nb = (nq + 7) >> 3;

        // ---- stage the round ------------------------------------------------------------------------
        // (a) per-candidate scalars, (b) y_q rows by cp.async (one warp per row, swizzled columns)
        if (tid < nb * 8) {
            double v0 = 0, v1 = 0, v2 = 0, v3 = 0, v4 = 0, v5 = 0;
            if (tid < nq) {
                const int64_t kk = p.ob_begin + s_cand[tid];
                v0 = p.geo[GEO_UX * p.nobs + kk]; v1 = p.geo[GEO_UY * p.nobs + kk]; v2 = p.geo[GEO_UZ * p.nobs + kk];
                v3 = p.geo[GEO_INVHW * p.nobs + kk]; v4 = p.geo[GEO_AMAX * p.nobs + kk];
                // beta / ((N-1) kdenom)   (ensrf.py:95, :119, :135-136); the localisation weight multiplies it below
                v5 = p.rec[REC_C1 * p.nobs + kk] * p.rec[REC_BETA * p.nobs + kk];
            }
            s_ob[0 * SM_Q + tid] = v0; s_ob[1 * SM_Q + tid] = v1; s_ob[2 * SM_Q + tid] = v2;
            s_ob[3 * SM_Q + tid] = v3; s_ob[4 * SM_Q + tid] = v4; s_ob[5 * SM_Q + tid] = v5;
        }
        for (int q = warp; q < nb * 8; q += SM_NT / 32) {
            double *dst = s_y + q * YST;
            const int sw = ((q >> 1) & 1) << 2;
            if (q < nq) {
                const int64_t kk = p.ob_begin + s_cand[q];
                const double *src = p.Yp + kk * nens;
                if ((nens & 1) == 0) {
                    for (int m = 2 * lane; m < nens; m += 64) {
                        const unsigned sa = (unsigned)__cvta_generic_to_shared(dst + (m ^ sw));
                        asm volatile("cp.async.ca.shared.global [%0], [%1], 16;\n" :: "r"(sa), "l"(src + m));
                    }
                } else {
                    for (int m = lane; m < nens; m += 32) {
                        const unsigned sa = (unsigned)__cvta_generic_to_shared(dst + (m ^ sw));
                        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" :: "r"(sa), "l"(src + m));
                    }
                }
                if (lane == 0)
                    dst[PC ^ sw] = -p.rec[REC_INNOV * p.nobs + kk] / p.rec[REC_BETA * p.nobs + kk];
            } else {
                for (int m = lane; m < nens; m += 32) dst[m ^ sw] = 0.0;
                if (lane == 0) dst[PC ^ sw] = 0.0;
            }
        }
        asm volatile("cp.async.commit_group;\n" ::);
        __syncthreads();
        // (c) omega[g][q] = beta * loc / ((N-1) kdenom), one (ob, grid point) pair at a time per thread
        for (int i = tid; i < nb * 8 * G; i += SM_NT) {
            const int q = (int)(((float)i + 0.5f) * inv_G), gg = i - q * G;
            double om = 0.0;
            if (q < nq && s_gvalid[gg]) {
                double w = 1.0;
                if (p.loc_mode == EXB_LOC_GC) {
                    const double a = hav_a(s_gu[gg], s_gu[SM_ROWS + gg], s_gu[2 * SM_ROWS + gg],
                                           s_ob[0 * SM_Q + q], s_ob[1 * SM_Q + q], s_ob[2 * SM_Q + q]);
                    w = loc_weight(a, s_ob[3 * SM_Q + q], s_ob[4 * SM_Q + q]);
                }
                if (w != 0.0 && lc == 0) npairs++;
                om = w * s_ob[5 * SM_Q + q];
            }
            s_om[gg * SM_Q + q] = om;
        }
        asm volatile("cp.async.wait_all;\n" ::);
        __syncthreads();

        // ---- Gram matrices of the batches: warp w takes batch w -------------------------------------
        for (int b = warp; b < nb; b += SM_NT / 32) {
            double g0 = 0.0, g1 = 0.0, h0 = 0.0, h1 = 0.0;
            const double *yrow = s_y + (8 * b + n) * YST;
            const int sw = ((n >> 1) & 1) << 2;
#pragma unroll
            for (int t = 0; t < NT3; ++t) {
                const double2 v = *reinterpret_cast<const double2 *>(yrow + 8 * t + ((2 * c) ^ sw));
                // the pseudo-member (last column: t = NT3-1, lane c = 3, second element) is not part of y.y
                const double v1 = (t == NT3 - 1 && c == 3) ? 0.0 : v.y;
                dmma884(g0, g1, v.x, v.x);
                dmma884(h0, h1, v1, v1);
            }
            s_G[b * 64 + n * 8 + 2 * c] = g0 + h0;
            s_G[b * 64 + n * 8 + 2 * c + 1] = g1 + h1;
        }
        __syncthreads();

        // ---- apply the batches in order ----------------------------------------------------------------
        for (int b = 0; b < nb; ++b) {
            // omega of this row's grid point for the 8 obs of the batch
            double om[8];
            {
                const double2 *po = reinterpret_cast<const double2 *>(s_om + gslot * SM_Q + 8 * b);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const double2 v = po[i];
                    om[2 * i] = active ? v.x : 0.0;
                    om[2 * i + 1] = active ? v.y : 0.0;
                }
            }
            bool any = false;
#pragma unroll
            for (int i = 0; i < 8; ++i) any |= (om[i] != 0.0);
            if (!__any_sync(0xffffffffu, any)) continue;           // no row of this warp is reached by the batch

            // step 1: g[row][ob] = x[row] . y_ob  (two accumulator chains)
            double ga0 = 0.0, ga1 = 0.0, gb0 = 0.0, gb1 = 0.0;
            {
                const double *yrow = s_y + (8 * b + n) * YST;     // B operand: ob = n, members of lane c
                const int sw = ((n >> 1) & 1) << 2;
#pragma unroll
                for (int t = 0; t < NT3; ++t) {
                    const double2 v = *reinterpret_cast<const double2 *>(yrow + 8 * t + ((2 * c) ^ sw));
                    const double a1 = (t == NT3 - 1 && c == 3) ? 0.0 : x[2 * t + 1];   // mask the mean
                    dmma884(ga0, ga1, x[2 * t], v.x);
                    dmma884(gb0, gb1, a1, v.y);
                }
            }
            ga0 += gb0;                                            // g[row][2c]
            ga1 += gb1;                                            // g[row][2c+1]
            // all-gather the 8 dots of the row over its 4 lanes
            double gq[8];
            {
                const double o0 = __shfl_xor_sync(0xffffffffu, ga0, 1), o1 = __shfl_xor_sync(0xffffffffu, ga1, 1);
                // after this exchange lanes {0,1} hold obs 0..3 and lanes {2,3} hold obs 4..7
                double q0, q1, q2, q3;
                if (c & 1) { q0 = o0; q1 = o1; q2 = ga0; q3 = ga1; } else { q0 = ga0; q1 = ga1; q2 = o0; q3 = o1; }
                const double r0 = __shfl_xor_sync(0xffffffffu, q0, 2), r1 = __shfl_xor_sync(0xffffffffu, q1, 2);
                const double r2 = __shfl_xor_sync(0xffffffffu, q2, 2), r3 = __shfl_xor_sync(0xffffffffu, q3, 2);
                if (c & 2) { gq[0] = r0; gq[1] = r1; gq[2] = r2; gq[3] = r3; gq[4] = q0; gq[5] = q1; gq[6] = q2; gq[7] = q3; }
                else { gq[0] = q0; gq[1] = q1; gq[2] = q2; gq[3] = q3; gq[4] = r0; gq[5] = r1; gq[6] = r2; gq[7] = r3; }
            }
            // step 2: the serial recurrence inside the batch (per row; every lane of the row computes it)
            const double *Gb = s_G + b * 64;
            double e[8];
            e[0] = om[0] * gq[0];
            e[1] = om[1] * (gq[1] - Gb[8] * e[0]);
            e[2] = om[2] * (gq[2] - Gb[16] * e[0] - Gb[17] * e[1]);
            e[3] = om[3] * (gq[3] - Gb[24] * e[0] - Gb[25] * e[1] - Gb[26] * e[2]);
            {
                // obs 4..7 see obs 0..3 through one more 8x8x4 product: corr[row][q] = sum_p e_p G[4+q][p]
                const double ea = (c == 0) ? e[0] : (c == 1) ? e[1] : (c == 2) ? e[2] : e[3];
                double k0 = 0.0, k1 = 0.0;
                dmma884(k0, k1, ea, Gb[(4 + (n & 3)) * 8 + c]);
                // lane c holds corr for obs 4+(2c&3), 5+(2c&3); fetch the other pair from lane c^1
                const double o0 = __shfl_xor_sync(0xffffffffu, k0, 1), o1 = __shfl_xor_sync(0xffffffffu, k1, 1);
                if (c & 1) { gq[4] -= o0; gq[5] -= o1; gq[6] -= k0; gq[7] -= k1; }
                else { gq[4] -= k0; gq[5] -= k1; gq[6] -= o0; gq[7] -= o1; }
            }
            e[4] = om[4] * gq[4];
            e[5] = om[5] * (gq[5] - Gb[44] * e[4]);
            e[6] = om[6] * (gq[6] - Gb[52] * e[4] - Gb[53] * e[5]);
            e[7] = om[7] * (gq[7] - Gb[60] * e[4] - Gb[61] * e[5] - Gb[62] * e[6]);

            // step 3: x[row][:] -= sum_q e_q y_q[:]   (A = -e in two k-steps, B = y, C = x)
            const double ea0 = -((c == 0) ? e[0] : (c == 1) ? e[1] : (c == 2) ? e[2] : e[3]);
            const double ea1 = -((c == 0) ? e[4] : (c == 1) ? e[5] : (c == 2) ? e[6] : e[7]);
            {
                const int sw = ((c >> 1) & 1) << 2;                 // rows 8b+c and 8b+4+c share this swizzle
                const double *y0p = s_y + (8 * b + c) * YST + (n ^ sw);
                const double *y1p = y0p + 4 * YST;
#pragma unroll
                for (int t = 0; t < NT3; ++t) {
                    dmma884(x[2 * t], x[2 * t + 1], ea0, y0p[8 * t]);
                    dmma884(x[2 * t], x[2 * t + 1], ea1, y1p[8 * t]);
                }
            }
            dirty = true;
        }
        __syncthreads();

        // ---- pop the processed candidates --------------------------------------------------------------
        const int rest = qcount - nq;
        int keep = 0;
        if (tid < rest) keep = s_cand[nq + tid];
        int keep2 = 0;
        if (SM_NT + tid < rest) keep2 = s_cand[nq + SM_NT + tid];
        __syncthreads();
        if (tid < rest) s_cand[tid] = keep;
        if (SM_NT + tid < rest) s_cand[SM_NT + tid] = keep2;
        qcount = rest;
        __syncthreads();
    }

    if (active && dirty) {
#pragma unroll
        for (int t = 0; t < NT3; ++t) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int m = 8 * t + 2 * c + h;
                if (m < nens) p.Xp[row * nens + m] = x[2 * t + h];
                else if (m == PC) p.xm[row] = x[2 * t + h];
            }
        }
    }
    if (p.counters && npairs) atomicAdd(&p.counters[1], npairs);
}

template <int NT3>
static int sm_launch(SmParams &p, cudaStream_t st) {
    constexpr int YST = sm_yst<NT3>();
    const int Lc = p.nlev < SM_ROWS ? p.nlev : SM_ROWS;
    const int G = SM_ROWS / Lc;
    int bty = 1, btx = G;
    for (int ty = 1; ty * ty <= G; ++ty) {
        const int tx = G / ty;
        if (ty * tx > bty * btx || (ty * tx == bty * btx && ty > bty)) { bty = ty; btx = tx; }
    }
    if (btx > p.nx) btx = p.nx;
    if (bty > p.ny) bty = p.ny;
    p.ty = bty; p.tx = btx; p.G = bty * btx; p.Lc = Lc;
    p.nlc = (p.nlev + Lc - 1) / Lc;
    p.ntx = (p.nx + btx - 1) / btx;
    const int nty = (p.ny + bty - 1) / bty;
    const size_t smem = sizeof(double) * ((size_t)SM_Q * YST + SM_ROWS * SM_Q + (SM_Q / 8) * 64 + 3 * SM_ROWS + 6 * SM_Q) +
                        sizeof(int) * (SM_Q + SM_NT + SM_ROWS + SM_NT / 32);
    EXB_CUDA(cudaFuncSetAttribute(state_update_mma_kernel<NT3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t nblocks = (int64_t)p.ntx * nty * p.nlc;
    EXB_REQUIRE(nblocks < 0x7fffffff, "too many patches for one launch");
    state_update_mma_kernel<NT3><<<(unsigned)nblocks, SM_NT, smem, st>>>(p);
    exb_count_launches(1);
    return exb_check_launch("state_update_mma_kernel");
}

// Called from state_update.cu for float64 ensembles the two-phase sweep does not take (more than 103 members).
// Returns EXB_ERR_UNSUPPORTED if no variant fits (256 members need 33 tiles).
int exb_state_update_mma_f64(double *xm, double *Xp, int64_t nlev, int64_t ny, int64_t nx, int nens,
                             const double *grid_u, const double *Yp, const double *rec, const double *obgeo,
                             const float4 *scan, int64_t nobs, int64_t ob_begin, int64_t ob_end, int loc_mode,
                             unsigned long long *counters, cudaStream_t st) {
    SmParams p;
    p.xm = xm; p.Xp = Xp; p.Yp = Yp; p.grid_u = grid_u; p.rec = rec; p.geo = obgeo; p.scan = scan;
    p.counters = counters; p.npts = ny * nx; p.nobs = nobs; p.ob_begin = ob_begin; p.ob_end = ob_end;
    p.nlev = (int)nlev; p.ny = (int)ny; p.nx = (int)nx; p.nens = nens; p.loc_mode = loc_mode;
    const int need = (nens + 1 + 7) / 8;            // 8-member tiles incl. the pseudo-member
#define SM_TRY(N) if (need <= N) return sm_launch<N>(p, st)
    SM_TRY(16);
    SM_TRY(20);
    SM_TRY(26);
    SM_TRY(32);
#undef SM_TRY
    return EXB_ERR_UNSUPPORTED;
}
