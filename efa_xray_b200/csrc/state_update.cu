// State sweep (pieces 2, 3 and 4 of the north star for the state rows): kcov, on-the-fly
// Gaspari-Cohn localisation, gain, mean update and square-root perturbation update of
// assimilation/ensrf.py:95-141, for every state row of a latitude-band shard.
//
// Tile-stationary: a CTA owns a small patch of grid points (all of its levels), keeps the patch's
// perturbations and means in REGISTERS, and walks the observations in serial order, applying every ob
// whose localisation footprint reaches the patch.  State rows never read other state rows (ensrf.py:95,
// :141 are row-wise), so this ordering gives the reference's result while the state crosses HBM once
// (one read, one write) instead of once per observation.  What is left per (row, ob) pair is the
// 2*Nens-flop dot + axpy, which makes the kernel FP64-pipe bound; see DESIGN.md for the roofline.
//
// Thread mapping: a state row is owned by a group of S lanes; lane s keeps members s, s+S, ... (MC per
// lane).  A CTA has NT/S groups = G grid points x Lc levels.  Per sub-batch of Q candidate obs the CTA
// first evaluates the Q*G localisation weights cooperatively (one pair per thread, no redundancy across
// the lanes of a group) and stages the Q obs ensembles ye in shared memory, then each group applies the
// Q obs in order to its row.
#include "common.cuh"
#include <type_traits>

int exb_state_update_mma_f64(double *xm, double *Xp, int64_t nlev, int64_t ny, int64_t nx, int nens,
                             const double *grid_u, const double *Yp, const double *rec, const double *obgeo,
                             const float4 *scan, int64_t nobs, int64_t ob_begin, int64_t ob_end, int loc_mode,
                             unsigned long long *counters, cudaStream_t st);

template <typename TS>
int exb_state_sweep_2p(TS *xm, TS *Xp, int64_t nlev, int64_t ny, int64_t nx, int nens, const double *grid_u, const TS *Yp,
                       const double *rec, const double *obgeo, const float4 *scan, int64_t nobs, int64_t ob_begin,
                       int64_t ob_end, int64_t y_begin, int64_t y_end, int loc_mode, unsigned long long *counters,
                       cudaStream_t st, const ExbSweepPlan *plan = nullptr);

#define SU_NT 256
#define SU_QCAP 16

struct SuParams {
    void *xm;
    void *Xp;
    const void *Yp;
    const double *grid_u;
    const double *rec;
    const double *geo;
    const float4 *scan;          // (ux, uy, uz, theta) per ob; theta < 0: never a candidate
    unsigned long long *counters;
    int64_t npts;                // ny * nx
    int64_t nobs;
    int64_t ob_begin, ob_end;
    int nlev, ny, nx, nens;
    int ty, tx, ntx;             // patch shape and number of patches along x
    int G, Lc, nlc, Q;
    int loc_mode;
};

template <typename T> __host__ __device__ constexpr int su_vec() { return 16 / (int)sizeof(T); }
// per-lane stride of the staged ye (elements): multiple of a 16-byte vector, and an odd number of
// vectors so that the S lane chunks of a group fall in distinct shared-memory banks
template <typename T, int MC> __host__ __device__ constexpr int su_mcp() {
    int v = su_vec<T>();
    int n = (MC + v - 1) / v;
    if (n % 2 == 0) n += 1;
    return n * v;
}

// one 16-byte shared-memory load into scalar registers
template <typename T> __device__ __forceinline__ void su_load_vec(const T *src, T *dst);
template <> __device__ __forceinline__ void su_load_vec<double>(const double *src, double *dst) {
    const double2 v = *reinterpret_cast<const double2 *>(src);
    dst[0] = v.x; dst[1] = v.y;
}
template <> __device__ __forceinline__ void su_load_vec<float>(const float *src, float *dst) {
    const float4 v = *reinterpret_cast<const float4 *>(src);
    dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
}

template <int S>
__device__ __forceinline__ double su_group_sum(double v, unsigned mask) {
#pragma unroll
    for (int off = S / 2; off > 0; off >>= 1) v += __shfl_xor_sync(mask, v, off);
    return v;
}

template <typename T, int S, int MC>
__global__ void __launch_bounds__(SU_NT)
state_update_kernel(const SuParams p) {
    constexpr int MCP = su_mcp<T, MC>();
    constexpr int YS = S * MCP;              // staged elements per ob
    constexpr int RPC = SU_NT / S;           // rows (groups) per CTA
    constexpr int VEC = su_vec<T>();

    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *s_y = reinterpret_cast<T *>(smem_raw);                                  // [Q][YS]
    double *s_w = reinterpret_cast<double *>(s_y + (size_t)SU_QCAP * YS);      // [Q][G]
    double *s_sc = s_w + SU_QCAP * RPC;                                        // [Q][3]
    double *s_gu = s_sc + SU_QCAP * 3;                                         // [3][RPC]
    int *s_cand = reinterpret_cast<int *>(s_gu + 3 * RPC);                     // [NT]
    int *s_gvalid = s_cand + SU_NT;                                            // [RPC]
    int *s_warp = s_gvalid + RPC;                                              // [NT/32 + 1]
    __shared__ float s_bound[5];                                               // cx cy cz rho  (+pad)

    const int tid = threadIdx.x;
    const int lane = tid % 32;
    const int s = tid % S;
    const int r = tid / S;                   // group
    const unsigned gmask = (S == 32) ? 0xffffffffu : (((1u << S) - 1u) << (lane & ~(S - 1)));
    const int G = p.G, Lc = p.Lc;

    const int lc = blockIdx.x % p.nlc;
    const int tile = blockIdx.x / p.nlc;
    const int y0 = (tile / p.ntx) * p.ty, x0 = (tile % p.ntx) * p.tx;
    const int l0 = lc * Lc;

    // ---- patch geometry ---------------------------------------------------------------
    if (tid < G) {
        const int gy = y0 + tid / p.tx, gx = x0 + tid % p.tx;
        const bool ok = gy < p.ny && gx < p.nx;
        // out-of-domain slots mirror the patch's first point (always in the domain)
        const int64_t pt = ok ? (int64_t)gy * p.nx + gx : (int64_t)y0 * p.nx + x0;
        s_gu[tid] = p.grid_u[pt];
        s_gu[RPC + tid] = p.grid_u[p.npts + pt];
        s_gu[2 * RPC + tid] = p.grid_u[2 * p.npts + pt];
        s_gvalid[tid] = ok;
    }
    for (int i = tid; i < SU_QCAP * YS; i += SU_NT) s_y[i] = (T)0;   // padding lanes stay zero
    __syncthreads();
    if (tid == 0) {
        double cx = 0, cy = 0, cz = 0;
        for (int g = 0; g < G; ++g) { cx += s_gu[g]; cy += s_gu[RPC + g]; cz += s_gu[2 * RPC + g]; }
        const double n = sqrt(cx * cx + cy * cy + cz * cz);
        if (n > 1e-12) { cx /= n; cy /= n; cz /= n; } else { cx = s_gu[0]; cy = s_gu[RPC]; cz = s_gu[2 * RPC]; }
        double cmin = 1.0;
        for (int g = 0; g < G; ++g) cmin = fmin(cmin, cx * s_gu[g] + cy * s_gu[RPC + g] + cz * s_gu[2 * RPC + g]);
        s_bound[0] = (float)cx; s_bound[1] = (float)cy; s_bound[2] = (float)cz;
        s_bound[3] = (float)(acos(fmax(-1.0, fmin(1.0, cmin))) + 1e-6);
    }

    // ---- this thread's row ---------------------------------------------------------------
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
    T *Xp = reinterpret_cast<T *>(p.Xp);
    T *xmv = reinterpret_cast<T *>(p.xm);
    const T *Yp = reinterpret_cast<const T *>(p.Yp);
    T x[MC];
#pragma unroll
    for (int i = 0; i < MC; ++i) {
        const int m = s + S * i;
        x[i] = (active && m < p.nens) ? Xp[row * p.nens + m] : (T)0;
    }
    double xmean = active ? (double)xmv[row] : 0.0;
    unsigned long long npairs = 0;
    bool dirty = false;
    __syncthreads();
    const float bcx = s_bound[0], bcy = s_bound[1], bcz = s_bound[2], brho = s_bound[3];

    // ---- walk the observations in order ------------------------------------------------------
    for (int64_t c0 = p.ob_begin; c0 < p.ob_end; c0 += SU_NT) {
        // candidate test: can ob k's footprint reach this patch?
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
        if (lane == 0) s_warp[tid / 32] = __popc(bal);
        __syncthreads();
        int base = 0, total = 0;
#pragma unroll
        for (int w = 0; w < SU_NT / 32; ++w) {
            const int c = s_warp[w];
            if (w < tid / 32) base += c;
            total += c;
        }
        if (hit) s_cand[base + __popc(bal & ((1u << lane) - 1u))] = (int)(k - c0);
        __syncthreads();

        for (int q0 = 0; q0 < total; q0 += p.Q) {
            const int qn = (total - q0) < p.Q ? (total - q0) : p.Q;
            // (1) localisation weights, one (ob, grid point) pair per thread
            if (tid < qn * G) {
                const int q = tid / G, gg = tid % G;
                const int64_t kk = c0 + s_cand[q0 + q];
                double w = 0.0;
                if (s_gvalid[gg]) {
                    w = 1.0;
                    if (p.loc_mode == EXB_LOC_GC) {
                        const double a = hav_a(s_gu[gg], s_gu[RPC + gg], s_gu[2 * RPC + gg],
                                               p.geo[GEO_UX * p.nobs + kk], p.geo[GEO_UY * p.nobs + kk],
                                               p.geo[GEO_UZ * p.nobs + kk]);
                        w = loc_weight(a, p.geo[GEO_INVHW * p.nobs + kk], p.geo[GEO_AMAX * p.nobs + kk]);
                    }
                    if (w != 0.0 && lc == 0) npairs++;
                }
                s_w[q * G + gg] = w;
            }
            // (2) stage ye of the qn obs, permuted so that lane s finds its members contiguous
            for (int e = tid; e < qn * p.nens; e += SU_NT) {
                const int q = e / p.nens, m = e % p.nens;
                const int64_t kk = c0 + s_cand[q0 + q];
                s_y[q * YS + (m % S) * MCP + (m / S)] = Yp[kk * p.nens + m];
            }
            if (tid < qn) {
                const int64_t kk = c0 + s_cand[q0 + tid];
                s_sc[tid * 3 + 0] = p.rec[REC_INNOV * p.nobs + kk];
                s_sc[tid * 3 + 1] = p.rec[REC_C1 * p.nobs + kk];
                s_sc[tid * 3 + 2] = p.rec[REC_BETA * p.nobs + kk];
            }
            __syncthreads();
            // (3) apply the qn obs in order to this group's row
            if (active) {
                for (int q = 0; q < qn; ++q) {
                    const double w = s_w[q * G + g];
                    if (w != 0.0) {
                        const T *yq = s_y + q * YS + s * MCP;
                        T ye[MCP];
#pragma unroll
                        for (int i = 0; i < MCP; i += VEC) {
                            if (i < MC) su_load_vec<T>(yq + i, &ye[i]);
                        }
                        T d0 = 0, d1 = 0, d2 = 0, d3 = 0;
#pragma unroll
                        for (int i = 0; i < MC; i += 4) {
                            d0 += x[i] * ye[i];
                            if (i + 1 < MC) d1 += x[i + 1] * ye[i + 1];
                            if (i + 2 < MC) d2 += x[i + 2] * ye[i + 2];
                            if (i + 3 < MC) d3 += x[i + 3] * ye[i + 3];
                        }
                        const double dot = su_group_sum<S>((double)((d0 + d1) + (d2 + d3)), gmask);
                        const double kmat = w * dot * s_sc[q * 3 + 1];        // loc*kcov/kdenom, ensrf.py:115-119
                        xmean += kmat * s_sc[q * 3 + 0];                      // ensrf.py:130
                        const T f = (T)(s_sc[q * 3 + 2] * kmat);              // beta*kmat, ensrf.py:136
#pragma unroll
                        for (int i = 0; i < MC; ++i) x[i] -= f * ye[i];       // ensrf.py:141
                        dirty = true;
                    }
                }
            }
            __syncthreads();
        }
    }

    if (active && dirty) {
#pragma unroll
        for (int i = 0; i < MC; ++i) {
            const int m = s + S * i;
            if (m < p.nens) Xp[row * p.nens + m] = x[i];
        }
        if (s == 0) xmv[row] = (T)xmean;
    }
    if (p.counters && npairs) atomicAdd(&p.counters[1], npairs);
}

// scan records: unit vector + support angle in fp32, theta = -1 for obs that were not assimilated
__global__ void su_scan_records_kernel(const double *__restrict__ geo, const double *__restrict__ rec,
                                       int64_t nobs, float4 *__restrict__ scan) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= nobs) return;
    float4 v;
    v.x = (float)geo[GEO_UX * nobs + k];
    v.y = (float)geo[GEO_UY * nobs + k];
    v.z = (float)geo[GEO_UZ * nobs + k];
    v.w = rec[REC_ASSIM * nobs + k] != 0.0 ? (float)geo[GEO_THETA * nobs + k] * 1.000001f + 1e-7f : -1.f;
    scan[k] = v;
}

template <typename T, int S, int MC>
static int su_launch(SuParams &p, cudaStream_t st) {
    constexpr int MCP = su_mcp<T, MC>();
    constexpr int YS = S * MCP;
    constexpr int RPC = SU_NT / S;
    const int Lc = p.nlev < RPC ? p.nlev : RPC;
    const int G = RPC / Lc;
    // patch shape: ty*tx <= G, as many points as possible, then as square as possible
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
    int Q = SU_NT / p.G;
    if (Q > SU_QCAP) Q = SU_QCAP;
    if (Q < 1) Q = 1;
    p.Q = Q;
    const size_t smem = (size_t)SU_QCAP * YS * sizeof(T) + sizeof(double) * (SU_QCAP * RPC + SU_QCAP * 3 + 3 * RPC) +
                        sizeof(int) * (SU_NT + RPC + SU_NT / 32 + 1);
    EXB_CUDA(cudaFuncSetAttribute(state_update_kernel<T, S, MC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t nblocks = (int64_t)p.ntx * nty * p.nlc;
    EXB_REQUIRE(nblocks < 0x7fffffff, "too many patches for one launch");
    state_update_kernel<T, S, MC><<<(unsigned)nblocks, SU_NT, smem, st>>>(p);
    exb_count_launches(1);
    return exb_check_launch("state_update_kernel");
}

// Eight lanes per row; the host picks the smallest MC with 8 * MC >= nens.  The kernel serves ensembles above 103
// members (state_update_impl), where 8 lanes per row keep MC at 32 or below up to EXB_MAX_NENS.
template <typename T>
static int su_dispatch(SuParams &p, cudaStream_t st) {
    if (p.nens <= 8 * 13) return su_launch<T, 8, 13>(p, st);
    if (p.nens <= 8 * 25) return su_launch<T, 8, 25>(p, st);
    if (p.nens <= 8 * 32) return su_launch<T, 8, 32>(p, st);
    exb_set_error("exb_state_update: no kernel variant for nens=%d (max %d)", p.nens, EXB_MAX_NENS);
    return EXB_ERR_UNSUPPORTED;
}

template <typename T>
static int state_update_impl(T *xm, T *Xp, int64_t nlev, int64_t ny, int64_t nx, int nens, const double *grid_u,
                             const T *Yp, const double *rec, const double *obgeo, int64_t nobs, int64_t ob_begin,
                             int64_t ob_end, int loc_mode, unsigned long long *counters, void *stream) {
    EXB_REQUIRE(xm && Xp && grid_u && Yp && rec && obgeo, "null pointer");
    EXB_REQUIRE(nlev > 0 && ny > 0 && nx > 0 && nens >= 2 && nobs > 0, "bad sizes");
    EXB_REQUIRE(nlev < (1 << 30) && ny < (1 << 30) && nx < (1 << 30), "dimension too large");
    EXB_REQUIRE(0 <= ob_begin && ob_begin <= ob_end && ob_end <= nobs, "bad ob range");
    EXB_REQUIRE(loc_mode == EXB_LOC_NONE || loc_mode == EXB_LOC_GC, "bad loc_mode");
    if (ob_begin == ob_end) return EXB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    float4 *scan = nullptr;
    EXB_CUDA(exb_malloc_async(&scan, (size_t)nobs * sizeof(float4), st));
    su_scan_records_kernel<<<(unsigned)ceil_div64(nobs, 256), 256, 0, st>>>(obgeo, rec, nobs, scan);
    exb_count_launches(1);
    // FP64 tensor-core sweeps (float32 states: float32 storage, float64 arithmetic in registers): the two-phase
    // sweep (state_sweep_2p.cu) up to 103 members, then state_update_mma.cu for float64 up to 255 members
    int rc = exb_state_sweep_2p<T>(xm, Xp, nlev, ny, nx, nens, grid_u, Yp, rec, obgeo, scan, nobs, ob_begin, ob_end,
                                   0, ny, loc_mode, counters, st);
    if (rc == EXB_ERR_UNSUPPORTED && std::is_same<T, double>::value)
        rc = exb_state_update_mma_f64((double *)xm, (double *)Xp, nlev, ny, nx, nens, grid_u, (const double *)Yp,
                                      rec, obgeo, scan, nobs, ob_begin, ob_end, loc_mode, counters, st);
    if (rc != EXB_ERR_UNSUPPORTED) {
        cudaFreeAsync(scan, st);
        return rc;
    }
    // the kernel above, arithmetic in T: float32 beyond 103 members, float64 at 256
    SuParams p;
    p.xm = xm; p.Xp = Xp; p.Yp = Yp; p.grid_u = grid_u; p.rec = rec; p.geo = obgeo; p.scan = scan;
    p.counters = counters; p.npts = ny * nx; p.nobs = nobs; p.ob_begin = ob_begin; p.ob_end = ob_end;
    p.nlev = (int)nlev; p.ny = (int)ny; p.nx = (int)nx; p.nens = nens; p.loc_mode = loc_mode;
    rc = su_dispatch<T>(p, st);
    cudaFreeAsync(scan, st);
    return rc;
}

extern "C" int exb_state_update_f64(double *xm, double *Xp, int64_t nlev, int64_t ny, int64_t nx, int nens,
                                    const double *grid_u, const double *Yp, const double *rec, const double *obgeo,
                                    int64_t nobs, int64_t ob_begin, int64_t ob_end, int loc_mode,
                                    unsigned long long *counters, void *stream) {
    return state_update_impl<double>(xm, Xp, nlev, ny, nx, nens, grid_u, Yp, rec, obgeo, nobs, ob_begin, ob_end,
                                     loc_mode, counters, stream);
}
extern "C" int exb_state_update_f32(float *xm, float *Xp, int64_t nlev, int64_t ny, int64_t nx, int nens,
                                    const double *grid_u, const float *Yp, const double *rec, const double *obgeo,
                                    int64_t nobs, int64_t ob_begin, int64_t ob_end, int loc_mode,
                                    unsigned long long *counters, void *stream) {
    return state_update_impl<float>(xm, Xp, nlev, ny, nx, nens, grid_u, Yp, rec, obgeo, nobs, ob_begin, ob_end,
                                    loc_mode, counters, stream);
}

// Fused sweep of grid rows [y_begin, y_end) of a shard that holds FULL ensemble values: mean/perturbation split
// (assimilation.py:146-147), the serial update of ensrf.py:95-141 and the recombination (assimilation.py:168) in one
// pass over the touched rows.  Returns EXB_ERR_UNSUPPORTED when no fused variant exists for this ensemble size
// (callers then use exb_split_mean_pert / exb_state_update / exb_recombine).
template <typename T>
static int state_sweep_impl(T *X, int64_t nlev, int64_t ny, int64_t nx, int nens, const double *grid_u, const T *Yp,
                            const double *rec, const double *obgeo, int64_t nobs, int64_t ob_begin, int64_t ob_end,
                            int64_t y_begin, int64_t y_end, int loc_mode, unsigned long long *counters, void *stream,
                            ExbSweepPlan *plan = nullptr) {
    EXB_REQUIRE(X && grid_u && Yp && rec && obgeo, "null pointer");
    EXB_REQUIRE(nlev > 0 && ny > 0 && nx > 0 && nens >= 2 && nobs > 0, "bad sizes");
    EXB_REQUIRE(nlev < (1 << 30) && ny < (1 << 30) && nx < (1 << 30), "dimension too large");
    EXB_REQUIRE(0 <= ob_begin && ob_begin <= ob_end && ob_end <= nobs, "bad ob range");
    EXB_REQUIRE(0 <= y_begin && y_begin <= y_end && y_end <= ny, "bad row range");
    EXB_REQUIRE(loc_mode == EXB_LOC_NONE || loc_mode == EXB_LOC_GC, "bad loc_mode");
    if (ob_begin == ob_end || y_begin == y_end) return EXB_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (plan) {
        // scan records and candidate lists were built ahead, from the same geometry and assimilate flags
        if (plan->nlev != nlev || plan->ny != ny || plan->nx != nx || plan->nobs != nobs || plan->loc_mode != loc_mode ||
            plan->grid_u != grid_u || plan->obgeo != obgeo) {
            exb_set_error("exb_state_sweep_planned: the plan was built for another grid / observation set");
            return EXB_ERR_ARG;
        }
        EXB_CUDA(cudaStreamWaitEvent(st, plan->ready, 0));
        const int rc = exb_state_sweep_2p<T>(nullptr, X, nlev, ny, nx, nens, grid_u, Yp, rec, obgeo, plan->scan, nobs, ob_begin,
                                             ob_end, y_begin, y_end, loc_mode, counters, st, plan);
        cudaEventRecord(plan->used, st);
        plan->was_used = true;
        return rc;
    }
    float4 *scan = nullptr;
    EXB_CUDA(exb_malloc_async(&scan, (size_t)nobs * sizeof(float4), st));
    su_scan_records_kernel<<<(unsigned)ceil_div64(nobs, 256), 256, 0, st>>>(obgeo, rec, nobs, scan);
    exb_count_launches(1);
    const int rc = exb_state_sweep_2p<T>(nullptr, X, nlev, ny, nx, nens, grid_u, Yp, rec, obgeo, scan, nobs, ob_begin,
                                         ob_end, y_begin, y_end, loc_mode, counters, st);
    cudaFreeAsync(scan, st);
    return rc;
}

extern "C" int exb_state_sweep_planned_f64(void *plan, double *X, int64_t nlev, int64_t ny, int64_t nx, int nens,
                                           const double *grid_u, const double *Yp, const double *rec, const double *obgeo,
                                           int64_t nobs, int64_t ob_begin, int64_t ob_end, int64_t y_begin, int64_t y_end,
                                           int loc_mode, unsigned long long *counters, void *stream) {
    EXB_REQUIRE(plan, "null plan");
    return state_sweep_impl<double>(X, nlev, ny, nx, nens, grid_u, Yp, rec, obgeo, nobs, ob_begin, ob_end, y_begin, y_end,
                                    loc_mode, counters, stream, static_cast<ExbSweepPlan *>(plan));
}
extern "C" int exb_state_sweep_planned_f32(void *plan, float *X, int64_t nlev, int64_t ny, int64_t nx, int nens,
                                           const double *grid_u, const float *Yp, const double *rec, const double *obgeo,
                                           int64_t nobs, int64_t ob_begin, int64_t ob_end, int64_t y_begin, int64_t y_end,
                                           int loc_mode, unsigned long long *counters, void *stream) {
    EXB_REQUIRE(plan, "null plan");
    return state_sweep_impl<float>(X, nlev, ny, nx, nens, grid_u, Yp, rec, obgeo, nobs, ob_begin, ob_end, y_begin, y_end,
                                   loc_mode, counters, stream, static_cast<ExbSweepPlan *>(plan));
}

extern "C" int exb_state_sweep_f64(double *X, int64_t nlev, int64_t ny, int64_t nx, int nens, const double *grid_u,
                                   const double *Yp, const double *rec, const double *obgeo, int64_t nobs,
                                   int64_t ob_begin, int64_t ob_end, int64_t y_begin, int64_t y_end, int loc_mode,
                                   unsigned long long *counters, void *stream) {
    return state_sweep_impl<double>(X, nlev, ny, nx, nens, grid_u, Yp, rec, obgeo, nobs, ob_begin, ob_end, y_begin, y_end,
                                    loc_mode, counters, stream);
}
extern "C" int exb_state_sweep_f32(float *X, int64_t nlev, int64_t ny, int64_t nx, int nens, const double *grid_u,
                                   const float *Yp, const double *rec, const double *obgeo, int64_t nobs,
                                   int64_t ob_begin, int64_t ob_end, int64_t y_begin, int64_t y_end, int loc_mode,
                                   unsigned long long *counters, void *stream) {
    return state_sweep_impl<float>(X, nlev, ny, nx, nens, grid_u, Yp, rec, obgeo, nobs, ob_begin, ob_end, y_begin, y_end,
                                   loc_mode, counters, stream);
}
