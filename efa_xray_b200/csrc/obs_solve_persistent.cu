// Obs-space serial solve as ONE persistent cooperative kernel.
//
// The Nobs obs-space rows of the reference's augmented state (assimilation.py:149-150) only ever read
// other obs-space rows (ensrf.py:61-64, :95, :141), so they are evolved here on their own, in the
// reference's serial order, and leave behind one record per ob (ye_k and a few scalars) from which
// the state sweep (state_update.cu) can update every state row independently.
//
// Blocked right-looking form of the serial loop, panel width PS_PB: the obs k = b0..b0+PS_PB-1 of a panel are
// processed strictly in order with the panel's rows in registers (the only truly serial part of the whole
// analysis), then every later row j >= b0+PS_PB applies the panel's obs in order.  Rows j < k are never read
// again by the reference (ensrf.py:61-64 reads row k at step k only), so they are not updated; row k is frozen
// at step k and therefore ends up holding ye_k.
//
// One kernel runs the whole solve, without a launch per panel:
//   CTA 0            the PANEL WORKER: walks the panels b = 0, 1, ... ; for each one it loads the 64 rows of
//                    chunk b, applies the previous panel to them itself, runs the 64 serial steps with the rows
//                    in registers, publishes the records, and sets panel_done = b+1 (release).
//   CTAs 1..NW       TRAILING WORKERS: chunk p (rows 64p..64p+63) is owned by worker p mod NW for the whole
//                    solve.  A worker repeatedly takes its lowest chunk that is behind, loads it once, applies
//                    every panel that has been published since (up to PS_MAXBATCH, never the chunk's
//                    predecessor panel p-1, which the panel worker applies), stores it and publishes upto[p].
// The only serial chain left is the panel worker; trailing work and all launch gaps are off it.
// Cross-CTA data (rows, records, flags) is read with ld.global.cg after an acquire of the flag; the launch
// is cooperative, so every CTA is resident and the spin waits cannot deadlock.
//
// Inside a panel the chain per ob is kept short: pairwise localisation weights are evaluated in parallel
// before the loop; each row keeps its running sum and sum of squares (updated in O(1) per applied ob), so
// the active ob's variance (ensrf.py:69) needs no reduction; the active row is broadcast before its scalars
// are ready so that the other rows' dot products overlap the reciprocal / square-root chain.
#include "common.cuh"
#include <cooperative_groups.h>

#define PS_PB 64
#define PS_GS 8
#define PS_THREADS (PS_PB * PS_GS)
#define PS_MAXBATCH 8
#define PS_CTL_PAD 32

template <int N>
__device__ __forceinline__ double ps_group_sum(double v, unsigned mask) {
#pragma unroll
    for (int off = N / 2; off > 0; off >>= 1) v += __shfl_xor_sync(mask, v, off);
    return v;
}

__device__ __forceinline__ int ps_load_flag(const int *p) {
    const int v = *reinterpret_cast<const volatile int *>(p);
    __threadfence();
    return v;
}

struct PsShared {
    double geo[5][PS_PB];        // ux uy uz inv_hw a_max of the panel being applied / factorised
    double sc[3][PS_PB];         // innov c1 beta of the panel being applied
    int assim[PS_PB];
    int task[4];                 // broadcast slots
};

template <typename T>
struct PsArgs {
    T *Ym;
    T *Yp;
    const double *ob_value;
    const double *ob_error;
    const uint8_t *ob_assim;
    const double *ob_thr;        // outlier threshold per ob (QC instantiations only)
    const double *geo;
    double *rec;
    unsigned long long *counters;
    int *ctl;                    // [0] panel_done, [PS_CTL_PAD + p] upto[p]
    int64_t nobs;
    int nens, loc_mode, npanels;
};

// rows of chunk p into registers (ld.cg: the rows are written by other CTAs during this launch)
template <typename T, int MC>
__device__ __forceinline__ void ps_load_rows(const PsArgs<T> &a, int64_t j, bool valid, int s, T (&x)[MC], double &mj) {
#pragma unroll
    for (int i = 0; i < MC; ++i) {
        const int m = s + PS_GS * i;
        x[i] = (valid && m < a.nens) ? __ldcg(a.Yp + j * a.nens + m) : (T)0;
    }
    mj = valid ? (double)__ldcg(a.Ym + j) : 0.0;
}

template <typename T, int MC>
__device__ __forceinline__ void ps_store_rows(const PsArgs<T> &a, int64_t j, bool valid, int s, const T (&x)[MC], double mj) {
    if (!valid) return;
#pragma unroll
    for (int i = 0; i < MC; ++i) {
        const int m = s + PS_GS * i;
        if (m < a.nens) a.Yp[j * a.nens + m] = x[i];
    }
    if (s == 0) a.Ym[j] = (T)mj;
}

// Apply the 64 (frozen) obs of panel b, in order, to the rows held in registers.  CTA-wide call.
template <typename T, int MC>
__device__ __forceinline__ void ps_apply_panel(const PsArgs<T> &a, PsShared &sh, int b, bool valid, double ux, double uy,
                                               double uz, T (&x)[MC], double &mj, unsigned long long &npairs) {
    const int tid = threadIdx.x, s = tid % PS_GS, lane = tid % 32;
    const int gbase = lane & ~(PS_GS - 1);
    const unsigned gmask = 0xffu << gbase;
    const int64_t nobs = a.nobs, b0 = (int64_t)b * PS_PB;
    __syncthreads();                                  // previous users of sh are done
    if (tid < PS_PB) {
        const int64_t kk = b0 + tid;                  // panels that get applied are always full
        sh.geo[0][tid] = a.geo[GEO_UX * nobs + kk];
        sh.geo[1][tid] = a.geo[GEO_UY * nobs + kk];
        sh.geo[2][tid] = a.geo[GEO_UZ * nobs + kk];
        sh.geo[3][tid] = a.geo[GEO_INVHW * nobs + kk];
        sh.geo[4][tid] = a.geo[GEO_AMAX * nobs + kk];
        sh.sc[0][tid] = __ldcg(a.rec + REC_INNOV * nobs + kk);
        sh.sc[1][tid] = __ldcg(a.rec + REC_C1 * nobs + kk);
        sh.sc[2][tid] = __ldcg(a.rec + REC_BETA * nobs + kk);
        sh.assim[tid] = __ldcg(a.rec + REC_ASSIM * nobs + kk) != 0.0;
    }
    __syncthreads();
    for (int k0 = 0; k0 < PS_PB; k0 += PS_GS) {
        const int kt = k0 + s;                        // each lane of the group tests one ob against this row
        double wk = 0.0;
        if (valid && sh.assim[kt]) {
            wk = 1.0;
            if (a.loc_mode == EXB_LOC_GC)
                wk = loc_weight(hav_a(ux, uy, uz, sh.geo[0][kt], sh.geo[1][kt], sh.geo[2][kt]), sh.geo[3][kt], sh.geo[4][kt]);
        }
        if (!__any_sync(0xffffffffu, wk != 0.0)) continue;
#pragma unroll
        for (int q = 0; q < PS_GS; ++q) {
            const double w = __shfl_sync(0xffffffffu, wk, gbase + q);
            if (w != 0.0) {
                const int k = k0 + q;
                const T *yrow = a.Yp + (b0 + k) * a.nens;
                T ye[MC];
                T d0 = 0, d1 = 0;
#pragma unroll
                for (int i = 0; i < MC; ++i) {
                    const int m = s + PS_GS * i;
                    ye[i] = (m < a.nens) ? __ldcg(yrow + m) : (T)0;
                }
#pragma unroll
                for (int i = 0; i < MC; i += 2) {
                    d0 += x[i] * ye[i];
                    if (i + 1 < MC) d1 += x[i + 1] * ye[i + 1];
                }
                const double dot = ps_group_sum<PS_GS>((double)(d0 + d1), gmask);
                const double kmat = w * dot * sh.sc[1][k];          // loc * kcov / kdenom, ensrf.py:115-119
                mj += kmat * sh.sc[0][k];                           // ensrf.py:130
                const T f = (T)(sh.sc[2][k] * kmat);                // ensrf.py:136
#pragma unroll
                for (int i = 0; i < MC; ++i) x[i] -= f * ye[i];     // ensrf.py:141
                if (s == 0) npairs++;
            }
        }
    }
}

struct PsObScalars {
    double innov, c1, beta, sum, sq;
};

// |innov| > t sqrt(kdenom) in float64 with a correctly rounded sqrt (DESIGN.md section 4.7).  Not inlined: inlined, the
// threshold load and the sqrt's slow path added spills to the instantiations above 152 members.
__device__ __noinline__ bool ps_outlier(const double *thr, int64_t k, double innov, double kdenom) {
    return fabs(innov) > thr[k] * sqrt(kdenom);
}

// QC: outlier check of every assimilated ob against its in-loop prior (DESIGN.md section 4.7).  The panel worker hands
// the rest of its panel zero scalars for a rejected ob (an exact identity update) and records it as not assimilated,
// so the trailing workers skip it.
template <typename T, int MC, bool QC>
__global__ void __launch_bounds__(PS_THREADS, 1) obs_solve_persistent_kernel(const PsArgs<T> a) {
    __shared__ PsShared sh;
    __shared__ T s_ye[2][PS_GS * MC];
    __shared__ PsObScalars s_ob[2];
    __shared__ double s_W[PS_PB * PS_PB];
    __shared__ int s_flag[PS_PB];

    const int tid = threadIdx.x;
    const int g = tid / PS_GS, s = tid % PS_GS, lane = tid % 32;
    const unsigned gmask = 0xffu << (lane & ~(PS_GS - 1));
    const int64_t nobs = a.nobs;
    const int nens = a.nens;
    int *panel_done = a.ctl;
    int *upto = a.ctl + PS_CTL_PAD;
    unsigned long long npairs = 0;
    T x[MC];
    double mj;

    if (blockIdx.x == 0) {
        // =========================== PANEL WORKER ===========================
        const double inv_n = 1.0 / (double)nens;
        for (int b = 0; b < a.npanels; ++b) {
            const int64_t b0 = (int64_t)b * PS_PB;
            const int64_t j = b0 + g;
            const bool valid = j < nobs;
            const int nb = (int)((nobs - b0) < PS_PB ? (nobs - b0) : PS_PB);
            if (b >= 2) {                                  // chunk b must carry panels 0..b-2 (its owner's job)
                if (tid == 0) {
                    while (ps_load_flag(upto + b) < b - 1) __nanosleep(64);
                }
                __syncthreads();
                __threadfence();
            }
            double ux = 0, uy = 0, uz = 0;
            if (valid) { ux = a.geo[GEO_UX * nobs + j]; uy = a.geo[GEO_UY * nobs + j]; uz = a.geo[GEO_UZ * nobs + j]; }
            ps_load_rows<T, MC>(a, j, valid, s, x, mj);
            if (b >= 1) ps_apply_panel<T, MC>(a, sh, b - 1, valid, ux, uy, uz, x, mj, npairs);
            __syncthreads();

            // ---- set-up of the panel: geometry, pair weights, flags, row statistics ----
            if (tid < PS_PB) {
                const int64_t kk = (b0 + tid < nobs) ? b0 + tid : nobs - 1;
                sh.geo[0][tid] = a.geo[GEO_UX * nobs + kk];
                sh.geo[1][tid] = a.geo[GEO_UY * nobs + kk];
                sh.geo[2][tid] = a.geo[GEO_UZ * nobs + kk];
                sh.geo[3][tid] = a.geo[GEO_INVHW * nobs + kk];
                sh.geo[4][tid] = a.geo[GEO_AMAX * nobs + kk];
                s_flag[tid] = (b0 + tid < nobs) ? (a.ob_assim[kk] != 0) : 0;
            }
            __syncthreads();
            for (int idx = tid; idx < PS_PB * PS_PB; idx += PS_THREADS) {
                const int k = idx / PS_PB, jj = idx % PS_PB;
                double w = 0.0;
                if (jj > k && jj < nb && s_flag[k]) {
                    w = 1.0;
                    if (a.loc_mode == EXB_LOC_GC)
                        w = loc_weight(hav_a(sh.geo[0][jj], sh.geo[1][jj], sh.geo[2][jj], sh.geo[0][k], sh.geo[1][k], sh.geo[2][k]),
                                       sh.geo[3][k], sh.geo[4][k]);
                }
                s_W[idx] = w;
            }
            double my_val = 0.0, my_err = 1.0, my_serr = 1.0, my_wself = 1.0;
            if (valid && s == 0) {
                my_val = a.ob_value[j];
                my_err = a.ob_error[j];
                my_serr = sqrt(my_err);
                my_wself = (a.loc_mode == EXB_LOC_GC) ? loc_weight(0.0, sh.geo[3][g], sh.geo[4][g]) : 1.0;
            }
            // running sum and sum of squares of this row
            double rs, rq;
            {
                double s0 = 0.0, q0 = 0.0;
#pragma unroll
                for (int i = 0; i < MC; ++i) { const double v = (double)x[i]; s0 += v; q0 += v * v; }
                rs = ps_group_sum<PS_GS>(s0, gmask);
                rq = ps_group_sum<PS_GS>(q0, gmask);
            }
            __syncthreads();

            // ---- the serial chain ----
            for (int k = 0; k < nb; ++k) {
                const int buf = k & 1;
                if (g == k) {
#pragma unroll
                    for (int i = 0; i < MC; ++i) s_ye[buf][s * MC + i] = x[i];
                }
                __syncthreads();                                            // (A) ye_k visible
                const bool act = s_flag[k] != 0;
                const double w = (g > k && valid && act) ? s_W[k * PS_PB + g] : 0.0;
                T ye[MC];
                double dot = 0.0;
                if (g == k) {
                    if (s == 0) {
                        // ensrf.py:63-70, :86, :91, :95, :135 from the running statistics of the row
                        const int64_t kk = b0 + k;
                        const double mean = rs * inv_n;
                        const double varye = fmax(rq * inv_n - mean * mean, 0.0);       // np.var, ddof 0
                        const double innov = my_val - mj;
                        const double kdenom = varye + my_err;
                        const double c1 = 1.0 / ((double)(nens - 1) * kdenom);
                        const double beta = 1.0 / (1.0 + my_serr * rsqrt(kdenom));      // 1/(1+sqrt(R/kdenom))
                        bool rej = false;                                               // |innov| > t sqrt(kdenom)
                        if constexpr (QC) rej = act && ps_outlier(a.ob_thr, kk, innov, kdenom);
                        s_ob[buf].innov = rej ? 0.0 : innov; s_ob[buf].c1 = rej ? 0.0 : c1; s_ob[buf].beta = beta;
                        s_ob[buf].sum = rs; s_ob[buf].sq = rq;
                        a.rec[REC_PRIOR_MEAN * nobs + kk] = mj;                          // ensrf.py:66
                        a.rec[REC_PRIOR_VAR * nobs + kk] = varye;                        // ensrf.py:70
                        a.rec[REC_INNOV * nobs + kk] = innov;
                        a.rec[REC_C1 * nobs + kk] = rej ? 0.0 : c1;
                        a.rec[REC_BETA * nobs + kk] = beta;
                        a.rec[REC_ASSIM * nobs + kk] = act && !rej ? 1.0 : 0.0;
                        if (act && !rej) {
                            // the ob's own row: weight at distance 0, kcov = ye.ye/(N-1)   (ensrf.py:144-147)
                            const double kmat = my_wself * rq * c1;
                            const double shrink = 1.0 - beta * kmat;
                            a.rec[REC_POST_MEAN * nobs + kk] = mj + kmat * innov;
                            a.rec[REC_POST_VAR * nobs + kk] = varye * shrink * shrink;
                            if (my_wself != 0.0) npairs++;
                        } else {
                            a.rec[REC_POST_MEAN * nobs + kk] = nan("");
                            a.rec[REC_POST_VAR * nobs + kk] = nan("");
                        }
                    }
                } else if (w != 0.0) {
                    T d0 = 0, d1 = 0, d2 = 0, d3 = 0;
#pragma unroll
                    for (int i = 0; i < MC; ++i) ye[i] = s_ye[buf][s * MC + i];
#pragma unroll
                    for (int i = 0; i < MC; i += 4) {
                        d0 += x[i] * ye[i];
                        if (i + 1 < MC) d1 += x[i + 1] * ye[i + 1];
                        if (i + 2 < MC) d2 += x[i + 2] * ye[i + 2];
                        if (i + 3 < MC) d3 += x[i + 3] * ye[i + 3];
                    }
                    dot = ps_group_sum<PS_GS>((double)((d0 + d1) + (d2 + d3)), gmask);
                }
                if (!act) continue;                                         // uniform: nothing to apply
                __syncthreads();                                            // (B) scalars of ob k visible
                if (w != 0.0) {
                    const double kmat = w * dot * s_ob[buf].c1;             // loc * kcov / kdenom, ensrf.py:115-119
                    mj += kmat * s_ob[buf].innov;                           // ensrf.py:130
                    const double fd = s_ob[buf].beta * kmat;                // ensrf.py:136
                    const T f = (T)fd;
#pragma unroll
                    for (int i = 0; i < MC; ++i) x[i] -= f * ye[i];         // ensrf.py:141
                    rs -= fd * s_ob[buf].sum;
                    rq += fd * (fd * s_ob[buf].sq - 2.0 * dot);
                    if (s == 0) npairs++;
                }
            }
            ps_store_rows<T, MC>(a, j, valid, s, x, mj);
            __threadfence();
            __syncthreads();
            if (tid == 0) { *reinterpret_cast<volatile int *>(panel_done) = b + 1; }
        }
    } else {
        // =========================== TRAILING WORKER ===========================
        const int NW = gridDim.x - 1, w = blockIdx.x - 1;
        if (w >= a.npanels) return;
        extern __shared__ int s_upto[];                  // progress of this worker's chunks (slot i -> chunk w + i*NW)
        const int nmine = (a.npanels - w + NW - 1) / NW;
        for (int i = tid; i < nmine; i += PS_THREADS) s_upto[i] = 0;
        __syncthreads();
        int first = 0;                                   // (thread 0 only) slots below `first` are finished
        while (true) {
            if (tid == 0) {
                int slot = -1, tgt = 0;
                while (true) {
                    while (first < nmine && s_upto[first] >= (w + first * NW) - 1) ++first;
                    if (first >= nmine) break;                         // every chunk of this worker is finished
                    const int done = ps_load_flag(panel_done);
                    for (int i = first; i < nmine; ++i) {
                        const int p = w + i * NW;
                        const int t = done < p - 1 ? done : p - 1;     // never the predecessor panel p-1
                        if (s_upto[i] < t) { slot = i; tgt = t; break; }
                    }
                    if (slot >= 0) break;
                    __nanosleep(200);
                }
                sh.task[0] = slot;
                sh.task[1] = tgt;
            }
            __syncthreads();
            const int slot = sh.task[0];
            if (slot < 0) break;
            const int p = w + slot * NW;
            const int from = s_upto[slot];
            int to = sh.task[1];
            if (to > from + PS_MAXBATCH) to = from + PS_MAXBATCH;
            __threadfence();
            const int64_t j = (int64_t)p * PS_PB + g;
            const bool valid = j < nobs;
            double ux = 0, uy = 0, uz = 0;
            if (valid) { ux = a.geo[GEO_UX * nobs + j]; uy = a.geo[GEO_UY * nobs + j]; uz = a.geo[GEO_UZ * nobs + j]; }
            ps_load_rows<T, MC>(a, j, valid, s, x, mj);
            for (int b = from; b < to; ++b) ps_apply_panel<T, MC>(a, sh, b, valid, ux, uy, uz, x, mj, npairs);
            ps_store_rows<T, MC>(a, j, valid, s, x, mj);
            __threadfence();
            __syncthreads();                             // also orders the reads of sh.task above before the next decision
            if (tid == 0) {
                s_upto[slot] = to;
                *reinterpret_cast<volatile int *>(upto + p) = to;
            }
        }
    }
    if (a.counters) {
        npairs = ps_group_sum<32>((double)npairs, 0xffffffffu) + 0.5;      // exact for < 2^53
        if (lane == 0 && npairs) atomicAdd(&a.counters[0], npairs);
    }
}

template <typename T, int MC>
static int ps_launch(PsArgs<T> &a, cudaStream_t st) {
    const void *kernel = a.ob_thr ? (const void *)obs_solve_persistent_kernel<T, MC, true>
                                  : (const void *)obs_solve_persistent_kernel<T, MC, false>;
    int dev = 0, sms = 0, coop = 0, per_sm = 0;
    EXB_CUDA(cudaGetDevice(&dev));
    EXB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    EXB_CUDA(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
    if (!coop) {
        exb_set_error("obs_solve_persistent: device %d does not support cooperative launch", dev);
        return EXB_ERR_UNSUPPORTED;
    }
    // A trailing worker keeps one progress word per chunk it owns in dynamic shared memory.  It is sized for one CTA
    // per SM, the fewest workers the launch can have; more CTAs per SM only give each worker fewer chunks.
    const auto clamp_grid = [&](int g) { return g > a.npanels + 1 ? a.npanels + 1 : (g < 2 ? 2 : g); };
    int grid = clamp_grid(sms);
    const size_t smem = sizeof(int) * (size_t)((a.npanels + grid - 2) / (grid - 1));
    cudaFuncAttributes fa;
    EXB_CUDA(cudaFuncGetAttributes(&fa, kernel));
    if (fa.sharedSizeBytes + smem > 48 * 1024)
        EXB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    EXB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, PS_THREADS, smem));
    if (per_sm < 1) {
        exb_set_error("obs_solve_persistent: a CTA of %d threads with %zu bytes of shared memory does not fit an SM",
                      PS_THREADS, fa.sharedSizeBytes + smem);
        return EXB_ERR_UNSUPPORTED;
    }
    grid = clamp_grid(sms * per_sm);
    int *ctl = nullptr;
    const size_t ctl_bytes = sizeof(int) * (PS_CTL_PAD + (size_t)a.npanels + 1);
    EXB_CUDA(exb_malloc_async(&ctl, ctl_bytes, st));
    EXB_CUDA(cudaMemsetAsync(ctl, 0, ctl_bytes, st));
    a.ctl = ctl;
    void *params[] = {(void *)&a};
    cudaError_t e = cudaLaunchCooperativeKernel(kernel, dim3(grid), dim3(PS_THREADS), params, smem, st);
    exb_count_launches(1);
    cudaFreeAsync(ctl, st);
    if (e != cudaSuccess) {
        exb_set_error("obs_solve_persistent: cooperative launch failed -> %s", cudaGetErrorString(e));
        return EXB_ERR_CUDA;
    }
    return exb_check_launch("obs_solve_persistent_kernel");
}

template <typename T>
int exb_obs_solve_persistent(T *Ym, T *Yp, const double *ob_value, const double *ob_error, const uint8_t *ob_assim,
                             const double *ob_thr, const double *geo, int64_t nobs, int nens, int loc_mode, double *rec,
                             unsigned long long *counters, cudaStream_t st) {
    PsArgs<T> a;
    a.Ym = Ym; a.Yp = Yp; a.ob_value = ob_value; a.ob_error = ob_error; a.ob_assim = ob_assim; a.ob_thr = ob_thr;
    a.geo = geo;
    a.rec = rec; a.counters = counters; a.ctl = nullptr; a.nobs = nobs; a.nens = nens; a.loc_mode = loc_mode;
    a.npanels = (int)((nobs + PS_PB - 1) / PS_PB);
    const int mc = (nens + PS_GS - 1) / PS_GS;
#define PS_DISPATCH(M) if (mc <= M) return ps_launch<T, M>(a, st)
    PS_DISPATCH(4);
    PS_DISPATCH(7);
    PS_DISPATCH(13);
    PS_DISPATCH(19);
    PS_DISPATCH(25);
    PS_DISPATCH(32);
#undef PS_DISPATCH
    return EXB_ERR_UNSUPPORTED;
}

template int exb_obs_solve_persistent<double>(double *, double *, const double *, const double *, const uint8_t *,
                                              const double *, const double *, int64_t, int, int, double *, unsigned long long *,
                                              cudaStream_t);
template int exb_obs_solve_persistent<float>(float *, float *, const double *, const double *, const uint8_t *,
                                             const double *, const double *, int64_t, int, int, double *, unsigned long long *,
                                             cudaStream_t);
