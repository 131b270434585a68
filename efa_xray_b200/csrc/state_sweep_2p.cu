// State sweep, two-phase FP64 tensor-core version (production path for ensembles of up to 103 members).
//
// Same mathematics as state_update_mma.cu (read its header first: blocked 8-ob form of ensrf.py:95-141 on
// mma.sync.m8n8k4.f64, the ensemble mean carried as a pseudo-member column).  What changes is who does the scalar FP64
// work.  The Gaspari-Cohn weights (observation.py:117-130, ~60 scalar FP64 instructions per (grid point, ob) pair) and
// the DMMAs share one issue port per SM sub-partition.  Producer warps that evaluate the weights WHILE consumer warps
// issue DMMAs must be given a sub-partition of their own, whose tensor pipe then sits idle: round 1's kernel did this
// with four producers and twelve consumers (ceiling 75 % of the FP64 tensor peak, measured 58 %; removed since).
// Here the two kinds of work never run at the same time:
//   phase A  all 16 warps of the CTA: scan the patch's candidate obs (fp32 cap test over the coarse tile's list),
//            evaluate omega[ob][grid point] = beta c1 GC(d) for batches of 8 obs and the batch's 8x8 Gram matrix, and
//            write one block per batch to a per-CTA scratch area in global memory (L2-resident);
//   phase B  the same 16 warps as consumers -- four per SM sub-partition, 8 state rows each, in registers for the whole
//            patch -- run
//            g = X Y^T -> 8-step recurrence -> X -= E Y  per batch; the stages are filled by bulk copies (cp.async.bulk,
//            completion on the stage's mbarrier by transaction bytes) that the warps take turns issuing: the 8 ye rows
//            of the batch straight from a padded copy of the ob ensembles (pseudo-member column and zero padding
//            already in place) and the batch's omega/Gram block.
// Every sub-partition's tensor pipe works in phase B and nothing but scalar FP64 runs in phase A.
// Measured (scratch/ubench/consumer_ubench.cu, gpurun_out/r02b/c_consumer_ubench.txt): the consumer loop alone runs at
// 27 clocks per (row, batch) as pure DMMA (97 % of the 16-clock issue interval), 29 with the shuffles, 32.5 with the
// recurrence at 16 warps; 15 warps are no faster per warp than 16 (the sub-partition with four warps sets the pace),
// a single accumulator chain in step 1 and folding the cross-block correction into the DMMA accumulator give 31.6.
// The kernel is persistent (one CTA per SM, patches handed out by a ticket counter in heaviest-first order), a patch's
// candidates are processed in chunks of at most S2_CAND so that the scratch area is bounded; between the chunks of one
// patch the consumers park their rows in the scratch area (phase A needs the registers).
//
// Shared-memory staging of the ye rows: row q of a batch starts at q*YST + (q>>1)*4 doubles.  With YST = 8 mod 16 the
// B-operand loads of step 1 (rows n, n+1 per quarter warp, 64 contiguous bytes each) and of step 3 (rows c = 0..3 per
// half warp, 4 consecutive doubles each) are both free of bank conflicts without an XOR swizzle of the columns, so the
// rows can be copied in as they are.
#include "common.cuh"
#include <cstdio>
#include <cstdlib>
#include <cstring>

// Warps per CTA: one CTA per SM, four warps per sub-partition, 128 registers per thread, 128 state rows per patch (a
// 17th warp would put five warps on one sub-partition's 16 K registers: 96 per thread).  Two CTAs of 8 warps per SM,
// so that one CTA's phase A overlaps the other's phase B, measured slower (DESIGN.md 4.3): the two kinds of work share
// the FP64 issue port, and the per-patch work is spread over half as many rows.
// Every warp is a consumer in phase B and takes turns issuing the copies.
#define S2_NW 16
#define S2_CAND 2048                   // candidate capacity of a chunk (256 batches)
#define S2_MAXSTAGES 16

struct S2Params {
    void *xm;                         // nullptr: fused mean/perturbation split + recombination   (storage type TS)
    void *Xp;                         // state rows, storage type TS (double or float); arithmetic is always double
    const double *Yw;                 // [nobs + 1][8*NT3]: ye rows widened to double, zero padded, pseudo-member column
                                      // -innov/beta in the last column; row nobs is all zeros
    const double *grid_u;
    const double *rec;
    const double *geo;
    const float4 *scan;               // (ux, uy, uz, theta) per ob; theta < 0: never a candidate
    const int64_t *tile_off;          // candidate lists per coarse tile (nullptr: walk the ob range)
    const int *tile_list;
    unsigned long long *counters;
    int *ticket;                      // patch dispenser
    double *scratch;                  // per CTA: S2_CAND/8 blocks of blk_doubles, then the parked rows
    const int *abort_flag;            // watchdog word of the obs-space solve that produced the records (may be null)
    unsigned long long *prof;         // EXB_S2_PROF=1: clocks of warp 0 per phase, summed over CTAs (null: off)
    int64_t npts, nobs, ob_begin, ob_end, scratch_stride;
    int nlev, ny, nx, nens;
    int y_begin, y_end;               // grid rows [y_begin, y_end) of the shard are swept by this launch
    int pr0, npr, pr_eq;              // first patch row / number of patch rows of this launch, patch row of the equator
    int ty, tx, ntx, nctx;            // patch shape, patches along x, coarse tiles along x
    int G, Lc, nlc;
    int loc_mode;
    int nstages, stage_doubles, blk_doubles, npatches;
    ExbLocConst kloc;                 // constants of the localisation weight (parameter block = constant bank)
};

__device__ __forceinline__ void s2_dmma(double &c0, double &c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
        : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
// volatile variant: keeps the program order of a sequence of DMMAs (the compiler may not re-pair them)
__device__ __forceinline__ void s2_dmma_v(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
__device__ __forceinline__ unsigned s2_smem(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void s2_mbar_init(unsigned long long *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(s2_smem(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void s2_mbar_arrive(unsigned long long *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(s2_smem(bar)) : "memory");
}
__device__ __forceinline__ void s2_mbar_arrive_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(s2_smem(bar)), "r"(bytes) : "memory");
}
// (two textually separate copies so that profiler samples of consumers waiting for data and of the issuer waiting
// for a free stage land on different source lines)
__device__ __forceinline__ void s2_mbar_wait_full(unsigned long long *bar, unsigned parity) {
    unsigned ok = 0;
    const unsigned a = s2_smem(bar);
    do {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(ok) : "r"(a), "r"(parity) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void s2_mbar_wait_empty(unsigned long long *bar, unsigned parity) {
    unsigned ok = 0;
    const unsigned a = s2_smem(bar);
    do {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(ok) : "r"(a), "r"(parity) : "memory");
    } while (!ok);
}
// global -> shared bulk copy (TMA engine, 1-D), completion counted in bytes on an mbarrier of this CTA
__device__ __forceinline__ void s2_bulk_g2s(void *dst_smem, const void *src_gmem, unsigned bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 ::"r"(s2_smem(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(s2_smem(bar)) : "memory");
}

// v[c] for a lane-dependent c in 0..3 as three predicated selects (written with ternaries the compiler emits divergent
// branches here, which serialise the four lanes of every row)
__device__ __forceinline__ double s2_sel4(double v0, double v1, double v2, double v3, int c) {
    double lo, hi, r;
    asm("{\n.reg .pred p, q;\nsetp.ne.s32 p, %3, 0;\nsetp.ne.s32 q, %4, 0;\n"
        "selp.f64 %0, %6, %5, p;\nselp.f64 %1, %8, %7, p;\nselp.f64 %2, %1, %0, q;\n}\n"
        : "=&d"(lo), "=&d"(hi), "=d"(r) : "r"(c & 1), "r"(c & 2), "d"(v0), "d"(v1), "d"(v2), "d"(v3));
    return r;
}

// read-only global load the compiler may not sink towards its use (prefetches one batch ahead stay where they are)
__device__ __forceinline__ double s2_ldg_now(const double *p) {
    double v;
    asm volatile("ld.global.nc.f64 %0, [%1];\n" : "=d"(v) : "l"(p));
    return v;
}

template <int NT3> __host__ __device__ constexpr int s2_yst() { return ((8 * NT3) % 16 == 8) ? 8 * NT3 : 8 * NT3 + 8; }
// doubles of the ye-row region of a stage: 8 rows at q*YST + (q>>1)*4
template <int NT3> __host__ __device__ constexpr int s2_ydoubles() { return 8 * s2_yst<NT3>() + 16; }

// Columns of a row of Yw and of the state rows in registers.  Lane c of a row holds columns 2c and 2c+1 of every
// 8-column tile t, as x[2t] and x[2t+1], and k-step h of tile t in step 1 covers the columns 2c+h of the four lanes.
// s2_slot gives the member slot that column 2c+h of tile t holds: slot m < nens is member m, slot 8*NT3-1 the
// pseudo-member (the mean), any other slot a zero pad.  LK is the number of k-steps of the last tile that carry members
// (nens - 8*(NT3-1) members there: none -> 0, 1..4 -> 1, 5..7 -> 2).  With LK == 1 the last tile is stored
// transposed, slot 4h+c in column 2c+h: its members sit in the even columns, the odd ones hold the pads and the mean,
// and step 1 and the Gram matrix skip that k-step.  Every tile before the last is in member order.
template <int NT3, int LK> __host__ __device__ constexpr int s2_slot(int t, int c, int h) {
    return (LK == 1 && t == NT3 - 1) ? 8 * t + 4 * h + c : 8 * t + 2 * c + h;
}
template <int NT3> static int s2_last_ksteps(int nens) {
    const int r = nens - 8 * (NT3 - 1);
    return r <= 0 ? 0 : r <= 4 ? 1 : 2;
}

// Tail of a batch block (after om[G][8]), in doubles: what phase B reads besides the weights, packed for vector loads.
//   [S2_TCORR + 4n + c]  B operand of the correction DMMA of lane (n, c): G[n][c] for n >= 4, zero for n < 4 (so the
//                        first 8 doubles are zeros: inactive rows read them as their weights)
//   [S2_TREC ..+12]      the recurrence's coefficients G10 G20 G21 G30 G31 G32 G54 G64 G65 G74 G75 G76
//   [S2_TMASK]           low 32 bits: bit w set when warp w has a row with a non-zero weight for an ob of the batch
#define S2_TCORR 0
#define S2_TREC 32
#define S2_TMASK 44

// Stage layout (doubles): y rows [s2_ydoubles] | block = om[G][8] (point-major) | tail[64]
template <int NT3, int LK, typename TS>
__global__ void __launch_bounds__(S2_NW * 32, 1) state_sweep_2p_kernel(const S2Params p) {
    constexpr int NW = S2_NW;
    constexpr int NTH = NW * 32;             // threads per CTA
    constexpr int ROWS = NW * 8;             // state rows per CTA
    constexpr int SCAN = 2 * NTH;            // list entries per scan step (2 per thread)
    TS *const gXp = static_cast<TS *>(p.Xp);
    TS *const gxm = static_cast<TS *>(p.xm);
    constexpr int YST = s2_yst<NT3>();
    constexpr int YD = s2_ydoubles<NT3>();
    constexpr int YW = 8 * NT3;              // doubles per row of Yw
    constexpr int PC = 8 * NT3 - 1;          // column of the pseudo-member (the mean)

    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *s_ring = reinterpret_cast<double *>(smem_raw);                                   // [nstages][stage_doubles]
    double *s_gu = s_ring + (size_t)p.nstages * p.stage_doubles;                             // [3][ROWS]
    double *s_sob = s_gu + 3 * ROWS;                                                      // [NW][8][6]
    double2 *s_xch = reinterpret_cast<double2 *>(s_sob + NW * 48);                          // [NW][32]
    unsigned long long *s_full = reinterpret_cast<unsigned long long *>(s_xch + NW * 32); // [S2_MAXSTAGES]
    unsigned long long *s_empty = s_full + S2_MAXSTAGES;                                      // [S2_MAXSTAGES]
    int *s_cand = reinterpret_cast<int *>(s_empty + S2_MAXSTAGES);                            // [S2_CAND]
    int *s_gwarps = s_cand + S2_CAND;                                                         // [ROWS]
    int *s_wcnt = s_gwarps + ROWS;                                                         // [NW]
    int *s_misc = s_wcnt + NW;                                                             // [4]
    float *s_bound = reinterpret_cast<float *>(s_misc + 4);                                   // [4]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int c = lane & 3, n = lane >> 2;
    const int G = p.G, Lc = p.Lc, nens = p.nens;
    const int S = p.nstages, SD = p.stage_doubles, BLK = p.blk_doubles;
    const unsigned lt = (1u << lane) - 1u;
    (void)lt;

    // ---- once per CTA ------------------------------------------------------------------------------------
    if (tid == 0) s_misc[0] = p.abort_flag ? *reinterpret_cast<const volatile int *>(p.abort_flag) : 0;
    if (tid < S) {
        s2_mbar_init(s_full + tid, 1);           // the issuer's arrive.expect_tx; the copies complete the bytes
        s2_mbar_init(s_empty + tid, NW);      // one arrive per consumer warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
    __syncthreads();
    if (s_misc[0] != 0) return;                  // the records are invalid (watchdog): leave the state alone

    double *const blocks = p.scratch + (size_t)blockIdx.x * p.scratch_stride;
    double *const xsave = blocks + (size_t)(S2_CAND / 8) * BLK;
    const bool fused = p.xm == nullptr;
    unsigned gbatch = 0;                         // batches that have gone through the ring so far (same in every thread)
    unsigned long long npairs = 0;

    // phase clocks of thread 0 (only with p.prof): 0 patch setup, 1 scan, 2 blocks, 3 rows in/out, 4 phase B, 5 barriers;
    // prof[10]: batches
    // (the sums live in shared memory: as a register array they would take registers or stack from the loops)
    __shared__ long long pacc[10];
    long long pt0 = 0;
#define S2_TICK(slot) do { if (p.prof && tid == 0) { const long long t_ = clock64(); pacc[slot] += t_ - pt0; pt0 = t_; } } while (0)
    if (p.prof && tid == 0) {
        for (int i = 0; i < 10; ++i) pacc[i] = 0;
        pt0 = clock64();
    }
    for (;;) {
        // ---- next patch -----------------------------------------------------------------------------------
        __syncthreads();                          // everybody is done with the previous patch's shared state
        S2_TICK(5);
        if (tid == 0) s_misc[1] = atomicAdd(p.ticket, 1);
        __syncthreads();
        const int tk = s_misc[1];
        if (tk >= p.npatches) break;
        const int lc = tk % p.nlc;
        const int tile = tk / p.nlc;
        // Patch rows are issued heaviest first: on a lat-lon grid the rows next to the poles meet the most candidate
        // obs per unit of area, so they must not be the tail of the launch.  Rows are taken alternately from the two
        // ends of the launch's range when it straddles the equator, else from the poleward end.
        int prow;
        {
            const int r = tile / p.ntx, nr = p.npr, eq = p.pr_eq;
            if (eq < 0) prow = p.pr0 + r;
            else if (eq <= p.pr0) prow = p.pr0 + nr - 1 - r;
            else if (eq >= p.pr0 + nr) prow = p.pr0 + r;
            else prow = (r & 1) ? p.pr0 + nr - 1 - (r >> 1) : p.pr0 + (r >> 1);
        }
        const int pcol = tile % p.ntx;
        const int y0 = prow * p.ty, x0 = pcol * p.tx;
        const int l0 = lc * Lc;

        if (tid < G) {
            const int gy = y0 + tid / p.tx, gx = x0 + tid % p.tx;
            const bool ok = gy >= p.y_begin && gy < p.y_end && gx < p.nx;
            const int cy = min(max(gy, p.y_begin), p.y_end - 1), cx = min(gx, p.nx - 1);
            const int64_t pt = (int64_t)cy * p.nx + cx;
            s_gu[tid] = p.grid_u[pt];
            s_gu[ROWS + tid] = p.grid_u[p.npts + pt];
            s_gu[2 * ROWS + tid] = p.grid_u[2 * p.npts + pt];
            // the warps that hold the point's rows of this level chunk (row slots tid*Lc + l, l < the chunk's levels);
            // zero for a point outside the launch's rows or the grid
            const int r0 = tid * Lc, r1 = r0 + min(Lc, p.nlev - l0) - 1;
            s_gwarps[tid] = ok ? (int)(((2u << (r1 >> 3)) - 1u) & ~((1u << (r0 >> 3)) - 1u)) : 0;
        }
        __syncthreads();
        if (warp == 0) {
            // bounding cap of the patch: centre = normalised sum of its unit vectors, radius = largest angle to a point
            double cx = 0, cy = 0, cz = 0;
            for (int g = lane; g < G; g += 32) { cx += s_gu[g]; cy += s_gu[ROWS + g]; cz += s_gu[2 * ROWS + g]; }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                cx += __shfl_xor_sync(0xffffffffu, cx, o); cy += __shfl_xor_sync(0xffffffffu, cy, o);
                cz += __shfl_xor_sync(0xffffffffu, cz, o);
            }
            const double nn = sqrt(cx * cx + cy * cy + cz * cz);
            if (nn > 1e-12) { cx /= nn; cy /= nn; cz /= nn; } else { cx = s_gu[0]; cy = s_gu[ROWS]; cz = s_gu[2 * ROWS]; }
            double cmin = 1.0;
            for (int g = lane; g < G; g += 32)
                cmin = fmin(cmin, cx * s_gu[g] + cy * s_gu[ROWS + g] + cz * s_gu[2 * ROWS + g]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) cmin = fmin(cmin, __shfl_xor_sync(0xffffffffu, cmin, o));
            if (lane == 0) {
                s_bound[0] = (float)cx; s_bound[1] = (float)cy; s_bound[2] = (float)cz;
                s_bound[3] = (float)(acos(fmax(-1.0, fmin(1.0, cmin))) + 1e-6);
            }
        }
        __syncthreads();
        const float bcx = s_bound[0], bcy = s_bound[1], bcz = s_bound[2], brho = s_bound[3];

        // candidate source in serial order: the list of the coarse tile that contains the patch, or the ob range
        int64_t lb, le;
        const int *list = nullptr;
        if (p.tile_off) {
            const int ct = (prow / SP_CT) * p.nctx + pcol / SP_CT;
            lb = p.tile_off[ct];
            le = p.tile_off[ct + 1];
            list = p.tile_list;
        } else {
            lb = p.ob_begin;
            le = p.ob_end;
        }

        // this thread's state row (consumers: warp w holds rows 8w .. 8w+7, four lanes per row)
        const int r = warp * 8 + n;               // row slot in the CTA
        const int g = r / Lc, l = r % Lc;
        bool active = false;
        int64_t row = 0;
        if (g < G && l0 + l < p.nlev) {
            const int gy = y0 + g / p.tx, gx = x0 + g % p.tx;
            if (gy >= p.y_begin && gy < p.y_end && gx < p.nx) {
                active = true;
                row = (int64_t)(l0 + l) * p.npts + (int64_t)gy * p.nx + gx;
            }
        }
        const int gslot = active ? g : G;          // om[G] of a block is the zeros at the start of its tail
        double x[2 * NT3];
        bool loaded = false, dirty = false;

        int64_t pos = lb;
        S2_TICK(0);
        for (;;) {
            // =============================== PHASE A (1): candidates of this chunk ===============================
            int ncand = 0;
            while (pos < le && ncand + SCAN <= S2_CAND) {
                const int64_t e0 = pos + 2 * tid;
                int i0 = -1, i1 = -1;
                if (e0 < le) i0 = list ? __ldg(list + e0) : (int)e0;
                if (e0 + 1 < le) i1 = list ? __ldg(list + e0 + 1) : (int)(e0 + 1);
                float4 q0 = make_float4(0.f, 0.f, 0.f, -1.f), q1 = q0;
                if (i0 >= p.ob_begin && i0 < p.ob_end) q0 = __ldg(p.scan + i0);
                if (i1 >= p.ob_begin && i1 < p.ob_end) q1 = __ldg(p.scan + i1);
                bool h0 = false, h1 = false;
                if (q0.w >= 0.f) {
                    const float ang = q0.w + brho;
                    h0 = (ang >= 3.1405f) || (q0.x * bcx + q0.y * bcy + q0.z * bcz >= __cosf(ang) - 4e-6f);
                }
                if (q1.w >= 0.f) {
                    const float ang = q1.w + brho;
                    h1 = (ang >= 3.1405f) || (q1.x * bcx + q1.y * bcy + q1.z * bcz >= __cosf(ang) - 4e-6f);
                }
                const int cnt = (h0 ? 1 : 0) + (h1 ? 1 : 0);
                int inc = cnt;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int y = __shfl_up_sync(0xffffffffu, inc, o);
                    if (lane >= o) inc += y;
                }
                if (lane == 31) s_wcnt[warp] = inc;
                __syncthreads();
                int base = ncand, total = 0;
#pragma unroll
                for (int w = 0; w < NW; ++w) {
                    const int v = s_wcnt[w];
                    if (w < warp) base += v;
                    total += v;
                }
                int o = base + inc - cnt;
                if (h0) s_cand[o++] = i0;
                if (h1) s_cand[o] = i1;
                ncand += total;
                pos += SCAN;
                __syncthreads();
            }
            S2_TICK(1);
            if (ncand == 0) break;                // (the scan only stops empty-handed at the end of the list)
            const int nb = (ncand + 7) >> 3;

            // the consumers' rows are parked while the registers are needed for the weights
            if (loaded) {
#pragma unroll
                for (int i = 0; i < 2 * NT3; ++i) xsave[(size_t)i * NTH + tid] = x[i];
            }

            // =============================== PHASE A (2): one block per batch ===============================
            // Block of batch b (doubles): om[G][8] (point-major: omega of ob q at grid point g in g*8 + q) | tail[64]
            // (see S2_TCORR).
            {
                double *sob = s_sob + warp * 48;
                // scalars of the obs of a batch, held by lanes 0..7; loaded one batch ahead
                struct ObSc { double ux, uy, uz, ihw, amax, c1, beta; int kk; };      // (no arithmetic on the loaded values
                                                                                     // here: it would wait for them)
                auto load_sc = [&](int b, ObSc &o) {
                    o.ux = o.uy = o.uz = o.ihw = o.amax = o.c1 = o.beta = 0.0;
                    o.kk = -1;
                    if (b < nb && lane < 8 && 8 * b + lane < ncand) {
                        const int kk = s_cand[8 * b + lane];
                        o.kk = kk;
                        o.ux = s2_ldg_now(p.geo + GEO_UX * p.nobs + kk); o.uy = s2_ldg_now(p.geo + GEO_UY * p.nobs + kk);
                        o.uz = s2_ldg_now(p.geo + GEO_UZ * p.nobs + kk); o.ihw = s2_ldg_now(p.geo + GEO_INVHW * p.nobs + kk);
                        o.amax = s2_ldg_now(p.geo + GEO_AMAX * p.nobs + kk);
                        o.c1 = s2_ldg_now(p.rec + REC_C1 * p.nobs + kk);
                        o.beta = s2_ldg_now(p.rec + REC_BETA * p.nobs + kk);
                    }
                };
                ObSc cur, nxt;
                load_sc(warp, cur);
                for (int b = warp; b < nb; b += NW) {
                    const int nq = min(8, ncand - 8 * b);
                    load_sc(b + NW, nxt);
                    __syncwarp();                                    // the previous batch's readers of sob are done
                    if (lane < 8) {          // per ob: ux uy uz 1/halfwidth a_max beta*c1
                        *reinterpret_cast<double2 *>(sob + 6 * lane) = make_double2(cur.ux, cur.uy);
                        *reinterpret_cast<double2 *>(sob + 6 * lane + 2) = make_double2(cur.uz, cur.ihw);
                        // beta / ((N-1) kdenom)   (ensrf.py:95, :119, :135-136); the localisation weight multiplies it
                        *reinterpret_cast<double2 *>(sob + 6 * lane + 4) = make_double2(cur.amax, cur.c1 * cur.beta);
                    }
                    __syncwarp();
                    S2_TICK(6);
                    // supports of all 8 obs within the range of the branch-free weight functions?
                    const bool fast = __all_sync(0xffffffffu, lane >= 8 || cur.amax <= EXB_FAST_AMAX);
                    const bool shortser = __all_sync(0xffffffffu, lane >= 8 || cur.amax <= EXB_SHORT_AMAX);
                    double *gblk = blocks + (size_t)b * BLK;
                    // omega[q][g] = beta * loc / ((N-1) kdenom).  Grid points in whole groups of 32 are taken one per
                    // lane with the obs of the batch in the outer loop: the point's unit vector stays in registers, the
                    // ob's scalars are a broadcast read, and all lanes of a weight evaluation see the same ob (same side of
                    // r = 1 unless the patch straddles the ob's half-width circle).  The remaining G % 32 points are
                    // flattened with their obs over the lanes.  One evaluation at a time per lane: four warps per
                    // sub-partition already saturate the scalar FP64 pipe (8 clocks latency, 2 per instruction).
                    int npb = 0;
                    auto weigh = [&](double gx, double gy, double gz, int q, bool valid) -> double {
                        const double2 o01 = *reinterpret_cast<const double2 *>(sob + 6 * q);
                        const double2 o23 = *reinterpret_cast<const double2 *>(sob + 6 * q + 2);
                        const double2 o45 = *reinterpret_cast<const double2 *>(sob + 6 * q + 4);
                        double w = 1.0;
                        if (p.loc_mode == EXB_LOC_GC) {
                            const double a = hav_a(gx, gy, gz, o01.x, o01.y, o23.x);
                            w = shortser ? loc_weight_lean<true>(p.kloc, a, o23.y, o45.x)
                                : fast   ? loc_weight_lean<false>(p.kloc, a, o23.y, o45.x)
                                         : loc_weight(a, o23.y, o45.x);
                        }
                        w = valid ? w : 0.0;
                        npb += (w != 0.0) ? 1 : 0;
                        return w * o45.y;
                    };
                    // wm: the warps whose rows got a non-zero weight (bits of s_gwarps), for phase B to skip the others
                    unsigned wm = 0u;
                    const int nfull = G >> 5, R = G & 31;
                    for (int sl = 0; sl < nfull; ++sl) {
                        const int gg = lane + 32 * sl;
                        const double gx = s_gu[gg], gy = s_gu[ROWS + gg], gz = s_gu[2 * ROWS + gg];
                        const int gw = s_gwarps[gg];
                        const bool gval = gw != 0;
                        bool hit = false;
#pragma unroll 1
                        for (int q = 0; q < 8; q += 2) {
                            const double w0 = weigh(gx, gy, gz, q, gval && q < nq);
                            const double w1 = weigh(gx, gy, gz, q + 1, gval && q + 1 < nq);
                            hit |= (w0 != 0.0) | (w1 != 0.0);
                            *reinterpret_cast<double2 *>(gblk + 8 * gg + q) = make_double2(w0, w1);
                        }
                        wm |= hit ? (unsigned)gw : 0u;
                    }
                    if (R) {
                        // pairs i = q * R + r of the last R points: q = i / R by a multiplication (exact for i < 2^20 / R)
                        const int g0 = 32 * nfull, npr = 8 * R, nit = (npr + 31) >> 5;       // same trip count in every lane
                        const unsigned rdiv = ((1u << 20) + (unsigned)R - 1u) / (unsigned)R;
                        for (int it = 0; it < nit; ++it) {
                            const int i = lane + 32 * it, ic = min(i, npr - 1);
                            const int q = (int)(((unsigned)ic * rdiv) >> 20);
                            const int gg = g0 + ic - q * R;
                            const int gw = s_gwarps[gg];
                            const double w = weigh(s_gu[gg], s_gu[ROWS + gg], s_gu[2 * ROWS + gg], q,
                                                   i < npr && q < nq && gw != 0);
                            wm |= (w != 0.0) ? (unsigned)gw : 0u;
                            if (i < npr) gblk[8 * gg + q] = w;
                        }
                    }
                    if (lc == 0) npairs += (unsigned long long)npb;
                    S2_TICK(7);
                    // Gram matrix of the batch (members only: the pseudo-member column is masked or skipped): row n of the
                    // batch, this lane's two columns of every 8-column tile, operands straight from Yw (L2)
                    {
                        double g0 = 0.0, g1 = 0.0, h0 = 0.0, h1 = 0.0;
                        const int krow = __shfl_sync(0xffffffffu, cur.kk, n);
                        const double *yrow = p.Yw + (size_t)(krow >= 0 ? krow : p.nobs) * YW + 2 * c;
#pragma unroll
                        for (int t = 0; t < NT3; ++t) {
                            const double2 v = __ldg(reinterpret_cast<const double2 *>(yrow + 8 * t));
                            if (t < NT3 - 1 || LK >= 1) s2_dmma(g0, g1, v.x, v.x);
                            if (t < NT3 - 1 || LK == 2) {
                                const double v1 = (t == NT3 - 1 && c == 3) ? 0.0 : v.y;
                                s2_dmma(h0, h1, v1, v1);
                            }
                        }
                        // lane (n, c) holds G[n][2c], G[n][2c+1]: scatter them into the tail's layout
                        const double gx = g0 + h0, gy = g1 + h1;
                        double *gt = gblk + 8 * G;
                        if (c < 2)
                            *reinterpret_cast<double2 *>(gt + S2_TCORR + 4 * n + 2 * c) =
                                n >= 4 ? make_double2(gx, gy) : make_double2(0.0, 0.0);
                        const int lo = n & 4;                                   // G[n][j], lo <= j < n: recurrence
                        double *gr = gt + S2_TREC + 6 * (n >> 2) + (n - lo) * (n - lo - 1) / 2 - lo;
                        if (2 * c >= lo && 2 * c < n) gr[2 * c] = gx;
                        if (2 * c + 1 >= lo && 2 * c + 1 < n) gr[2 * c + 1] = gy;
                        wm = __reduce_or_sync(0xffffffffu, wm);
                        if (lane == 0) *reinterpret_cast<unsigned *>(gt + S2_TMASK) = wm;
                    }
                    cur = nxt;
                    S2_TICK(8);
                }
                S2_TICK(9);
            }
            // the blocks were written through the generic proxy and are read by bulk copies (async proxy)
            // (and the ring, read through the generic proxy in the previous phase B, is written by them again)
            __threadfence();
            asm volatile("fence.proxy.async.global;\n" ::: "memory");
            asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
            S2_TICK(2);
            __syncthreads();
            S2_TICK(5);

            // =============================== rows into registers ===============================
            {
                if (!loaded) {
                    double sum = 0.0;
#pragma unroll
                    for (int t = 0; t < NT3; ++t) {
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            const int m = s2_slot<NT3, LK>(t, c, h);
                            double v = 0.0;
                            if (active && m < nens) { v = (double)gXp[row * nens + m]; sum += v; }
                            x[2 * t + h] = v;
                        }
                    }
                    if (fused) {
                        // ensemble mean and perturbations of the row (assimilation.py:146-147)
                        sum += __shfl_xor_sync(0xffffffffu, sum, 1);
                        sum += __shfl_xor_sync(0xffffffffu, sum, 2);
                        const double mean = sum / (double)nens;
#pragma unroll
                        for (int t = 0; t < NT3; ++t) {
#pragma unroll
                            for (int h = 0; h < 2; ++h) {
                                const int m = s2_slot<NT3, LK>(t, c, h);
                                if (m < nens) x[2 * t + h] -= mean;
                            }
                        }
                        if (c == 3) x[2 * NT3 - 1] = active ? mean : 0.0;
                    } else if (c == 3) {
                        x[2 * NT3 - 1] = active ? (double)gxm[row] : 0.0;      // the mean rides along in the last column
                    }
                    loaded = true;
                } else {
#pragma unroll
                    for (int i = 0; i < 2 * NT3; ++i) x[i] = xsave[(size_t)i * NTH + tid];
                }
            }

            S2_TICK(3);
            // =============================== PHASE B ===============================
            {
                // Batch j of the chunk lives in ring stage (gbatch + j) % S.  Copies: 8 rows (lanes 0..7) + the block
                // (lane 8) onto the stage's `full` barrier.  Who issues: the first min(S, nb) batches one per warp at
                // the start; batch j >= S by warp (j - S + D) % 16 right after that warp has finished batch j - S + D
                // (D = S/4): the stage was released D batches ago by every warp that is not lagging, so the wait on
                // `empty` practically never blocks, and the copy has S - D batches of time to land.
                constexpr unsigned ROW_BYTES = YW * sizeof(double);
                const unsigned blk_bytes = (unsigned)BLK * sizeof(double);
                const int D = S >> 2;
                auto issue = [&](int j) {
                    const unsigned gbj = gbatch + (unsigned)j;
                    const int st = (int)(gbj % (unsigned)S);
                    const unsigned par = (gbj / (unsigned)S) & 1u;
                    s2_mbar_wait_empty(s_empty + st, par ^ 1u);
                    double *sy = s_ring + (size_t)st * SD;
                    if (lane < 8) {
                        const int idx = 8 * j + lane;
                        const int64_t k = idx < ncand ? (int64_t)s_cand[idx] : p.nobs;       // past the end: the zero row
                        s2_bulk_g2s(sy + lane * YST + (lane >> 1) * 4, p.Yw + (size_t)k * YW, ROW_BYTES, s_full + st);
                    } else if (lane == 8) {
                        s2_bulk_g2s(sy + YD, blocks + (size_t)j * BLK, blk_bytes, s_full + st);
                    }
                    if (lane == 0) s2_mbar_arrive_expect_tx(s_full + st, 8u * ROW_BYTES + blk_bytes);
                };
                for (int j = warp; j < S && j < nb; j += NW) issue(j);
                int rs = (int)(gbatch % (unsigned)S);
                unsigned rpar = (gbatch / (unsigned)S) & 1u;
                for (int b = 0; b < nb; ++b) {
                    s2_mbar_wait_full(s_full + rs, rpar);
                    const double *sy = s_ring + (size_t)rs * SD;
                    const double *som = sy + YD;
                    const double *Gt = som + 8 * G;

                    // does any row of this warp have a non-zero weight for an ob of the batch?  (phase A's warp mask)
                    if ((*reinterpret_cast<const unsigned *>(Gt + S2_TMASK) >> warp) & 1u) {
                        // omega of this row's grid point for the 8 obs of the batch (point-major block: om[G][8])
                        const double2 *omp = reinterpret_cast<const double2 *>(som + 8 * gslot);
                        const double2 om01 = omp[0], om23 = omp[1], om45 = omp[2], om67 = omp[3];
                        // step 1: g[row][ob] = x[row] . y_ob   (one accumulator chain: four warps per sub-partition keep
                        // the pipe fed, and the two halves need not be added afterwards); k-steps of the last tile
                        // without members are skipped (s2_slot)
                        double ga0 = 0.0, ga1 = 0.0;
                        {
                            const double *yrow = sy + n * YST + (n >> 1) * 4 + 2 * c;     // B operand: ob = n, columns of lane c
#pragma unroll
                            for (int t = 0; t < NT3; ++t) {
                                const double2 v = *reinterpret_cast<const double2 *>(yrow + 8 * t);
                                if (t < NT3 - 1 || LK >= 1) s2_dmma(ga0, ga1, x[2 * t], v.x);
                                if (t < NT3 - 1 || LK == 2) {
                                    const double a1 = (t == NT3 - 1 && c == 3) ? 0.0 : x[2 * t + 1];   // mask the mean
                                    s2_dmma(ga0, ga1, a1, v.y);
                                }
                            }
                        }
                        // lane c of a row holds g[row][2c], g[row][2c+1]: the row's 4 lanes exchange them through shared
                        // memory (1 store + 2 loads of 16 bytes instead of 8 shuffles; measured 2 % of the loop): obs 0..3
                        // now, obs 4..7 after their correction by obs 0..3 below
                        double gq[8];
                        double2 *xg = s_xch + warp * 32 + (lane & ~3);
                        xg[c] = make_double2(ga0, ga1);
                        __syncwarp();
                        {
                            const double2 t0 = xg[0], t1 = xg[1];
                            gq[0] = t0.x; gq[1] = t0.y; gq[2] = t1.x; gq[3] = t1.y;
                        }
                        // step 2: the serial recurrence inside the batch (per row; every lane of the row computes it)
                        // (coefficients G10 G20 | G21 G30 | G31 G32 | G54 G64 | G65 G74 | G75 G76)
                        const double2 *gr = reinterpret_cast<const double2 *>(Gt + S2_TREC);
                        const double2 r0 = gr[0], r1 = gr[1], r2 = gr[2];
                        double e[8];
                        e[0] = om01.x * gq[0];
                        e[1] = om01.y * (gq[1] - r0.x * e[0]);
                        e[2] = om23.x * (gq[2] - r0.y * e[0] - r1.x * e[1]);
                        e[3] = om23.y * (gq[3] - r1.y * e[0] - r2.x * e[1] - r2.y * e[2]);
                        const double ea = -s2_sel4(e[0], e[1], e[2], e[3], c);     // -e[c]: A operand below and in step 3
                        {
                            // obs 4..7 see obs 0..3 through one more 8x8x4 product on top of their own dots: the
                            // accumulator starts from g (lanes c = 2, 3 hold g[row][4..7] in fragment layout), A = -e,
                            // B[k][j] = G[j][k] for the columns j = 4..7 and zero for j = 0..3
                            double k0 = ga0, k1 = ga1;
                            s2_dmma(k0, k1, ea, Gt[S2_TCORR + lane]);
                            __syncwarp();                           // everybody has read obs 0..3
                            xg[c] = make_double2(k0, k1);
                            __syncwarp();
                            const double2 t2 = xg[2], t3 = xg[3];
                            gq[4] = t2.x; gq[5] = t2.y; gq[6] = t3.x; gq[7] = t3.y;
                        }
                        const double2 r3 = gr[3], r4 = gr[4], r5 = gr[5];
                        e[4] = om45.x * gq[4];
                        e[5] = om45.y * (gq[5] - r3.x * e[4]);
                        e[6] = om67.x * (gq[6] - r3.y * e[4] - r4.x * e[5]);
                        e[7] = om67.y * (gq[7] - r4.y * e[4] - r5.x * e[5] - r5.y * e[6]);
                        const double ea0 = ea;                 // A operand of the first k-step: -e[c]
                        const double ea1 = -s2_sel4(e[4], e[5], e[6], e[7], c);

                        // step 3: x[row][:] -= sum_q e_q y_q[:]   (A = -e in two k-steps, B = y, C = x)
                        {
                            const double *y0p = sy + c * YST + (c >> 1) * 4 + n;
                            const double *y1p = sy + (4 + c) * YST + ((4 + c) >> 1) * 4 + n;
                            // all tiles with obs 0..3 first, then all with obs 4..7: a tile's second DMMA depends on its
                            // first (26 clocks), back to back it would stall the warp's in-order issue
#pragma unroll
                            for (int t = 0; t < NT3; ++t) s2_dmma_v(x[2 * t], x[2 * t + 1], ea0, y0p[8 * t]);
#pragma unroll
                            for (int t = 0; t < NT3; ++t) s2_dmma_v(x[2 * t], x[2 * t + 1], ea1, y1p[8 * t]);
                        }
                        dirty = true;
                    }
                    __syncwarp();
                    if (lane == 0) s2_mbar_arrive(s_empty + rs);
                    rs = (rs + 1 == S) ? 0 : rs + 1;
                    rpar ^= (rs == 0) ? 1u : 0u;
                    // this warp's turn to refill a stage?
                    const int j = b - D + S;
                    if (b >= D && j < nb && ((b - D) & (NW - 1)) == warp) issue(j);
                }
                gbatch += (unsigned)nb;
            }
            S2_TICK(4);
            if (pos >= le) break;
            __syncthreads();                      // phase B is over before the next chunk's scan rewrites s_cand
            S2_TICK(5);
        }

        // ---- write the patch back: xam of the row (ensrf.py:130) lives in lane c = 3 ---------------------------
        if (loaded) {
            double mean = __shfl_sync(0xffffffffu, x[2 * NT3 - 1], (lane & ~3) | 3);
            if (!fused) mean = 0.0;
            if (active && dirty) {
#pragma unroll
                for (int t = 0; t < NT3; ++t) {
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int m = s2_slot<NT3, LK>(t, c, h);
                        if (m < nens) gXp[row * nens + m] = (TS)(x[2 * t + h] + mean);          // assimilation.py:168 when fused
                        else if (m == PC && !fused) gxm[row] = (TS)x[2 * t + h];
                    }
                }
            }
        }
    }
    if (p.prof && tid == 0) {
        S2_TICK(3);
#pragma unroll
        for (int i = 0; i < 10; ++i) atomicAdd(&p.prof[i], (unsigned long long)pacc[i]);
        atomicAdd(&p.prof[10], (unsigned long long)gbatch);
    }
    if (p.counters) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) npairs += __shfl_xor_sync(0xffffffffu, npairs, o);
        if (lane == 0 && npairs) atomicAdd(&p.counters[1], npairs);
    }
}

// Yw[k][:] = (ye_k widened to double, zeros, -innov_k/beta_k in the last column), columns in the order of s2_slot;
// row nobs = zeros
template <int NT3, int LK, typename TS>
__global__ void sweep_rows_kernel(const TS *__restrict__ Yp, const double *__restrict__ rec, int64_t nobs, int nens,
                                  double *__restrict__ Yw) {
    constexpr int YW = 8 * NT3;
    const int64_t k = blockIdx.x;
    for (int col = threadIdx.x; col < YW; col += blockDim.x) {
        const int m = s2_slot<NT3, LK>(col >> 3, (col & 7) >> 1, col & 1);
        double v = 0.0;
        if (k < nobs) {
            if (m < nens) v = (double)Yp[k * nens + m];
            else if (m == YW - 1 && rec[REC_ASSIM * nobs + k] != 0.0)
                v = -rec[REC_INNOV * nobs + k] / rec[REC_BETA * nobs + k];       // xam = xbm + kmat*innov rides along (ensrf.py:130)
        }
        Yw[k * YW + col] = v;
    }
}

// ------------------------------------------------------------------------------------------
// candidate lists per coarse tile
// ------------------------------------------------------------------------------------------
// bounding cap (centre, angular radius) of every coarse tile: one warp per tile
__global__ void sweep_tile_caps_kernel(const double *__restrict__ grid_u, int64_t npts, int nx, int y_begin, int y_end, int pr0,
                                       int cty, int ctx, int nctx, int ntiles, float4 *__restrict__ caps) {
    const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (t >= ntiles) return;
    const int ya = max((pr0 / SP_CT + t / nctx) * cty, y_begin), yb = min((pr0 / SP_CT + t / nctx + 1) * cty, y_end);
    const int xa = (t % nctx) * ctx, xb = min(xa + ctx, nx);
    const int w = xb - xa, npt = max(yb - ya, 0) * w;
    double cx = 0, cy = 0, cz = 0;
    for (int i = lane; i < npt; i += 32) {
        const int64_t pt = (int64_t)(ya + i / w) * nx + xa + i % w;
        cx += grid_u[pt]; cy += grid_u[npts + pt]; cz += grid_u[2 * npts + pt];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        cx += __shfl_xor_sync(0xffffffffu, cx, o); cy += __shfl_xor_sync(0xffffffffu, cy, o); cz += __shfl_xor_sync(0xffffffffu, cz, o);
    }
    const double nn = sqrt(cx * cx + cy * cy + cz * cz);
    if (nn > 1e-9) { cx /= nn; cy /= nn; cz /= nn; }
    double cmin = 1.0;
    for (int i = lane; i < npt; i += 32) {
        const int64_t pt = (int64_t)(ya + i / w) * nx + xa + i % w;
        cmin = fmin(cmin, cx * grid_u[pt] + cy * grid_u[npts + pt] + cz * grid_u[2 * npts + pt]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cmin = fmin(cmin, __shfl_xor_sync(0xffffffffu, cmin, o));
    if (lane == 0) {
        // degenerate centre (tile wraps the globe): radius pi -> everything is a candidate
        const double rho = (nn > 1e-9 && npt > 0) ? acos(fmax(-1.0, fmin(1.0, cmin))) + 1e-4 : 3.2;
        caps[t] = make_float4((float)cx, (float)cy, (float)cz, (float)rho);
    }
}

// FILL = false: cnt[t] = number of obs whose support can touch tile t; FILL = true: their ascending list
template <bool FILL>
__global__ void sweep_tile_list_kernel(const float4 *__restrict__ caps, int ntiles, const float4 *__restrict__ scan,
                                       int64_t ob_begin, int64_t ob_end, int *__restrict__ cnt,
                                       const int64_t *__restrict__ off, int *__restrict__ list) {
    const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (t >= ntiles) return;
    const float4 cap = caps[t];
    int64_t pos = FILL ? off[t] : 0;
    int count = 0;
    const unsigned lt = (1u << lane) - 1u;
    // One warp walks all obs for its tile: the loop is bound by the latency of the scan-record loads, so the records of
    // TL_UNROLL groups of 32 obs are fetched before the first of them is tested (the groups are still taken in order).
    constexpr int TL_UNROLL = 8;
    for (int64_t base = ob_begin; base < ob_end; base += 32 * TL_UNROLL) {
        float4 sc[TL_UNROLL];
#pragma unroll
        for (int u = 0; u < TL_UNROLL; ++u) {
            const int64_t k = base + 32 * u + lane;
            sc[u] = (k < ob_end) ? __ldg(scan + k) : make_float4(0.f, 0.f, 0.f, -1.f);
        }
#pragma unroll
        for (int u = 0; u < TL_UNROLL; ++u) {
            const int64_t k = base + 32 * u + lane;
            bool hit = false;
            if (sc[u].w >= 0.f) {                  // (past the end of the range: w = -1)
                const float ang = sc[u].w + cap.w;
                hit = (ang >= 3.1405f) || (sc[u].x * cap.x + sc[u].y * cap.y + sc[u].z * cap.z >= __cosf(ang) - 4e-6f);
            }
            if (FILL) {
                const unsigned b = __ballot_sync(0xffffffffu, hit);
                if (hit) list[pos + __popc(b & lt)] = (int)k;
                pos += __popc(b);
            } else {
                count += hit ? 1 : 0;
            }
        }
    }
    if (!FILL) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) count += __shfl_xor_sync(0xffffffffu, count, o);
        if (lane == 0) cnt[t] = count;
    }
}

// grid row of [y_begin, y_end) closest to the equator (|sin lat| of its first column smallest) -> mapped host word
__global__ void sweep_eq_row_kernel(const double *__restrict__ uz, int nx, int y_begin, int y_end, long long *__restrict__ out) {
    __shared__ double bv[256];
    __shared__ int bi[256];
    double best = 2.0;
    int besty = y_begin;
    for (int y = y_begin + threadIdx.x; y < y_end; y += 256) {
        const double v = fabs(uz[(int64_t)y * nx]);
        if (v < best) { best = v; besty = y; }
    }
    bv[threadIdx.x] = best; bi[threadIdx.x] = besty;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o && bv[threadIdx.x + o] < bv[threadIdx.x]) { bv[threadIdx.x] = bv[threadIdx.x + o]; bi[threadIdx.x] = bi[threadIdx.x + o]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = bi[0];
}

// exclusive prefix sum of cnt[n] into off[n+1], n small (one CTA, serial over chunks of 1024)
__global__ void __launch_bounds__(1024) sweep_scan_kernel(const int *__restrict__ cnt, int n, int64_t *__restrict__ off,
                                                         long long *__restrict__ total_host) {
    __shared__ long long part[1024];
    __shared__ long long carry_s;
    const int t = threadIdx.x;
    if (t == 0) carry_s = 0;
    __syncthreads();
    for (int b = 0; b < n; b += 1024) {
        const int i = b + t;
        const long long v = i < n ? cnt[i] : 0;
        part[t] = v;
        __syncthreads();
        for (int d = 1; d < 1024; d <<= 1) {
            const long long y = t >= d ? part[t - d] : 0;
            __syncthreads();
            part[t] += y;
            __syncthreads();
        }
        const long long carry = carry_s;
        if (i < n) off[i] = carry + part[t] - v;
        __syncthreads();
        if (t == 1023) carry_s = carry + part[1023];
        __syncthreads();
    }
    if (t == 0) {
        off[n] = carry_s;
        *total_host = carry_s;        // mapped pinned host word: no D2H copy queued behind band downloads
    }
}

// ------------------------------------------------------------------------------------------
// host side: candidate lists per coarse tile
// ------------------------------------------------------------------------------------------
static bool sweep_lists_wanted(int loc_mode, int64_t ob_begin, int64_t ob_end) {
    return loc_mode == EXB_LOC_GC && ob_end - ob_begin > 4096;
}

// Builds, for every coarse tile (SP_CT x SP_CT patches of bty x btx grid points) that intersects grid rows
// [y_begin, y_end), the ascending list of obs in [ob_begin, ob_end) whose support can touch the tile.  Synchronises the
// stream once (list sizes).  out->tile_off is indexed by ABSOLUTE coarse-tile number (coarse row * nctx + coarse col).
static int sweep_build_lists(const double *grid_u, int64_t npts, int nx, int y_begin, int y_end, int bty, int btx,
                             const float4 *scan, int64_t ob_begin, int64_t ob_end, cudaStream_t st, SweepLists *out) {
    const int pr0 = y_begin / bty, pr1 = (y_end + bty - 1) / bty;
    const int cty = bty * SP_CT, ctx = btx * SP_CT;
    out->nctx = (nx + ctx - 1) / ctx;
    const int cr0 = pr0 / SP_CT, cr1 = (pr1 + SP_CT - 1) / SP_CT;
    const int ntiles = (cr1 - cr0) * out->nctx;
    EXB_CUDA(exb_malloc_async(&out->caps, sizeof(float4) * ntiles, st));
    EXB_CUDA(exb_malloc_async(&out->cnt, sizeof(int) * ntiles, st));
    EXB_CUDA(exb_malloc_async(&out->off, sizeof(int64_t) * (ntiles + 1), st));
    const unsigned gridw = (unsigned)ceil_div64((int64_t)ntiles * 32, 256);
    sweep_tile_caps_kernel<<<gridw, 256, 0, st>>>(grid_u, npts, nx, y_begin, y_end, pr0, cty, ctx, out->nctx, ntiles, out->caps);
    sweep_tile_list_kernel<false><<<gridw, 256, 0, st>>>(out->caps, ntiles, scan, ob_begin, ob_end, out->cnt, nullptr, nullptr);
    ExbHostWords hw;                   // this call's own mapped words: [0] list total, [1] equator row
    const int rcw = exb_host_words_acquire(&hw);
    if (rcw != EXB_OK) return rcw;
    struct WordsGuard { ExbHostWords w; ~WordsGuard() { exb_host_words_release(w); } } wguard{hw};
    sweep_scan_kernel<<<1, 1024, 0, st>>>(out->cnt, ntiles, out->off, hw.dev);
    sweep_eq_row_kernel<<<1, 256, 0, st>>>(grid_u + 2 * npts, nx, y_begin, y_end, hw.dev + 1);
    exb_count_launches(4);
    EXB_CUDA(cudaStreamSynchronize(st));
    const long long total = hw.host[0];
    out->eq_row = (int)hw.host[1];
    EXB_CUDA(exb_malloc_async(&out->list, sizeof(int) * (size_t)(total > 0 ? total : 1), st));
    sweep_tile_list_kernel<true><<<gridw, 256, 0, st>>>(out->caps, ntiles, scan, ob_begin, ob_end, nullptr, out->off, out->list);
    exb_count_launches(1);
    // the kernels index tiles by absolute coarse row: shift the offsets' base
    out->tile_off = out->off - (int64_t)cr0 * out->nctx;
    return exb_check_launch("sweep_tile_list_kernel");
}

static void sweep_free_lists(SweepLists &l, cudaStream_t st) {
    if (l.caps) cudaFreeAsync(l.caps, st);
    if (l.cnt) cudaFreeAsync(l.cnt, st);
    if (l.off) cudaFreeAsync(l.off, st);
    if (l.list) cudaFreeAsync(l.list, st);
    l.caps = nullptr; l.cnt = nullptr; l.off = nullptr; l.list = nullptr;
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static void s2_patch_shape(int64_t nlev, int64_t ny, int64_t nx, int *Lc_out, int *bty_out, int *btx_out) {
    const int rows = 8 * S2_NW;
    const int Lc = nlev < rows ? (int)nlev : rows;
    const int G = rows / Lc;
    int bty = 1, btx = G;
    for (int ty = 1; ty * ty <= G; ++ty) {
        const int tx = G / ty;
        if (ty * tx > bty * btx || (ty * tx == bty * btx && ty > bty)) { bty = ty; btx = tx; }
    }
    if (btx > nx) btx = (int)nx;
    if (bty > ny) bty = (int)ny;
    *Lc_out = Lc; *bty_out = bty; *btx_out = btx;
}

template <int NT3, int LK, typename TS>
static int s2_launch(S2Params &p, const TS *Yp, cudaStream_t st, const ExbSweepPlan *plan) {
    constexpr int NTH = S2_NW * 32, ROWS = S2_NW * 8;
    int Lc, bty, btx;
    s2_patch_shape(p.nlev, p.ny, p.nx, &Lc, &bty, &btx);
    p.ty = bty; p.tx = btx; p.G = bty * btx; p.Lc = Lc;
    p.nlc = (p.nlev + Lc - 1) / Lc;
    p.ntx = (p.nx + btx - 1) / btx;
    p.pr0 = p.y_begin / bty;
    const int pr1 = (p.y_end + bty - 1) / bty;              // patch rows [pr0, pr1)
    p.npr = pr1 - p.pr0;
    p.pr_eq = -1;
    p.blk_doubles = 8 * p.G + 64;
    p.stage_doubles = s2_ydoubles<NT3>() + p.blk_doubles;
    int dev = 0, max_smem = 0, sms = 0;
    EXB_CUDA(cudaGetDevice(&dev));
    EXB_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    EXB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const size_t fixed = sizeof(double) * (3 * ROWS + S2_NW * 48 + S2_NW * 64) + sizeof(unsigned long long) * 2 * S2_MAXSTAGES +
                         sizeof(int) * (S2_CAND + ROWS + S2_NW + 4) + sizeof(float) * 4 + 128;
    // ring stages: whatever is left of the largest opt-in block, less 1 KB of headroom
    int S = (int)(((size_t)max_smem - 1024 - fixed) / (sizeof(double) * p.stage_doubles));
    if (S > S2_MAXSTAGES) S = S2_MAXSTAGES;
    if (S < 4) return EXB_ERR_UNSUPPORTED;
    p.nstages = S;
    const size_t smem = fixed + sizeof(double) * (size_t)S * p.stage_doubles;
    EXB_CUDA(cudaFuncSetAttribute(state_sweep_2p_kernel<NT3, LK, TS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));

    const int64_t npatches = (int64_t)p.ntx * p.npr * p.nlc;
    if (npatches >= 0x7fffffff) {
        exb_set_error("exb_state_sweep: too many patches for one launch");
        return EXB_ERR_ARG;
    }
    if (npatches <= 0) return EXB_OK;
    p.npatches = (int)npatches;
    const int grid = npatches < (int64_t)sms ? (int)npatches : sms;

    // candidate lists per coarse tile (localised runs only; the kernel walks the ob range otherwise)
    SweepLists lists;
    p.tile_off = nullptr;
    p.tile_list = nullptr;
    p.nctx = 1;
    if (plan && plan->have_lists && plan->y_begin <= p.y_begin && p.y_end <= plan->y_end && plan->ob_begin == p.ob_begin &&
        plan->ob_end == p.ob_end) {
        // lists built ahead (exb_sweep_plan_create): indexed by absolute coarse tile, so they serve any row sub-range
        p.nctx = plan->lists.nctx;
        p.pr_eq = plan->lists.eq_row / bty;
        p.tile_off = plan->lists.tile_off;
        p.tile_list = plan->lists.list;
    } else if (sweep_lists_wanted(p.loc_mode, p.ob_begin, p.ob_end)) {
        const int rcl = sweep_build_lists(p.grid_u, p.npts, p.nx, p.y_begin, p.y_end, bty, btx, p.scan, p.ob_begin, p.ob_end, st, &lists);
        if (rcl != EXB_OK) { sweep_free_lists(lists, st); return rcl; }
        p.nctx = lists.nctx;
        p.pr_eq = lists.eq_row / bty;
        p.tile_off = lists.tile_off;
        p.tile_list = lists.list;
    }
    // padded ob rows, scratch, ticket
    constexpr int YW = 8 * NT3;
    double *Yw = nullptr, *scratch = nullptr;
    int *ticket = nullptr;
    p.scratch_stride = (int64_t)(S2_CAND / 8) * p.blk_doubles + (int64_t)2 * NT3 * NTH;
    cudaError_t e = exb_malloc_async(&Yw, sizeof(double) * (size_t)(p.nobs + 1) * YW, st);
    if (e == cudaSuccess) e = exb_malloc_async(&scratch, sizeof(double) * (size_t)p.scratch_stride * grid, st);
    if (e == cudaSuccess) e = exb_malloc_async(&ticket, sizeof(int), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(ticket, 0, sizeof(int), st);
    int rc = EXB_OK;
    if (e != cudaSuccess) {
        exb_set_error("exb_state_sweep: work buffers -> %s", cudaGetErrorString(e));
        rc = EXB_ERR_CUDA;
    } else {
        sweep_rows_kernel<NT3, LK, TS><<<(unsigned)(p.nobs + 1), 128, 0, st>>>(Yp, p.rec, p.nobs, p.nens, Yw);
        p.Yw = Yw; p.scratch = scratch; p.ticket = ticket;
        p.abort_flag = exb_status_slot_last_dev();
        unsigned long long *prof = nullptr;
        if (getenv("EXB_S2_PROF") && atoi(getenv("EXB_S2_PROF"))) {       // debugging aid: per-phase clocks of warp 0
            if (cudaMalloc(&prof, 11 * sizeof(unsigned long long)) == cudaSuccess) cudaMemsetAsync(prof, 0, 11 * sizeof(unsigned long long), st);
            else prof = nullptr;
        }
        p.prof = prof;
        state_sweep_2p_kernel<NT3, LK, TS><<<(unsigned)grid, NTH, smem, st>>>(p);
        exb_count_launches(2);
        rc = exb_check_launch("state_sweep_2p_kernel");
        if (prof) {
            unsigned long long h[11];
            cudaStreamSynchronize(st);
            cudaMemcpy(h, prof, sizeof(h), cudaMemcpyDeviceToHost);
            cudaFree(prof);
            double tot = 0;
            for (int i = 0; i < 6; ++i) tot += (double)h[i];
            for (int i = 6; i < 10; ++i) tot += (double)h[i];
            fprintf(stderr, "[s2 prof] grid %d patches %d: setup %.1f%% scan %.1f%% park+fence %.1f%% rows %.1f%% phaseB %.1f%% barriers %.1f%% | blocks: scalars %.1f%% omega %.1f%% gram %.1f%% rest %.1f%%  (%.3e clk per CTA)\n",
                    grid, p.npatches, 100 * h[0] / tot, 100 * h[1] / tot, 100 * h[2] / tot, 100 * h[3] / tot, 100 * h[4] / tot, 100 * h[5] / tot,
                    100 * h[6] / tot, 100 * h[7] / tot, 100 * h[8] / tot, 100 * h[9] / tot, tot / grid);
            // clocks per (row, batch): a CTA takes its batches one after the other, over all of its ROWS row slots
            const double rb = (double)(h[10] > 0 ? h[10] : 1) * ROWS;
            fprintf(stderr, "[s2 prof] %llu batches: %.2f clk per (row, batch), phase B %.2f, blocks %.2f (omega %.2f, gram %.2f)\n",
                    h[10], tot / rb, h[4] / rb, (h[6] + h[7] + h[8] + h[9]) / rb, h[7] / rb, h[8] / rb);
        }
    }
    if (Yw) cudaFreeAsync(Yw, st);
    if (scratch) cudaFreeAsync(scratch, st);
    if (ticket) cudaFreeAsync(ticket, st);
    sweep_free_lists(lists, st);
    return rc;
}

// the instantiation for the members in the last tile (s2_slot)
template <int NT3, typename TS>
static int s2_launch_lk(S2Params &p, const TS *Yp, cudaStream_t st, const ExbSweepPlan *plan) {
    switch (s2_last_ksteps<NT3>(p.nens)) {
    case 0: return s2_launch<NT3, 0, TS>(p, Yp, st, plan);
    case 1: return s2_launch<NT3, 1, TS>(p, Yp, st, plan);
    default: return s2_launch<NT3, 2, TS>(p, Yp, st, plan);
    }
}

// Called from state_update.cu.  TS is the storage type of state and ye rows (float64, or float32 with float64
// arithmetic in registers: every row is read and rounded back exactly once).  xm == nullptr selects the fused
// split/recombine mode (Xp then holds full ensemble values).  Returns EXB_ERR_UNSUPPORTED if no instantiation fits
// (more than 103 members).
template <typename TS>
int exb_state_sweep_2p(TS *xm, TS *Xp, int64_t nlev, int64_t ny, int64_t nx, int nens, const double *grid_u, const TS *Yp,
                       const double *rec, const double *obgeo, const float4 *scan, int64_t nobs, int64_t ob_begin,
                       int64_t ob_end, int64_t y_begin, int64_t y_end, int loc_mode, unsigned long long *counters,
                       cudaStream_t st, const ExbSweepPlan *plan) {
    S2Params p;
    memset(&p, 0, sizeof(p));
    p.xm = xm; p.Xp = Xp; p.grid_u = grid_u; p.rec = rec; p.geo = obgeo; p.scan = scan;
    p.counters = counters; p.npts = ny * nx; p.nobs = nobs; p.ob_begin = ob_begin; p.ob_end = ob_end;
    p.nlev = (int)nlev; p.ny = (int)ny; p.nx = (int)nx; p.nens = nens; p.loc_mode = loc_mode;
    p.y_begin = (int)y_begin; p.y_end = (int)y_end;
    p.kloc = exb_loc_const();
    const int need = (nens + 1 + 7) / 8;            // 8-member tiles incl. the pseudo-member
    if (need <= 4) return s2_launch_lk<4, TS>(p, Yp, st, plan);
    if (need <= 7) return s2_launch_lk<7, TS>(p, Yp, st, plan);
    if (need <= 10) return s2_launch_lk<10, TS>(p, Yp, st, plan);
    if (need <= 13) return s2_launch_lk<13, TS>(p, Yp, st, plan);
    return EXB_ERR_UNSUPPORTED;                       // larger ensembles: state_update_mma.cu / state_update.cu
}

template int exb_state_sweep_2p<double>(double *, double *, int64_t, int64_t, int64_t, int, const double *, const double *,
                                        const double *, const double *, const float4 *, int64_t, int64_t, int64_t, int64_t,
                                        int64_t, int, unsigned long long *, cudaStream_t, const ExbSweepPlan *);
template int exb_state_sweep_2p<float>(float *, float *, int64_t, int64_t, int64_t, int, const double *, const float *,
                                       const double *, const double *, const float4 *, int64_t, int64_t, int64_t, int64_t,
                                       int64_t, int, unsigned long long *, cudaStream_t, const ExbSweepPlan *);

// Row granularity of the patches for a state with nlev levels: sweeping row ranges whose edges are multiples of
// this value never splits a patch between two calls.
extern "C" int exb_state_sweep_row_granularity(int64_t nlev, int64_t ny, int64_t nx) {
    int Lc, bty, btx;
    s2_patch_shape(nlev, ny, nx, &Lc, &bty, &btx);
    return bty;
}

// ------------------------------------------------------------------------------------------
// sweep plan: the geometry-only part of the sweep, built ahead of the obs-space solve
// ------------------------------------------------------------------------------------------
__global__ void sweep_scan_from_flags_kernel(const double *__restrict__ geo, const uint8_t *__restrict__ assim, int64_t nobs,
                                             float4 *__restrict__ scan) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= nobs) return;
    float4 v;
    v.x = (float)geo[GEO_UX * nobs + k];
    v.y = (float)geo[GEO_UY * nobs + k];
    v.z = (float)geo[GEO_UZ * nobs + k];
    // same record as su_scan_records_kernel (state_update.cu) builds from rec[REC_ASSIM] after the solve
    v.w = assim[k] ? (float)geo[GEO_THETA * nobs + k] * 1.000001f + 1e-7f : -1.f;
    scan[k] = v;
}

static void sweep_plan_free(ExbSweepPlan *pl) {
    if (!pl) return;
    if (pl->was_used && pl->used) cudaStreamWaitEvent(pl->st, pl->used, 0);
    if (pl->scan) cudaFreeAsync(pl->scan, pl->st);
    sweep_free_lists(pl->lists, pl->st);
    if (pl->ready) cudaEventDestroy(pl->ready);
    if (pl->used) cudaEventDestroy(pl->used);
    delete pl;
}

extern "C" int exb_sweep_plan_create(const double *grid_u, int64_t nlev, int64_t ny, int64_t nx, const double *obgeo,
                                     const uint8_t *ob_assimilate, int64_t nobs, int64_t ob_begin, int64_t ob_end,
                                     int64_t y_begin, int64_t y_end, int loc_mode, void *stream, void **plan) {
    EXB_REQUIRE(grid_u && obgeo && ob_assimilate && plan, "null pointer");
    EXB_REQUIRE(nlev > 0 && ny > 0 && nx > 0 && nobs > 0, "bad sizes");
    EXB_REQUIRE(0 <= ob_begin && ob_begin <= ob_end && ob_end <= nobs && 0 <= y_begin && y_begin < y_end && y_end <= ny, "bad ranges");
    *plan = nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    ExbSweepPlan *pl = new ExbSweepPlan();
    struct Guard { ExbSweepPlan *p; ~Guard() { if (p) sweep_plan_free(p); } } guard{pl};
    pl->nlev = nlev; pl->ny = ny; pl->nx = nx; pl->nobs = nobs; pl->ob_begin = ob_begin; pl->ob_end = ob_end;
    pl->y_begin = y_begin; pl->y_end = y_end; pl->loc_mode = loc_mode; pl->grid_u = grid_u; pl->obgeo = obgeo; pl->st = st;
    EXB_CUDA(cudaEventCreateWithFlags(&pl->ready, cudaEventDisableTiming));
    EXB_CUDA(cudaEventCreateWithFlags(&pl->used, cudaEventDisableTiming));
    EXB_CUDA(exb_malloc_async(&pl->scan, (size_t)nobs * sizeof(float4), st));
    sweep_scan_from_flags_kernel<<<(unsigned)ceil_div64(nobs, 256), 256, 0, st>>>(obgeo, ob_assimilate, nobs, pl->scan);
    exb_count_launches(1);
    if (sweep_lists_wanted(loc_mode, ob_begin, ob_end)) {
        int Lc, bty, btx;
        s2_patch_shape(nlev, ny, nx, &Lc, &bty, &btx);
        const int rc = sweep_build_lists(grid_u, ny * nx, (int)nx, (int)y_begin, (int)y_end, bty, btx, pl->scan, ob_begin,
                                         ob_end, st, &pl->lists);
        if (rc != EXB_OK) return rc;
        pl->have_lists = true;
    }
    EXB_CUDA(cudaEventRecord(pl->ready, st));
    guard.p = nullptr;
    *plan = pl;
    return exb_check_launch("sweep_scan_from_flags_kernel");
}

extern "C" int exb_sweep_plan_destroy(void *plan) {
    sweep_plan_free(static_cast<ExbSweepPlan *>(plan));
    return EXB_OK;
}
