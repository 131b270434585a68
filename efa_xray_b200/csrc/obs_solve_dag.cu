// Obs-space serial solve as a DEPENDENCY-DRIVEN (sync-free sparse-triangular) kernel.
//
// The serial loop of ensrf.py:50-149 restricted to the obs rows is   for k: for j > k:  row_j -= f_kj(row_j . ye_k) ye_k
// with f_kj = 0 unless ob j lies inside ob k's localisation support (observation.py:117-130).  Ob j therefore
// depends only on the EARLIER obs whose support reaches it; two obs that are far apart never see each other and
// the order in which their updates are issued does not matter, as long as every row receives ITS updates in
// index order.  That is a sparse lower-triangular solve, and it is run like one:
//   * dag_list_kernel     builds, for every row j, the ascending list of predecessors k < j that may reach it
//                         (conservative fp32 dot-product test on packed unit vectors; CSR, two passes: count + fill);
//   * dag_solve_kernel    one WARP per row, rows handed out in index order by a ticket counter.  The warp walks
//                         its predecessor list in order; for each k it needs the published record of ob k
//                         (ye_k and the scalars innov_k, c1_k, beta_k), applies the rank-1 update
//                         (ensrf.py:95-141) to its row, and after the last predecessor computes its own scalars
//                         (ensrf.py:61-91, :135) and publishes its record.
// The serial chain is no longer Nobs steps long but the longest dependency path (config 3: 3 864 instead of
// 100 000), and thousands of rows are in flight at once.  The result is the same arithmetic in the same order for
// every row, i.e. the serial order of the reference is preserved exactly.
//
// Publication without flags or fences: records go to a side buffer P (row stride 32*MC elements) / S (2 doubles
// per ob) that is pre-filled with an all-ones bit pattern (a NaN the arithmetic never produces; the writer
// canonicalises).  A reader loads the record with gpu-scope relaxed loads and accepts it when no word is the
// sentinel; each lane checks exactly the words it consumes, each word is written by one aligned store, so no
// ordering between words is needed.  Waiting warps poll one 16-byte word of S with back-off.
// Deadlock freedom: a warp only waits for rows with a lower ticket, and those were taken by warps that are
// already running.  A watchdog turns a would-be hang into an error status.
#include "common.cuh"
#include <cstdlib>
#include <cstring>
#include <vector>

#define DG_TILE 2048            // candidates staged in shared memory per step of the list builder
#define DG_LWARPS 4             // warps per CTA of the list builder
#define DG_LROWS (32 * DG_LWARPS) // rows per CTA of the list builder (one lane per row)
#define DG_WARPS 4              // warps per CTA of the solve kernel
#define DG_MINBLOCKS 8          // -> at most 64 registers per thread, 32 rows in flight per SM
// measured on config 3: the tensor-pipe reduction below is no faster than the shuffle butterfly (18.6 vs 18.1 ms)
#ifndef DG_DMMA_REDUCE
#define DG_DMMA_REDUCE 0
#endif
#define DG_SENT 0xFFFFFFFFFFFFFFFFull
#define DG_FULL 0xffffffffu
// A dependency wait is declared dead after this many seconds without progress (EXB_WATCHDOG_S overrides; a wait is
// legitimately as long as everything that precedes the row, so the default also grows with nobs)
#define DG_WATCHDOG_S 20.0

template <typename T>
int exb_obs_solve_dag(T *Ym, T *Yp, const double *ob_value, const double *ob_error, const uint8_t *ob_assim,
                      const double *ob_thr, const double *geo, int64_t nobs, int nens, int loc_mode, double *rec,
                      unsigned long long *counters, cudaStream_t st, bool force, void *plan);

__device__ __forceinline__ int64_t ceil_div64_dev(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Rows of a distributed solve are dealt to the ranks in BLOCKS of `block` consecutive obs: rank r owns the obs j with
// (j / block) % world == r; its v-th row is dg_row(v).  block = 1 is round-robin; world = 1 the identity.  The map is
// strictly increasing in v, which is all the list builder and the ticket order need.
struct DgDeal { int block, world, rank; };
__host__ __device__ __forceinline__ int64_t dg_row(const DgDeal &d, int64_t v) {
    return ((v / d.block) * d.world + d.rank) * (int64_t)d.block + v % d.block;
}
// ------------------------------------------------------------------------------------------
// predecessor lists
// ------------------------------------------------------------------------------------------
// float4 per ob: unit vector and, in .w, the smallest u_j . u_k at which row j is still inside the support of
// THIS ob acting as k (squared chord = 2 - 2 dot), lowered so that the fp32 test never misses a pair the fp64
// weight would keep; > 1 for obs that are not assimilated (never a predecessor).
__global__ void dag_pack_kernel(const double *__restrict__ geo, const uint8_t *__restrict__ assim, int64_t nobs,
                                int loc_mode, float4 *__restrict__ pk) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= nobs) return;
    float4 q;
    q.x = (float)geo[GEO_UX * nobs + k];
    q.y = (float)geo[GEO_UY * nobs + k];
    q.z = (float)geo[GEO_UZ * nobs + k];
    float cmin = 3.0f;
    if (assim[k]) {
        const double amax = geo[GEO_AMAX * nobs + k];
        if (loc_mode != EXB_LOC_GC || amax >= 1.0) cmin = -3.0f;
        else {
            // weight != 0 needs a < amax, i.e. squared chord 4a < 4 amax.  The fp32 dot of two rounded unit
            // vectors is within ~4e-7 of the exact one: 2e-6 on the squared chord covers it with room.
            cmin = __double2float_rd(1.0 - 0.5 * (4.0 * amax + 2e-6));
        }
    }
    q.w = cmin;
    pk[k] = q;
}

// FILL = false: cnt[j] = number of candidates k < j of row j.  FILL = true: list[off[j] - list_base ...] = them,
// ascending.  One LANE per row: a warp owns 32 consecutive rows and walks the staged candidates one at a time
// (a broadcast shared-memory read), so every lane meets its row's predecessors in ascending order and appends
// them without any cross-lane prefix.  CTA = DG_LROWS consecutive rows; candidate tiles are staged once per CTA.
template <bool FILL>
__global__ void __launch_bounds__(DG_LWARPS * 32)
dag_list_kernel(const float4 *__restrict__ pk, int64_t row_begin, int64_t row_end, int *__restrict__ cnt,
                const int64_t *__restrict__ off, int64_t list_base, int *__restrict__ list, const DgDeal deal) {
    // [row_begin, row_end) are indices v into the rows this process solves: ob index j = dg_row(deal, v)
    // (world 1: all rows; the distributed solve builds the lists of its own rows only).  cnt / off / the
    // list segments are indexed by v.
    __shared__ float4 tile[DG_TILE];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // Row block b costs ~b: a CTA takes block blockIdx.x and its mirror image, so every CTA has the same work.
    const int64_t nblk = ceil_div64_dev(row_end - row_begin, DG_LROWS);
    for (int half = 0; half < 2; ++half) {
    const int64_t blk = half == 0 ? (int64_t)blockIdx.x : nblk - 1 - (int64_t)blockIdx.x;
    if (half == 1 && blk <= (int64_t)blockIdx.x) break;
    const int64_t v0 = row_begin + blk * DG_LROWS;
    const int64_t vw = v0 + warp * 32, v = vw + lane;
    const int64_t jw = dg_row(deal, vw);                              // first row of this warp
    const int64_t j = dg_row(deal, v);
    const bool valid = v < row_end;
    const int64_t jtop = dg_row(deal, (v0 + DG_LROWS < row_end ? v0 + DG_LROWS : row_end) - 1);         // last row of this CTA
    const float qnan = __int_as_float(0x7fc00000);                    // rows past the end: every test is false
    float4 me = make_float4(qnan, qnan, qnan, 0.f);
    if (valid) me = pk[j];
    int *out = list;
    if (FILL && valid) out = list + (off[v] - list_base);
    int count = 0;
    for (int64_t t0 = 0; t0 < jtop; t0 += DG_TILE) {
        __syncthreads();
        for (int i = threadIdx.x; i < DG_TILE; i += DG_LWARPS * 32) {
            const int64_t k = t0 + i;
            tile[i] = (k < jtop) ? pk[k] : make_float4(0.f, 0.f, 0.f, 3.0f);
        }
        __syncthreads();
        if (vw >= row_end) continue;
        // candidates k < jw precede every row of the warp
        const int64_t rem = jw - t0;
        const int full = rem <= 0 ? 0 : (rem < DG_TILE ? (int)rem : DG_TILE);
#pragma unroll 8
        for (int i = 0; i < full; ++i) {
            const float4 q = tile[i];
            const float dot = fmaf(me.x, q.x, fmaf(me.y, q.y, me.z * q.z));
            if (dot >= q.w) {
                if (FILL) out[count] = (int)(t0 + i);
                ++count;
            }
        }
        // the warp's own 32 rows: k < j per lane
        const int64_t last = dg_row(deal, vw + 31) - t0;
        const int lim = last < DG_TILE ? (int)last : DG_TILE;
        for (int i = full; i < lim; ++i) {
            const float4 q = tile[i];
            const float dot = fmaf(me.x, q.x, fmaf(me.y, q.y, me.z * q.z));
            if (t0 + i < j && dot >= q.w) {
                if (FILL) out[count] = (int)(t0 + i);
                ++count;
            }
        }
    }
    if (!FILL && valid) cnt[v] = count;
    }
}

// exclusive prefix sum of cnt[n] into off[n+1] (one CTA walking coalesced chunks of 1024; n is ~1e5..1e6)
__global__ void __launch_bounds__(1024) dag_scan_kernel(const int *__restrict__ cnt, int64_t n, int64_t *__restrict__ off) {
    __shared__ long long wsum[32];
    __shared__ long long carry_s;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t == 0) carry_s = 0;
    __syncthreads();
    for (int64_t b = 0; b < n; b += 1024) {
        const int64_t i = b + t;
        const long long v = (i < n) ? cnt[i] : 0;
        long long x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long y = __shfl_up_sync(DG_FULL, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) wsum[warp] = x;
        __syncthreads();
        if (warp == 0) {
            long long w = wsum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const long long y = __shfl_up_sync(DG_FULL, w, o);
                if (lane >= o) w += y;
            }
            wsum[lane] = w;
        }
        __syncthreads();
        const long long carry = carry_s;
        const long long excl = carry + (warp ? wsum[warp - 1] : 0) + x - v;
        if (i < n) off[i] = excl;
        __syncthreads();
        if (t == 1023) carry_s = carry + wsum[31];
        __syncthreads();
    }
    if (t == 0) off[n] = carry_s;
}

// ------------------------------------------------------------------------------------------
// the solve
// ------------------------------------------------------------------------------------------
template <typename T>
struct DgArgs {
    T *Ym;
    T *Yp;
    const double *ob_value;
    const double *ob_error;
    const uint8_t *ob_assim;
    const double *ob_thr;        // outlier threshold per ob (QC instantiations only)
    const double *geo;
    double *rec;
    unsigned long long *counters;
    const int64_t *off;
    const int *list;
    int64_t list_base;
    T *P;                        // published ye rows, stride 32*MC, sentinel-initialised
    double *S;                   // published scalars [nobs][2] = c1*innov, c1*beta; sentinel-initialised
    int *ticket;
    int *status;                 // != 0: watchdog fired (value = 1 + index of the record that never arrived)
    unsigned long long watchdog_ns;
    int64_t nobs, row_begin, row_end;
    int nens, loc_mode;
    double inv_n;                // 1 / nens (IEEE division on the host, as on the device): a parameter holds no register
    // distributed variant (DIST): the rows dg_row(deal, t) are solved here; records are published into the P / S
    // buffers of every GPU of the group (peer memory over NVLink), readers always poll their own copy
    int world, rank;
    DgDeal deal;
    void *P_peer[8];
    void *S_peer[8];
};

__device__ __forceinline__ void dg_ld16(const void *p, unsigned long long &a, unsigned long long &b) {
    asm volatile("ld.relaxed.gpu.global.v2.b64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ void dg_st16(void *p, unsigned long long a, unsigned long long b) {
    asm volatile("st.relaxed.gpu.global.v2.b64 [%0], {%1, %2};" ::"l"(p), "l"(a), "l"(b) : "memory");
}
// 256-bit accesses (sm_100): one instruction per 32-byte sector
__device__ __forceinline__ void dg_ld32(const void *p, unsigned long long &a, unsigned long long &b, unsigned long long &c,
                                        unsigned long long &d) {
    asm volatile("ld.relaxed.gpu.global.v4.b64 {%0, %1, %2, %3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p) : "memory");
}
__device__ __forceinline__ void dg_st32(void *p, unsigned long long a, unsigned long long b, unsigned long long c,
                                        unsigned long long d) {
    asm volatile("st.relaxed.gpu.global.v4.b64 [%0], {%1, %2, %3, %4};" ::"l"(p), "l"(a), "l"(b), "l"(c), "l"(d) : "memory");
}

// system-scope stores for records published into peer memory
__device__ __forceinline__ void dg_st16_sys(void *p, unsigned long long a, unsigned long long b) {
    asm volatile("st.relaxed.sys.global.v2.b64 [%0], {%1, %2};" ::"l"(p), "l"(a), "l"(b) : "memory");
}
__device__ __forceinline__ void dg_st32_sys(void *p, unsigned long long a, unsigned long long b, unsigned long long c,
                                            unsigned long long d) {
    asm volatile("st.relaxed.sys.global.v4.b64 [%0], {%1, %2, %3, %4};" ::"l"(p), "l"(a), "l"(b), "l"(c), "l"(d) : "memory");
}

// The sentinel is recognised by 32 bits per element: the high half of a double / the whole float equal to
// 0xFFFFFFFF (a NaN either way; the writer replaces such a value by the canonical quiet NaN).
__device__ __forceinline__ unsigned dg_hi(unsigned long long w) { return (unsigned)(w >> 32); }
__device__ __forceinline__ unsigned dg_lo(unsigned long long w) { return (unsigned)w; }

template <typename T> struct DgWord;
template <> struct DgWord<double> {
    static constexpr int PER = 1;                                    // elements per 64-bit word
    static __device__ __forceinline__ bool pending(unsigned long long w) { return dg_hi(w) == 0xFFFFFFFFu; }
    static __device__ __forceinline__ void unpack(unsigned long long w, double *o) { o[0] = __longlong_as_double((long long)w); }
    static __device__ __forceinline__ unsigned long long pack(const double *v) {
        const unsigned long long w = (unsigned long long)__double_as_longlong(v[0]);
        return dg_hi(w) == 0xFFFFFFFFu ? 0x7FF8000000000000ull : w;
    }
};
template <> struct DgWord<float> {
    static constexpr int PER = 2;
    static __device__ __forceinline__ bool pending(unsigned long long w) {
        return dg_lo(w) == 0xFFFFFFFFu || dg_hi(w) == 0xFFFFFFFFu;
    }
    static __device__ __forceinline__ void unpack(unsigned long long w, float *o) {
        o[0] = __uint_as_float(dg_lo(w));
        o[1] = __uint_as_float(dg_hi(w));
    }
    static __device__ __forceinline__ unsigned long long pack(const float *v) {
        unsigned lo = __float_as_uint(v[0]), hi = __float_as_uint(v[1]);
        if (lo == 0xFFFFFFFFu) lo = 0x7FC00000u;
        if (hi == 0xFFFFFFFFu) hi = 0x7FC00000u;
        return (unsigned long long)lo | ((unsigned long long)hi << 32);
    }
};
__device__ __forceinline__ unsigned long long dg_pack_scalar(double v) {
    const unsigned long long w = (unsigned long long)__double_as_longlong(v);
    return dg_hi(w) == 0xFFFFFFFFu ? 0x7FF8000000000000ull : w;
}

__device__ __forceinline__ double dg_warp_sum_shfl(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(DG_FULL, v, o);
    return v;
}
__device__ __forceinline__ void dg_dmma(double &c0, double &c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
        : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
// Sum of one value per lane, result in every lane, on the (otherwise idle) FP64 tensor pipe: the kernel is bound by
// the load/store pipe, which also executes shuffles (10 SHFL for a 64-bit butterfly), and a DMMA chain has half the
// latency of five shuffle levels.  m8n8k4 fragments: A[8x4] lane l -> A[l/4][l%4]; B[4x8] lane l -> B[l%4][l/4];
// C[8x8] lane l -> C[l/4][2(l%4)], C[l/4][2(l%4)+1].
//   1. A = v, B = 1            -> every lane of group r = l/4 holds R_r = sum of the group's 4 values
//   2. A = [k == 0], B = R     -> lane l holds R_{2m}, R_{2m+1} (m = l%4), exactly;  u_m = R_{2m} + R_{2m+1}
//   3. A = u (A[r][k] = u_k), B = 1 -> every lane holds u_0 + u_1 + u_2 + u_3
__device__ __forceinline__ double dg_warp_sum(double v) {
#if DG_DMMA_REDUCE
    const int lane = threadIdx.x & 31;
    double r0 = 0.0, r1 = 0.0;
    dg_dmma(r0, r1, v, 1.0);
    double p0 = 0.0, p1 = 0.0;
    dg_dmma(p0, p1, (lane & 3) == 0 ? 1.0 : 0.0, r0);
    const double u = p0 + p1;
    double t0 = 0.0, t1 = 0.0;
    dg_dmma(t0, t1, u, 1.0);
    return t0;
#else
    return dg_warp_sum_shfl(v);
#endif
}

// One published record as held by a lane: NW 64-bit words of the ye row + the two scalars
// s[0] = c1*innov (mean gain per unit weight*dot), s[1] = c1*beta (perturbation factor per unit weight*dot).
template <int NW>
struct DgRec {
    unsigned long long w[NW];
    unsigned long long s[2];
};

template <typename T, int MC>
struct DgCfg {
    static constexpr int NW = MC / DgWord<T>::PER;                   // 64-bit words per lane
    static_assert(NW >= 2 && NW % 2 == 0, "a lane must own whole 16-byte chunks");
};

template <typename T, int MC>
__device__ __forceinline__ void dg_fetch(const DgArgs<T> &a, int k, int lane, DgRec<DgCfg<T, MC>::NW> &r) {
    constexpr int NW = DgCfg<T, MC>::NW;
    const unsigned long long *p = reinterpret_cast<const unsigned long long *>(a.P + ((int64_t)k * 32 + lane) * MC);
    if (lane * MC >= a.nens) {                    // pad lane: nothing to read, never pending
#pragma unroll
        for (int c = 0; c < NW; ++c) r.w[c] = 0ull;
    } else if constexpr (NW % 4 == 0) {
#pragma unroll
        for (int c = 0; c < NW; c += 4) dg_ld32(p + c, r.w[c], r.w[c + 1], r.w[c + 2], r.w[c + 3]);
    } else {
#pragma unroll
        for (int c = 0; c < NW; c += 2) dg_ld16(p + c, r.w[c], r.w[c + 1]);
    }
    dg_ld16(a.S + (int64_t)k * 2, r.s[0], r.s[1]);
}

template <typename T, int MC>
__device__ __forceinline__ bool dg_ready(const DgRec<DgCfg<T, MC>::NW> &r) {
    constexpr int NW = DgCfg<T, MC>::NW;
    bool ok = (dg_hi(r.s[0]) != 0xFFFFFFFFu) && (dg_hi(r.s[1]) != 0xFFFFFFFFu);
#pragma unroll
    for (int c = 0; c < NW; ++c) ok = ok && !DgWord<T>::pending(r.w[c]);
    return __all_sync(DG_FULL, ok);
}

// Waits until the polled word of ob k's record has been written.  Returns false when the watchdog fired (here
// or elsewhere).  Takes no reference to the caller's record so that it stays in registers.
__device__ __forceinline__ unsigned long long dg_globaltimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __noinline__ bool dg_wait(const double *S, int *status, unsigned long long watchdog_ns, int k, int lane) {
    const double *s = S + (int64_t)k * 2;
    unsigned polls = 0;
    unsigned long long t0 = 0;
    while (true) {
        unsigned long long b0, b1;
        dg_ld16(s, b0, b1);
        if (dg_hi(b1) != 0xFFFFFFFFu) return true;
        ++polls;
        if (polls > 1) __nanosleep(polls < 8 ? 50 : (polls < 32 ? 200 : 500));
        if ((polls & 1023u) == 0) {
            // wall-clock watchdog (the poll count says little on a time-sliced or preempted GPU)
            if (*reinterpret_cast<volatile int *>(status) != 0) return false;
            const unsigned long long now = dg_globaltimer();
            if (t0 == 0) t0 = now;
            else if (now - t0 > watchdog_ns) {
                if (lane == 0) atomicCAS(status, 0, k + 1);
                return false;
            }
        }
    }
}

// Per-row state of a warp while it walks its predecessor list.
template <typename T, int MC>
struct DgRow {
    T x[MC];
    double mj;
    int kl;             // this lane's list entry of the current batch
    double wl;          // and its weight
    unsigned m;         // entries of the batch still to apply
    int k;              // ob whose record is in `cur`
    double w;
    bool dead;
};

// One step of the pipelined walk: `cur` holds (maybe incompletely) the record of ob r.k.  Makes it complete,
// starts the fetch of the next entry into `nxt`, applies cur.  Returns false when the batch is exhausted (or dead).
template <typename T, int MC>
__device__ __forceinline__ bool dg_step(const DgArgs<T> &a, int lane, DgRow<T, MC> &r, DgRec<DgCfg<T, MC>::NW> &cur,
                                        DgRec<DgCfg<T, MC>::NW> &nxt) {
    constexpr int NW = DgCfg<T, MC>::NW;
    constexpr int PER = DgWord<T>::PER;
    if (!dg_ready<T, MC>(cur)) {
        if (r.m == 0) {
            // The last entry of a batch of 32 predecessors is where a row sits while it is the next link of the
            // dependency chain: poll the record itself, without back-off, so that the hop does not pay a sleep interval
            // plus a second round trip to L2 after the wake-up.  (Few warps are in this state at a time.)
            unsigned spins = 0;
            unsigned long long t0 = 0;
            do {
                __nanosleep(20);
                dg_fetch<T, MC>(a, r.k, lane, cur);
                if ((++spins & 8191u) == 0) {
                    if (*reinterpret_cast<volatile int *>(a.status) != 0) { r.dead = true; return false; }
                    const unsigned long long now = dg_globaltimer();
                    if (t0 == 0) t0 = now;
                    else if (now - t0 > a.watchdog_ns) {
                        if (lane == 0) atomicCAS(a.status, 0, r.k + 1);
                        r.dead = true;
                        return false;
                    }
                }
            } while (!dg_ready<T, MC>(cur));
        } else {
            do {
                if (!dg_wait(a.S, a.status, a.watchdog_ns, r.k, lane)) { r.dead = true; return false; }
                dg_fetch<T, MC>(a, r.k, lane, cur);
            } while (!dg_ready<T, MC>(cur));
        }
    }
    const bool more = r.m != 0;
    const double w = r.w;
    if (more) {                                   // speculative: re-fetched at its turn if not complete yet
        const int i = __ffs(r.m) - 1;
        r.m &= r.m - 1;
        r.k = __shfl_sync(DG_FULL, r.kl, i);
        r.w = __shfl_sync(DG_FULL, r.wl, i);
        dg_fetch<T, MC>(a, r.k, lane, nxt);
    }
    // rank-1 update of this row by the ob in cur   (ensrf.py:95, :115-119, :130, :135-141)
    T ye[MC];
#pragma unroll
    for (int c = 0; c < NW; ++c) DgWord<T>::unpack(cur.w[c], ye + c * PER);
    T d0 = 0, d1 = 0;
#pragma unroll
    for (int q = 0; q < MC; q += 2) {
        d0 += r.x[q] * ye[q];
        d1 += r.x[q + 1] * ye[q + 1];
    }
    const double wd = w * dg_warp_sum((double)(d0 + d1));                 // loc * (row . ye)
    r.mj += wd * __longlong_as_double((long long)cur.s[0]);                // + kmat * innov
    const T f = (T)(wd * __longlong_as_double((long long)cur.s[1]));       // beta * kmat
#pragma unroll
    for (int q = 0; q < MC; ++q) r.x[q] -= f * ye[q];
    return more;
}

// |innov| > t sqrt(kdenom) in float64 with a correctly rounded sqrt (DESIGN.md section 4.7).  Not inlined, and called
// by lane 0 only: inlined, the threshold load and the sqrt's slow path raised the register pressure of the whole
// kernel and added spills to the predecessor loop.
__device__ __noinline__ bool dg_outlier(const double *thr, int64_t j, double innov, double kdenom) {
    return fabs(innov) > thr[j] * sqrt(kdenom);
}

// QC: outlier check of every assimilated ob against its in-loop prior (DESIGN.md section 4.7).  A rejected ob still
// publishes its record, with scalars (0, 0): its successors' lists were built from the user flags and wait for it,
// and zero scalars make their update by it exactly the identity.
template <typename T, int MC, bool DIST, bool QC>
__global__ void __launch_bounds__(DG_WARPS * 32, DG_MINBLOCKS) dag_solve_kernel(const DgArgs<T> a) {
    constexpr int NW = DgCfg<T, MC>::NW;
    constexpr int PER = DgWord<T>::PER;
    const int lane = threadIdx.x & 31;
    const int64_t nobs = a.nobs;
    const int nens = a.nens;
    const bool gc = a.loc_mode == EXB_LOC_GC;
    unsigned long long npairs = 0;

    while (true) {
        int t = 0;
        if (lane == 0) t = atomicAdd(a.ticket, 1);
        t = __shfl_sync(DG_FULL, t, 0);
        int64_t j = a.row_begin + t;
        if (DIST) j = dg_row(a.deal, t);                  // t-th row of this rank (row_begin is 0 when distributed)
        if (j >= a.row_end) break;

        // ---- this row: perturbations (lane owns members [MC*lane, MC*lane+MC)), mean, geometry ----
        DgRow<T, MC> r;
#pragma unroll
        for (int i = 0; i < MC; ++i) {
            const int m = lane * MC + i;
            r.x[i] = (m < nens) ? __ldcg(a.Yp + j * nens + m) : (T)0;
        }
        r.mj = (double)__ldcg(a.Ym + j);
        r.dead = false;
        const double ux = a.geo[GEO_UX * nobs + j], uy = a.geo[GEO_UY * nobs + j], uz = a.geo[GEO_UZ * nobs + j];
        const int64_t oi = DIST ? (int64_t)t : j;       // lists are indexed by the rank's own row number when distributed
        const int64_t lb = a.off[oi] - a.list_base, le = a.off[oi + 1] - a.list_base;

        // ---- predecessors, 32 at a time: weights lane-parallel, updates strictly in list order ----
        int kl_next = (lb + lane < le) ? __ldg(a.list + lb + lane) : -1;
        for (int64_t base = lb; base < le; base += 32) {
            r.kl = kl_next;
            kl_next = (base + 32 + lane < le) ? __ldg(a.list + base + 32 + lane) : -1;
            r.wl = 0.0;
            if (r.kl >= 0) {
                r.wl = 1.0;
                if (gc)
                    r.wl = loc_weight(hav_a(ux, uy, uz, __ldg(a.geo + GEO_UX * nobs + r.kl), __ldg(a.geo + GEO_UY * nobs + r.kl),
                                            __ldg(a.geo + GEO_UZ * nobs + r.kl)),
                                      __ldg(a.geo + GEO_INVHW * nobs + r.kl), __ldg(a.geo + GEO_AMAX * nobs + r.kl));
            }
            r.m = __ballot_sync(DG_FULL, r.wl != 0.0);
            if (!r.m) continue;
            if (lane == 0) npairs += __popc(r.m);
            DgRec<NW> ra, rb;
            const int i = __ffs(r.m) - 1;
            r.m &= r.m - 1;
            r.k = __shfl_sync(DG_FULL, r.kl, i);
            r.w = __shfl_sync(DG_FULL, r.wl, i);
            dg_fetch<T, MC>(a, r.k, lane, ra);
            while (true) {                        // ping-pong between the two record buffers
                if (!dg_step<T, MC>(a, lane, r, ra, rb)) break;
                if (!dg_step<T, MC>(a, lane, r, rb, ra)) break;
            }
            if (r.dead) break;
        }
        if (r.dead) break;

        // ---- this ob's own step: ensrf.py:61-91, :135, :144-149 ----
        // (its own value / error / flag are loaded here and not at the start of the row: carried through the
        // predecessor loop they cost registers the loop does not have -- measured 18.7 against 17.6 ms)
        const double my_val = a.ob_value[j], my_err = a.ob_error[j];
        const bool act = a.ob_assim[j] != 0;
        const double sq_err = sqrt(my_err);
        // The ye row goes out first (data before the polled word): its stores travel while the scalars are computed.
        // Skipped obs are never anyone's predecessor: their scalars stay unpublished; the distributed variant still
        // publishes their ye row, so that every rank ends up with all ye rows in its own record buffer.
        if (act || DIST) {
            unsigned long long pw[NW];
#pragma unroll
            for (int c = 0; c < NW; ++c) pw[c] = DgWord<T>::pack(r.x + c * PER);
            if (!DIST) {
                unsigned long long *p = reinterpret_cast<unsigned long long *>(a.P + (j * 32 + lane) * MC);
                if (lane * MC < nens) {
                    if constexpr (NW % 4 == 0) {
#pragma unroll
                        for (int c = 0; c < NW; c += 4) dg_st32(p + c, pw[c], pw[c + 1], pw[c + 2], pw[c + 3]);
                    } else {
#pragma unroll
                        for (int c = 0; c < NW; c += 2) dg_st16(p + c, pw[c], pw[c + 1]);
                    }
                }
            } else {
                // own copy first (local readers are the closest in index; gpu scope is enough for them), then the peers
                for (int q = 0; q < a.world; ++q) {
                    const int dst = (a.rank + q) % a.world;
                    unsigned long long *p = reinterpret_cast<unsigned long long *>(static_cast<T *>(a.P_peer[dst]) + (j * 32 + lane) * MC);
                    if (lane * MC < nens) {
                        if (q == 0) {
                            if constexpr (NW % 4 == 0) {
#pragma unroll
                                for (int c = 0; c < NW; c += 4) dg_st32(p + c, pw[c], pw[c + 1], pw[c + 2], pw[c + 3]);
                            } else {
#pragma unroll
                                for (int c = 0; c < NW; c += 2) dg_st16(p + c, pw[c], pw[c + 1]);
                            }
                        } else if constexpr (NW % 4 == 0) {
#pragma unroll
                            for (int c = 0; c < NW; c += 4) dg_st32_sys(p + c, pw[c], pw[c + 1], pw[c + 2], pw[c + 3]);
                        } else {
#pragma unroll
                            for (int c = 0; c < NW; c += 2) dg_st16_sys(p + c, pw[c], pw[c + 1]);
                        }
                    }
                }
            }
        }
        double s0 = 0.0, q0 = 0.0;
#pragma unroll
        for (int q = 0; q < MC; ++q) { const double v = (double)r.x[q]; s0 += v; q0 += v * v; }
        const double rs = dg_warp_sum(s0), rq = dg_warp_sum(q0);
        const double mj = r.mj;
        const double mean = rs * a.inv_n;
        const double varye = fmax(rq * a.inv_n - mean * mean, 0.0);                    // np.var, ddof 0
        const double innov = my_val - mj;
        const double kdenom = varye + my_err;
        const double c1 = 1.0 / ((double)(nens - 1) * kdenom);
        const double beta = 1.0 / (1.0 + sq_err * rsqrt(kdenom));                    // 1/(1+sqrt(R/kdenom))
        bool rej = false;                 // outlier: only lane 0 decides, and only lane 0 publishes and records
        if (act && lane == 0) {
            if constexpr (QC) rej = dg_outlier(a.ob_thr, j, innov, kdenom);
            const unsigned long long s0w = rej ? 0ull : dg_pack_scalar(c1 * innov);
            const unsigned long long s1w = rej ? 0ull : dg_pack_scalar(c1 * beta);
            if (!DIST) {
                dg_st16(a.S + j * 2, s0w, s1w);
            } else {
                for (int q = 0; q < a.world; ++q) {
                    const int dst = (a.rank + q) % a.world;
                    if (q == 0) dg_st16(static_cast<double *>(a.S_peer[dst]) + j * 2, s0w, s1w);
                    else dg_st16_sys(static_cast<double *>(a.S_peer[dst]) + j * 2, s0w, s1w);
                }
            }
        }
        // outputs of the C ABI: ye_j / mye_j in place, per-ob records
#pragma unroll
        for (int i = 0; i < MC; ++i) {
            const int mm = lane * MC + i;
            if (mm < nens) a.Yp[j * nens + mm] = r.x[i];
        }
        if (lane == 0) {
            a.Ym[j] = (T)mj;
            a.rec[REC_PRIOR_MEAN * nobs + j] = mj;                                   // ensrf.py:66
            a.rec[REC_PRIOR_VAR * nobs + j] = varye;                                 // ensrf.py:70
            a.rec[REC_INNOV * nobs + j] = innov;
            a.rec[REC_C1 * nobs + j] = rej ? 0.0 : c1;
            a.rec[REC_BETA * nobs + j] = beta;
            a.rec[REC_ASSIM * nobs + j] = act && !rej ? 1.0 : 0.0;
            if (act && !rej) {
                // the ob's own row: weight at distance 0, kcov = ye.ye/(N-1)   (ensrf.py:144-147)
                const double wself = gc ? loc_weight(0.0, a.geo[GEO_INVHW * nobs + j], a.geo[GEO_AMAX * nobs + j]) : 1.0;
                const double kmat = wself * rq * c1;
                const double shrink = 1.0 - beta * kmat;
                a.rec[REC_POST_MEAN * nobs + j] = mj + kmat * innov;
                a.rec[REC_POST_VAR * nobs + j] = varye * shrink * shrink;
                if (wself != 0.0) npairs++;
            } else {
                a.rec[REC_POST_MEAN * nobs + j] = nan("");
                a.rec[REC_POST_VAR * nobs + j] = nan("");
            }
        }
    }
    if (a.counters && lane == 0 && npairs) atomicAdd(&a.counters[0], npairs);
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static unsigned long long dg_watchdog_ns(int64_t nobs) {
    double sec = DG_WATCHDOG_S + 1e-4 * (double)nobs;
    if (const char *e = getenv("EXB_WATCHDOG_S")) { const double v = atof(e); if (v > 0.0) sec = v; }
    return (unsigned long long)(sec * 1e9);
}

namespace {
struct AsyncBuf {
    void *p = nullptr;
    cudaStream_t st;
    explicit AsyncBuf(cudaStream_t s) : st(s) {}
    ~AsyncBuf() { if (p) cudaFreeAsync(p, st); }
    cudaError_t alloc(size_t bytes) { return exb_malloc_async(&p, bytes ? bytes : 1, st); }
    template <typename U> U *as() { return static_cast<U *>(p); }
};
}   // namespace

// ------------------------------------------------------------------------------------------
// plan = everything that depends on the observation geometry only (predecessor lists).  It can be built on a side
// stream while the ob priors are still being computed (exb_obs_plan_create) and is consumed by
// exb_obs_solve_planned_*; exb_obs_solve_* builds a temporary one.
// ------------------------------------------------------------------------------------------
struct ExbObsPlan {
    int64_t nobs = 0;
    int loc_mode = 0;
    DgDeal deal{1, 1, 0};                 // rows of this plan: dg_row(deal, v) (distributed solve: blocks dealt to the ranks)
    int64_t nrows = 0;                    // number of those rows
    cudaStream_t st = nullptr;            // stream the plan was built on (its buffers are freed there)
    float4 *pk = nullptr;
    int64_t *off = nullptr;
    int *list = nullptr;                  // filled when all lists fit one block, else built per block at solve time
    std::vector<int64_t> off_h;
    bool dense = false;                   // dependency graph too dense for the dependency-driven solve to pay
    int64_t budget = 0;
    cudaEvent_t ready = nullptr, used = nullptr;
    bool was_used = false;
    bool finished = false;
    int64_t *off_pinned = nullptr;        // page-locked staging buffer of the row offsets (exb_pinned_acquire)
};

static void dg_plan_free(ExbObsPlan *pl) {
    if (!pl) return;
    if (pl->off_pinned) { cudaStreamSynchronize(pl->st); exb_pinned_release(pl->off_pinned); pl->off_pinned = nullptr; }
    if (pl->was_used && pl->used) cudaStreamWaitEvent(pl->st, pl->used, 0);
    if (pl->pk) cudaFreeAsync(pl->pk, pl->st);
    if (pl->off) cudaFreeAsync(pl->off, pl->st);
    if (pl->list) cudaFreeAsync(pl->list, pl->st);
    if (pl->ready) cudaEventDestroy(pl->ready);
    if (pl->used) cudaEventDestroy(pl->used);
    delete pl;
}

// Step 1 (asynchronous): enqueues packing, the count pass, the prefix sum and the download of the row offsets on st.
static int dg_plan_begin(const double *geo, const uint8_t *ob_assim, int64_t nobs, int loc_mode, cudaStream_t st, ExbObsPlan **out,
                         DgDeal deal = DgDeal{1, 1, 0}) {
    *out = nullptr;
    if (nobs >= 0x7fffffff) return EXB_ERR_UNSUPPORTED;
    ExbObsPlan *pl = new ExbObsPlan();
    pl->nobs = nobs; pl->loc_mode = loc_mode; pl->st = st;
    pl->deal = deal;
    {
        const int64_t cyc = (int64_t)deal.block * deal.world, rem = nobs % cyc - (int64_t)deal.rank * deal.block;
        pl->nrows = (nobs / cyc) * deal.block + (rem < 0 ? 0 : (rem > deal.block ? deal.block : rem));
    }
    const int64_t nrows = pl->nrows > 0 ? pl->nrows : 1;
    struct Guard { ExbObsPlan *p; ~Guard() { if (p) dg_plan_free(p); } } guard{pl};
    int *cnt = nullptr;
    EXB_CUDA(cudaEventCreateWithFlags(&pl->ready, cudaEventDisableTiming));
    EXB_CUDA(cudaEventCreateWithFlags(&pl->used, cudaEventDisableTiming));
    EXB_CUDA(exb_malloc_async(&pl->pk, (size_t)nobs * sizeof(float4), st));
    EXB_CUDA(exb_malloc_async(&pl->off, (size_t)(nrows + 1) * sizeof(int64_t), st));
    EXB_CUDA(exb_malloc_async(&cnt, (size_t)nrows * sizeof(int), st));
    dag_pack_kernel<<<(unsigned)ceil_div64(nobs, 256), 256, 0, st>>>(geo, ob_assim, nobs, loc_mode, pl->pk);
    EXB_CUDA(cudaMemsetAsync(cnt, 0, (size_t)nrows * sizeof(int), st));
    dag_list_kernel<false><<<(unsigned)ceil_div64(ceil_div64(nrows, DG_LROWS), 2), DG_LWARPS * 32, 0, st>>>(
        pl->pk, 0, pl->nrows, cnt, nullptr, 0, nullptr, deal);
    dag_scan_kernel<<<1, 1024, 0, st>>>(cnt, nrows, pl->off);
    exb_count_launches(3);
    cudaFreeAsync(cnt, st);
    EXB_CUDA(cudaGetLastError());
    pl->off_h.resize((size_t)nrows + 1);
    {
        void *hp = nullptr;
        const int rcp = exb_pinned_acquire((size_t)(nrows + 1) * sizeof(int64_t), &hp);
        if (rcp != EXB_OK) return rcp;
        pl->off_pinned = static_cast<int64_t *>(hp);
        EXB_CUDA(cudaMemcpyAsync(pl->off_pinned, pl->off, (size_t)(nrows + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    }
    guard.p = nullptr;
    *out = pl;
    return EXB_OK;
}

// Step 2: waits for the offsets (synchronises the plan's stream), sizes and fills the lists.
static int dg_plan_finish(ExbObsPlan *pl) {
    if (pl->finished) return EXB_OK;
    const int64_t nobs = pl->nobs, nrows = pl->nrows > 0 ? pl->nrows : 1;
    cudaStream_t st = pl->st;
    EXB_CUDA(cudaStreamSynchronize(st));
    if (pl->off_pinned) {
        memcpy(pl->off_h.data(), pl->off_pinned, ((size_t)nrows + 1) * sizeof(int64_t));
        exb_pinned_release(pl->off_pinned);
        pl->off_pinned = nullptr;
    }
    const int64_t total = pl->off_h[(size_t)nrows];
    const double dense = 0.5 * (double)nobs * (double)(nobs - 1) / (double)pl->deal.world;
    pl->dense = nobs > 2048 && (double)total > 0.5 * dense;
    pl->budget = (int64_t)1 << 30;                                      // list entries per row block (4 GiB)
    if (const char *e = getenv("EXB_DAG_BUDGET")) {
        const long long v = atoll(e);
        if (v > 0) pl->budget = v;
    }
    if (!pl->dense && total > 0 && total <= pl->budget) {
        EXB_CUDA(exb_malloc_async(&pl->list, (size_t)total * sizeof(int), st));
        dag_list_kernel<true><<<(unsigned)ceil_div64(ceil_div64(nrows, DG_LROWS), 2), DG_LWARPS * 32, 0, st>>>(
            pl->pk, 0, pl->nrows, nullptr, pl->off, 0, pl->list, pl->deal);
        exb_count_launches(1);
        EXB_CUDA(cudaGetLastError());
    }
    EXB_CUDA(cudaEventRecord(pl->ready, st));
    pl->finished = true;
    return EXB_OK;
}

static int dg_plan_build(const double *geo, const uint8_t *ob_assim, int64_t nobs, int loc_mode, cudaStream_t st, ExbObsPlan **out) {
    const int rc = dg_plan_begin(geo, ob_assim, nobs, loc_mode, st, out);
    if (rc != EXB_OK) return rc;
    const int rc2 = dg_plan_finish(*out);
    if (rc2 != EXB_OK) { dg_plan_free(*out); *out = nullptr; }
    return rc2;
}

template <typename T, int MC, bool DIST, bool QC>
static int dg_run(DgArgs<T> a, const ExbObsPlan &pl, cudaStream_t st) {
    int dev = 0, sms = 0, per_sm = 0;
    EXB_CUDA(cudaGetDevice(&dev));
    EXB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    EXB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, dag_solve_kernel<T, MC, DIST, QC>, DG_WARPS * 32, 0));
    if (per_sm < 1) return EXB_ERR_UNSUPPORTED;
    const int64_t nobs = a.nobs;
    const std::vector<int64_t> &off_h = pl.off_h;
    AsyncBuf P(st), S(st), list(st), ticket(st);
    if (!DIST) {
        const size_t p_bytes = (size_t)nobs * 32 * MC * sizeof(T), s_bytes = (size_t)nobs * 2 * sizeof(double);
        EXB_CUDA(P.alloc(p_bytes));
        EXB_CUDA(S.alloc(s_bytes));
        EXB_CUDA(cudaMemsetAsync(P.p, 0xFF, p_bytes, st));
        EXB_CUDA(cudaMemsetAsync(S.p, 0xFF, s_bytes, st));
        a.P = P.as<T>();
        a.S = S.as<double>();
    } else {
        // the caller owns the (symmetric) buffers, has filled them with the sentinel and synchronised the group
        a.P = static_cast<T *>(a.P_peer[a.rank]);
        a.S = static_cast<double *>(a.S_peer[a.rank]);
    }
    EXB_CUDA(ticket.alloc(sizeof(int)));
    a.ticket = ticket.as<int>();
    a.off = pl.off;
    // row blocks whose predecessor lists fit the budget (one block, filled by the plan, in the usual case)
    int64_t r0 = 0, max_block = 0;
    std::vector<std::pair<int64_t, int64_t>> blocks;
    if (pl.list || off_h.back() == 0) {
        blocks.push_back({0, nobs});
    } else {
        while (r0 < nobs) {
            int64_t r1 = r0 + 1;
            while (r1 < nobs && off_h[r1 + 1] - off_h[r0] <= pl.budget) ++r1;
            blocks.push_back({r0, r1});
            if (off_h[r1] - off_h[r0] > max_block) max_block = off_h[r1] - off_h[r0];
            r0 = r1;
        }
        EXB_CUDA(list.alloc((size_t)max_block * sizeof(int)));
    }
    a.list = pl.list ? pl.list : list.as<int>();
    for (auto &b : blocks) {
        a.row_begin = b.first;
        a.row_end = b.second;
        a.list_base = DIST ? 0 : off_h[b.first];
        const int64_t nrows = b.second - b.first;
        if (!pl.list && !DIST && off_h[b.second] > off_h[b.first]) {
            dag_list_kernel<true><<<(unsigned)ceil_div64(ceil_div64(nrows, DG_LROWS), 2), DG_LWARPS * 32, 0, st>>>(
                pl.pk, b.first, b.second, nullptr, a.off, a.list_base, list.as<int>(), DgDeal{1, 1, 0});
            exb_count_launches(1);
        }
        EXB_CUDA(cudaMemsetAsync(a.ticket, 0, sizeof(int), st));
        int64_t grid = (int64_t)sms * per_sm;
        const int64_t need = ceil_div64(DIST ? pl.nrows + 1 : nrows, DG_WARPS);
        if (grid > need) grid = need;
        dag_solve_kernel<T, MC, DIST, QC><<<(unsigned)grid, DG_WARPS * 32, 0, st>>>(a);
        exb_count_launches(1);
    }
    return exb_check_launch("dag_solve_kernel");
}

// members per lane (MC) and outlier check (a.ob_thr != NULL) -> kernel instantiation
template <typename T, bool DIST>
static int dg_dispatch(const DgArgs<T> &a, const ExbObsPlan &pl, cudaStream_t st) {
    const bool qc = a.ob_thr != nullptr;
    if (a.nens <= 128) return qc ? dg_run<T, 4, DIST, true>(a, pl, st) : dg_run<T, 4, DIST, false>(a, pl, st);
    if (a.nens <= 256) return qc ? dg_run<T, 8, DIST, true>(a, pl, st) : dg_run<T, 8, DIST, false>(a, pl, st);
    return EXB_ERR_UNSUPPORTED;
}

// force = false: returns EXB_ERR_UNSUPPORTED when the dependency graph is too dense for this method to pay
// (the caller then uses the panel kernel).  plan may be null (a temporary one is built on st).
template <typename T>
int exb_obs_solve_dag(T *Ym, T *Yp, const double *ob_value, const double *ob_error, const uint8_t *ob_assim,
                      const double *ob_thr, const double *geo, int64_t nobs, int nens, int loc_mode, double *rec,
                      unsigned long long *counters, cudaStream_t st, bool force, void *plan_in) {
    ExbObsPlan *pl = static_cast<ExbObsPlan *>(plan_in), *tmp = nullptr;
    if (!pl) {
        const int rc = dg_plan_build(geo, ob_assim, nobs, loc_mode, st, &tmp);
        if (rc != EXB_OK) return rc;
        pl = tmp;
    } else {
        if (pl->nobs != nobs || pl->loc_mode != loc_mode || pl->deal.world != 1) {
            exb_set_error("exb_obs_solve: the plan was built for another observation set (or for a distributed solve)");
            return EXB_ERR_ARG;
        }
        const int rcf = dg_plan_finish(pl);
        if (rcf != EXB_OK) return rcf;
        EXB_CUDA(cudaStreamWaitEvent(st, pl->ready, 0));
    }
    struct TmpGuard { ExbObsPlan *p; ~TmpGuard() { if (p) dg_plan_free(p); } } tguard{tmp};
    if (!force && pl->dense) return EXB_ERR_UNSUPPORTED;
    DgArgs<T> a;
    {
        int *sh = nullptr, *sd = nullptr;
        const int rcs = exb_status_slot_next(&sh, &sd);
        if (rcs != EXB_OK) return rcs;
        EXB_CUDA(cudaMemsetAsync(sd, 0, sizeof(int), st));      // stream-ordered: an earlier solve's verdict is its own
        a.status = sd;
        a.watchdog_ns = dg_watchdog_ns(nobs);
    }
    a.Ym = Ym; a.Yp = Yp; a.ob_value = ob_value; a.ob_error = ob_error; a.ob_assim = ob_assim; a.ob_thr = ob_thr;
    a.geo = geo; a.rec = rec;
    a.counters = counters; a.off = pl->off; a.list = nullptr; a.list_base = 0; a.P = nullptr; a.S = nullptr;
    a.ticket = nullptr; a.nobs = nobs; a.row_begin = 0; a.row_end = nobs; a.nens = nens;
    a.loc_mode = loc_mode; a.inv_n = 1.0 / (double)nens;
    a.world = 1; a.rank = 0; a.deal = DgDeal{1, 1, 0};
    for (int q = 0; q < 8; ++q) { a.P_peer[q] = nullptr; a.S_peer[q] = nullptr; }
    const int rc = dg_dispatch<T, false>(a, *pl, st);
    if (!tmp) {
        cudaEventRecord(pl->used, st);
        pl->was_used = true;
    } else {
        // the temporary plan's buffers are freed on st, after the kernels above
        tmp->was_used = false;
    }
    return rc;
}

// Distributed obs-space solve: rank `rank` of `world` (<= 8 GPUs of one NVLink domain) solves the rows j with
// j % world == rank and publishes their records into the P / S buffers of every rank (P_peers / S_peers: device
// pointers valid on THIS device, e.g. torch symmetric memory; P: nobs*32*MC elements of T with MC = 4 up to 128
// members, 8 above; S: nobs*2 doubles).  Preconditions: all buffers filled with 0xFF bytes and the group synchronised
// after that; every rank calls this with the same inputs.  Outputs (Ym, Yp, rec, counters[0]) are written for the
// rank's own rows only: the caller zeroes the others and sums over the group.
template <typename T>
static int dg_solve_dist(void *plan, T *Ym, T *Yp, const double *ob_value, const double *ob_error, const uint8_t *ob_assim,
                         const double *ob_thr, const double *geo, int64_t nobs, int nens, int loc_mode, double *rec,
                         unsigned long long *counters, int rank, int world, void *const *P_peers, void *const *S_peers, cudaStream_t st) {
    EXB_REQUIRE(plan && Ym && Yp && ob_value && ob_error && ob_assim && geo && rec && P_peers && S_peers, "null pointer");
    EXB_REQUIRE(world >= 1 && world <= 8 && rank >= 0 && rank < world, "bad rank / world");
    ExbObsPlan *pl = static_cast<ExbObsPlan *>(plan);
    if (pl->nobs != nobs || pl->loc_mode != loc_mode || pl->deal.world != world || pl->deal.rank != rank) {
        exb_set_error("exb_obs_solve_dist: the plan was built for another observation set, rank or group size");
        return EXB_ERR_ARG;
    }
    const int rcf = dg_plan_finish(pl);
    if (rcf != EXB_OK) return rcf;
    if (pl->dense || (!pl->list && pl->off_h.back() > 0)) return EXB_ERR_UNSUPPORTED;
    EXB_CUDA(cudaStreamWaitEvent(st, pl->ready, 0));
    DgArgs<T> a;
    {
        int *sh = nullptr, *sd = nullptr;
        const int rcs = exb_status_slot_next(&sh, &sd);
        if (rcs != EXB_OK) return rcs;
        EXB_CUDA(cudaMemsetAsync(sd, 0, sizeof(int), st));      // stream-ordered: an earlier solve's verdict is its own
        a.status = sd;
        a.watchdog_ns = dg_watchdog_ns(nobs);
    }
    a.Ym = Ym; a.Yp = Yp; a.ob_value = ob_value; a.ob_error = ob_error; a.ob_assim = ob_assim; a.ob_thr = ob_thr;
    a.geo = geo; a.rec = rec;
    a.counters = counters; a.off = pl->off; a.list = nullptr; a.list_base = 0; a.P = nullptr; a.S = nullptr;
    a.ticket = nullptr; a.nobs = nobs; a.row_begin = 0; a.row_end = nobs; a.nens = nens;
    a.loc_mode = loc_mode; a.inv_n = 1.0 / (double)nens;
    a.world = world; a.rank = rank; a.deal = pl->deal;
    for (int q = 0; q < 8; ++q) { a.P_peer[q] = q < world ? P_peers[q] : nullptr; a.S_peer[q] = q < world ? S_peers[q] : nullptr; }
    const int rc = dg_dispatch<T, true>(a, *pl, st);
    cudaEventRecord(pl->used, st);
    pl->was_used = true;
    return rc;
}

extern "C" int exb_obs_solve_dist_f64(void *plan, double *Ym, double *Yp, const double *ob_value, const double *ob_error,
                                      const uint8_t *ob_assim, const double *obgeo, int64_t nobs, int nens, int loc_mode,
                                      double *rec, unsigned long long *counters, int rank, int world, void *const *P_peers,
                                      void *const *S_peers, void *stream) {
    return dg_solve_dist<double>(plan, Ym, Yp, ob_value, ob_error, ob_assim, nullptr, obgeo, nobs, nens, loc_mode, rec, counters,
                                 rank, world, P_peers, S_peers, (cudaStream_t)stream);
}
extern "C" int exb_obs_solve_dist_f32(void *plan, float *Ym, float *Yp, const double *ob_value, const double *ob_error,
                                      const uint8_t *ob_assim, const double *obgeo, int64_t nobs, int nens, int loc_mode,
                                      double *rec, unsigned long long *counters, int rank, int world, void *const *P_peers,
                                      void *const *S_peers, void *stream) {
    return dg_solve_dist<float>(plan, Ym, Yp, ob_value, ob_error, ob_assim, nullptr, obgeo, nobs, nens, loc_mode, rec, counters,
                                rank, world, P_peers, S_peers, (cudaStream_t)stream);
}
extern "C" int exb_obs_solve_dist_qc_f64(void *plan, double *Ym, double *Yp, const double *ob_value, const double *ob_error,
                                         const uint8_t *ob_assim, const double *ob_threshold, const double *obgeo, int64_t nobs,
                                         int nens, int loc_mode, double *rec, unsigned long long *counters, int rank, int world,
                                         void *const *P_peers, void *const *S_peers, void *stream) {
    return dg_solve_dist<double>(plan, Ym, Yp, ob_value, ob_error, ob_assim, ob_threshold, obgeo, nobs, nens, loc_mode, rec,
                                 counters, rank, world, P_peers, S_peers, (cudaStream_t)stream);
}
extern "C" int exb_obs_solve_dist_qc_f32(void *plan, float *Ym, float *Yp, const double *ob_value, const double *ob_error,
                                         const uint8_t *ob_assim, const double *ob_threshold, const double *obgeo, int64_t nobs,
                                         int nens, int loc_mode, double *rec, unsigned long long *counters, int rank, int world,
                                         void *const *P_peers, void *const *S_peers, void *stream) {
    return dg_solve_dist<float>(plan, Ym, Yp, ob_value, ob_error, ob_assim, ob_threshold, obgeo, nobs, nens, loc_mode, rec,
                                counters, rank, world, P_peers, S_peers, (cudaStream_t)stream);
}

extern "C" int exb_obs_plan_create(const double *obgeo, const uint8_t *ob_assim, int64_t nobs, int loc_mode, void *stream,
                                   void **plan) {
    EXB_REQUIRE(obgeo && ob_assim && plan && nobs > 0, "null pointer or nobs <= 0");
    ExbObsPlan *pl = nullptr;
    const int rc = dg_plan_begin(obgeo, ob_assim, nobs, loc_mode, (cudaStream_t)stream, &pl);
    *plan = pl;
    return rc;
}

// Plan of this rank's rows only (blocks of `block` consecutive obs dealt round-robin to the ranks), for
// exb_obs_solve_dist_*.
extern "C" int exb_obs_plan_create_dist(const double *obgeo, const uint8_t *ob_assim, int64_t nobs, int loc_mode, int rank,
                                        int world, int block, void *stream, void **plan) {
    EXB_REQUIRE(obgeo && ob_assim && plan && nobs > 0, "null pointer or nobs <= 0");
    EXB_REQUIRE(world >= 1 && world <= 8 && rank >= 0 && rank < world && block >= 1, "bad rank / world / block");
    ExbObsPlan *pl = nullptr;
    const int rc = dg_plan_begin(obgeo, ob_assim, nobs, loc_mode, (cudaStream_t)stream, &pl, DgDeal{block, world, rank});
    *plan = pl;
    return rc;
}

extern "C" int exb_obs_plan_finish(void *plan) {
    EXB_REQUIRE(plan, "null plan");
    return dg_plan_finish(static_cast<ExbObsPlan *>(plan));
}

extern "C" int exb_obs_plan_destroy(void *plan) {
    dg_plan_free(static_cast<ExbObsPlan *>(plan));
    return EXB_OK;
}

template int exb_obs_solve_dag<double>(double *, double *, const double *, const double *, const uint8_t *, const double *,
                                       const double *, int64_t, int, int, double *, unsigned long long *, cudaStream_t, bool,
                                       void *);
template int exb_obs_solve_dag<float>(float *, float *, const double *, const double *, const uint8_t *, const double *,
                                      const double *, int64_t, int, int, double *, unsigned long long *, cudaStream_t, bool,
                                      void *);
