// Smoothing and percentile thresholds of the anomaly scores (SURVEY.md §8 f-1).
//
//   gb200_smooth   : pandas `rolling(w).median()` / `rolling(w).mean()` / `ewm(span=w).mean()` of every
//                    column of a row-major [rows, C] matrix, restarted at each job's first row
//                    (diff.py:302-308; the smooth-* columns of .anomaly(), diff.py:387-415).
//   gb200_quantile : pandas `DataFrame.quantile(q)` (linear interpolation, NaN skipped) per column
//                    over each job's rows (diff.py:631-635: the KFCV thresholds).
//
// Smoothing: one thread owns (column, run of S consecutive output rows) and slides its window over
// the run after warming up on the w-1 rows in front of it; threads of a warp sit on adjacent columns,
// so a row step of a warp is one contiguous read and one contiguous write.  The moving median keeps
// the window as a ring of integer keys in shared memory and tracks the rank-k element with one uniform
// pass per output (smm_rank_kernel).  Mean / EWMA (smooth_kernel) carry their state in float64 registers,
// in the recurrences pandas uses.  NaN and +-inf are missing values for all three, as pandas'
// `_prep_values` makes them.
// Quantile: coalesced whole-row reads, 4 x 8-bit radix select passes over global histograms (further down).
#include "common.cuh"
#include <math.h>
#include <stdlib.h>

namespace {

struct SmoothArgs {
    const int64_t* lo; const int64_t* hi;
    const float* v; float* out;
    int C, window, method;
    int S;              // output rows per thread
    int halo;           // rows of warm-up in front of a run (window-1, or the EWMA truncation length)
    double alpha;       // EWMA: 2 / (span + 1)
};

__global__ void smooth_kernel(const __grid_constant__ SmoothArgs a) {
    const int nt = blockDim.x, tid = threadIdx.x;
    const int job = blockIdx.y;
    const int c0 = blockIdx.z * nt;
    const int Cc = min(a.C - c0, nt);
    const int nsub = nt / Cc;
    const int sub = tid / Cc, col = c0 + tid - sub * Cc;
    if (sub >= nsub) return;
    const int64_t j0 = a.lo[job], j1 = a.hi[job];
    const int64_t o0 = j0 + ((int64_t)blockIdx.x * nsub + sub) * a.S;
    const int64_t o1 = min(o0 + (int64_t)a.S, j1);
    if (o0 >= o1) return;
    const int64_t h0 = max(j0, o0 - (int64_t)a.halo);
    const int C = a.C, w = a.window;
    const float* v = a.v + col;
    float* out = a.out + col;

    // Both loops are latency-bound: they load the next row's values one step ahead (the store to `out` may alias `v`,
    // so the compiler moves no load above it) and stay rolled, which keeps the kernel at 48 registers, 5 CTAs per SM.
    if (a.method == GB200_SMOOTH_SMA) {
        double sum = 0.0; int nobs = 0;
        const double inv_w = 1.0 / (double)w;
        float nx = v[h0 * C], ox = NAN;                  // the row entering / leaving the window (NaN: none leaves)
        #pragma unroll 1
        for (int64_t r = h0; r < o1; ++r) {
            const float x_new = nx, x_old = ox;
            if (r + 1 < o1) { nx = v[(r + 1) * C]; ox = (r + 1 - w >= h0) ? v[(r + 1 - w) * C] : NAN; }
            if (fabsf(x_new) < INFINITY) { sum += (double)x_new; ++nobs; }
            if (fabsf(x_old) < INFINITY) { sum -= (double)x_old; --nobs; }
            if (r >= o0) out[r * C] = nobs == w ? (float)(sum * inv_w) : NAN;
        }
    } else {
        // pandas ewm(span=w, adjust=True, ignore_na=False).mean(): avg <- (old_wt*avg + x)/(old_wt + 1)
        // with old_wt decayed by (1 - alpha) at every row; the history before h0 carries a relative
        // weight below 2^-64 and is dropped
        // ... counted from the LAST OBSERVED row in front of the run: missing rows carry the average forward unchanged,
        // so behind a gap longer than the halo the state is whatever the rows before the gap left
        const double decay = 1.0 - a.alpha;
        double avg = NAN, old_wt = 1.0;
        int64_t last = o0 - 1;
        while (last >= j0 && !(fabsf(v[last * C]) < INFINITY)) --last;
        const int64_t e0 = last < j0 ? o0 : max(j0, last - (int64_t)a.halo);
        float nx = v[e0 * C];
        #pragma unroll 1
        for (int64_t r = e0; r < o1; ++r) {
            const float x = nx;
            if (r + 1 < o1) nx = v[(r + 1) * C];
            const bool obs = fabsf(x) < INFINITY;
            if (r > e0) {
                if (avg == avg) {
                    old_wt *= decay;
                    if (obs) {
                        if (avg != (double)x) avg = (old_wt * avg + (double)x) / (old_wt + 1.0);
                        old_wt += 1.0;
                    }
                } else if (obs) avg = (double)x;
            } else if (obs) avg = (double)x;
            if (r >= o0) out[r * C] = (float)avg;
        }
    }
}

// ---------------------------------------------------------------- order-preserving keys of floats
__device__ __forceinline__ uint32_t f2key(float x) {
    const uint32_t u = __float_as_uint(x);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// ---------------------------------------------------------------- moving median, rank-tracking version
// A sorted window per thread (round 1's kernel) pays two binary searches (dependent shared-memory loads) and a shift
// whose length differs per lane -- a warp waits for its slowest lane, ~0.85 w moves on white noise -- per output: 87 ms
// for the c2-sized matrix at w = 144.  This version keeps the window as an UNSORTED ring of order-preserving integer
// keys and tracks the median itself: when one value leaves and one enters, every rank moves by at most one, so with
// r = the previous element of rank k (k = w / 2)
//      new rank-k element   is one of { pred(r), r, succ(r) },
//      new rank-(k-1) one   is one of { second largest below r, pred(r), r }            (even windows only),
// decided by cL = #{x < r} and E = #{x == r}.  One pass over the ring per output -- the same trip count in every lane,
// 128-bit conflict-free loads, no dependent addressing -- yields pred / second pred / succ and E:
//      u = key - r (mod 2^32): the keys below r are exactly the ones with u >= 2^32 - r, in key order, so max u = pred
//      v = r - key (mod 2^32): the keys above r are exactly the ones with v >  r, reversed,            so max v = succ
//      E = w - sum min(u, 1)
// cL needs no pass: it is kept up to date from the two values that moved; after r moves DOWN the count below the new r
// is unknown (its multiplicity is) but the count above is exact (w - old cL), and the other way round after a move UP,
// so whichever count is known is carried and the other one follows from E after the next pass.  Ties, signed zeros
// and +-inf (pandas turns them into missing values before any rolling function, window/rolling.py `_prep_values`)
// therefore cost nothing extra.  A window that held a missing value is re-selected from scratch when the last one
// leaves (<= k + 1 passes walking up from below the minimum).
constexpr uint32_t SMM_MISSING = 0xffffffffu;        // the key of a negative-NaN bit pattern: no stored value has it

template <bool EVEN>
struct RingScan {
    uint32_t p1 = 0, p2 = 0, s1 = 0, z = 0;
    __device__ __forceinline__ void add(uint32_t key, uint32_t r) {
        const uint32_t u = key - r, v = r - key;
        if (EVEN) p2 = max(p2, min(p1, u));
        p1 = max(p1, u);
        s1 = max(s1, v);
        // min through asm: left to itself the compiler turns `z += min(u, 1)` into a compare, an add and a predicated
        // move instead of one VIMNMX and a share of an IADD3.  (The loop is bound by the ALU pipe -- 5 min/max/add3 per
        // key for even windows, 3.5 for odd ones, 80 % busy in profiles/r2h -- but counting through the multiplier,
        // #{u != 0} = sum(u) - sum(hi32(u * (2^32 - 1))), was slower: IMAD.HI costs more than the VIMNMX it frees.)
        uint32_t nz;
        asm("min.u32 %0, %1, 1;" : "=r"(nz) : "r"(u));
        z += nz;
    }
    // ring: this thread's first quad; quads are nt apart
    __device__ __forceinline__ void run(const uint4* ring, int nt, int w, uint32_t r) {
        const int nq = w >> 2;
        #pragma unroll 2
        for (int q = 0; q < nq; ++q) {
            const uint4 k4 = ring[(size_t)q * nt];
            add(k4.x, r); add(k4.y, r); add(k4.z, r); add(k4.w, r);
        }
        const int rem = w & 3;
        if (rem) {
            const uint4 k4 = ring[(size_t)nq * nt];
            add(k4.x, r);
            if (rem > 1) add(k4.y, r);
            if (rem > 2) add(k4.z, r);
        }
    }
};

template <bool EVEN>
__global__ void __launch_bounds__(384, 1) smm_rank_kernel(const __grid_constant__ SmoothArgs a) {
    extern __shared__ uint4 s_ring[];                      // [ceil(w / 4)][threads] quads of keys
    const int nt = blockDim.x, tid = threadIdx.x;
    const int job = blockIdx.y;
    const int c0 = blockIdx.z * nt;
    const int Cc = min(a.C - c0, nt);
    const int nsub = nt / Cc;
    const int sub = tid / Cc, col = c0 + tid - sub * Cc;
    if (sub >= nsub) return;
    const int64_t j0 = a.lo[job], j1 = a.hi[job];
    const int64_t o0 = j0 + ((int64_t)blockIdx.x * nsub + sub) * a.S;
    const int64_t o1 = min(o0 + (int64_t)a.S, j1);
    if (o0 >= o1) return;
    const int64_t h0 = max(j0, o0 - (int64_t)a.halo);
    const int C = a.C, w = a.window, k = w >> 1;
    const float* v = a.v + col;
    float* out = a.out + col;
    const uint4* ring = s_ring + tid;
    uint32_t* words = reinterpret_cast<uint32_t*>(s_ring + tid);            // word (i) at words[(i >> 2) * nt * 4 + (i & 3)]

    int pos = 0, n_in = 0, n_missing = 0;
    bool valid = false, known_lo = true;
    uint32_t r = 0;                 // key of the current rank-k element
    int cL = 0, cG = 0;             // #{key < r}, #{key > r}: the one `known_lo` names is exact between passes
    float nx = v[h0 * C];
    for (int64_t row = h0; row < o1; ++row) {
        const float x = nx;
        if (row + 1 < o1) nx = v[(row + 1) * C];
        const bool present = fabsf(x) < INFINITY;          // false for NaN and +-inf
        const uint32_t kn = present ? f2key(x) : SMM_MISSING;
        uint32_t* slot = words + (size_t)(pos >> 2) * nt * 4 + (pos & 3);
        const uint32_t ko = *slot;
        *slot = kn;
        pos = pos + 1 == w ? 0 : pos + 1;
        if (n_in == w) n_missing -= (ko == SMM_MISSING); else ++n_in;
        n_missing += !present;
        float m = NAN;
        if (n_in == w) {
            if (n_missing == 0) {
                RingScan<EVEN> sc;
                int E;
                uint32_t hi, lo;
                if (!valid) {
                    r = 0; cL = 0;
                    for (;;) {
                        sc = RingScan<EVEN>();
                        sc.run(ring, nt, w, r);
                        E = w - (int)sc.z;
                        if (cL + E > k) break;
                        cL += E; r -= sc.s1;
                    }
                    cG = w - cL - E;
                    hi = r; lo = cL <= k - 1 ? r : r + sc.p1;
                    valid = true; known_lo = true;
                } else {
                    if (known_lo) cL += (int)(kn < r) - (int)(ko < r);
                    else          cG += (int)(kn > r) - (int)(ko > r);
                    sc.run(ring, nt, w, r);
                    E = w - (int)sc.z;
                    if (known_lo) cG = w - cL - E; else cL = w - cG - E;
                    if (cL > k) {                               // rank k slid below r
                        hi = r + sc.p1; lo = r + sc.p2;
                        cG = w - cL; known_lo = false; r = hi;
                    } else if (cL + E <= k) {                   // ... above r
                        hi = r - sc.s1; lo = E > 0 ? r : r + sc.p1;
                        cL += E; known_lo = true; r = hi;
                    } else {
                        hi = r; lo = cL <= k - 1 ? r : r + sc.p1;
                        known_lo = true;
                    }
                }
                m = EVEN ? (float)(0.5 * ((double)key2f(lo) + (double)key2f(hi))) : key2f(hi);
            } else {
                valid = false;
            }
        }
        if (row >= o0) out[row * C] = m;
    }
}

int max_rows_host(int n_jobs, const int64_t* lo, const int64_t* hi, cudaStream_t stream, int64_t* out) {
    int64_t* h = (int64_t*)malloc(sizeof(int64_t) * 2 * n_jobs);
    if (!h) { gb_set_error("out of host memory"); return GB_ERR_ARG; }
    cudaError_t e = cudaMemcpyAsync(h, lo, sizeof(int64_t) * n_jobs, cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(h + n_jobs, hi, sizeof(int64_t) * n_jobs, cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) { free(h); gb_set_error("row range copy: %s", cudaGetErrorString(e)); return GB_ERR_CUDA; }
    int64_t mx = 0;
    for (int i = 0; i < n_jobs; ++i) { const int64_t n = h[n_jobs + i] - h[i]; if (n > mx) mx = n; }
    free(h);
    *out = mx;
    return GB_OK;
}

}  // namespace

int gb_launch_smooth(int n_jobs, const int64_t* lo, const int64_t* hi, const float* v, int n_cols,
                     int method, int window, float* out, cudaStream_t stream) {
    if (n_jobs <= 0) return GB_OK;
    GB_REQUIRE(window >= 1, "smooth: window must be >= 1");
    GB_REQUIRE(method == GB200_SMOOTH_SMM || method == GB200_SMOOTH_SMA || method == GB200_SMOOTH_EWMA,
               "smooth: method must be GB200_SMOOTH_SMM / _SMA / _EWMA");
    int64_t max_rows = 0;
    int rc = max_rows_host(n_jobs, lo, hi, stream, &max_rows);
    if (rc) return rc;
    if (max_rows == 0) return GB_OK;
    SmoothArgs a{};
    a.lo = lo; a.hi = hi; a.v = v; a.out = out; a.C = n_cols; a.window = window; a.method = method;
    int nt = 256;
    size_t smem = 0;                // moving median only
    const bool smm = method == GB200_SMOOTH_SMM;
    if (smm) {
        // ring of ceil(w / 4) key quads per thread; as many threads as the shared memory of one SM holds
        const size_t per_thread = (size_t)((window + 3) / 4) * sizeof(uint4);
        nt = 384;
        while (nt > 32 && (size_t)nt * per_thread > GB_SMEM_OPTIN_MAX) nt -= 32;
        GB_REQUIRE((size_t)nt * per_thread <= GB_SMEM_OPTIN_MAX, "smooth: moving-median window %d too long (max %d)",
                   window, (int)(GB_SMEM_OPTIN_MAX / (32 * sizeof(uint4)) * 4));
        smem = (size_t)nt * per_thread;
        a.halo = window - 1;
    } else if (method == GB200_SMOOTH_SMA) {
        a.halo = window - 1;
    } else {
        a.alpha = 2.0 / ((double)window + 1.0);
        // (1 - alpha)^halo < 2^-64
        const double need = ceil(64.0 * log(2.0) / -log1p(-a.alpha));
        a.halo = need > 1e9 ? 1000000000 : (int)need;
    }
    // rows per thread: long enough to amortise the warm-up (and, for the rank-tracking median, the selection from
    // scratch at the first full window: up to w / 2 + 1 passes), short enough to fill the GPU
    int S = a.halo > 512 ? a.halo : 512;
    const int Cc = n_cols < nt ? n_cols : nt;
    const int nsub = nt / Cc;
    if (smm) {
        // one CTA per SM and a per-run overhead of halo + ~w/2 selection passes: pick the number of CTAs per job
        // (j = 1, 2, ...; S = the rows that leaves per thread) that minimises waves x (S + overhead).  With S fixed
        // at 2048 the c2-sized matrix made 896 CTAs = 6.05 waves of 148.
        const int64_t zb = (n_cols + nt - 1) / nt, overhead = a.halo + window / 2 + 1;
        int64_t best = -1;
        for (int64_t j = 1; j <= 4096; ++j) {
            const int64_t Sj = (max_rows + nsub * j - 1) / (nsub * j);
            const int64_t waves = (n_jobs * j * zb + 147) / 148;
            const int64_t cost = waves * (Sj + overhead);
            if (best < 0 || cost < best) { best = cost; S = (int)Sj; }
            if (Sj <= 32) break;
        }
    } else {
        while (S > 64 && S / 2 >= a.halo && ((max_rows + S - 1) / S) * (int64_t)n_jobs * n_cols < 148LL * 2048) S >>= 1;
    }
    a.S = S;
    const int64_t rows_per_block = (int64_t)nsub * S;
    dim3 grid((unsigned)((max_rows + rows_per_block - 1) / rows_per_block), n_jobs, (n_cols + nt - 1) / nt);
    if (smm) {
        auto launch = [&](auto kern) -> int {
            if (smem > 48 * 1024) GB_CUDA_CHECK(gb_allow_max_smem(kern));
            kern<<<grid, nt, smem, stream>>>(a);
            GB_CUDA_CHECK(cudaGetLastError());
            return GB_OK;
        };
        return (window & 1) ? launch(smm_rank_kernel<false>) : launch(smm_rank_kernel<true>);
    }
    smooth_kernel<<<grid, nt, 0, stream>>>(a);
    GB_CUDA_CHECK(cudaGetLastError());
    return GB_OK;
}


namespace {
// ---------------------------------------------------------------- quantile, coalesced multi-CTA version
// A CTA per (job, 8 columns) (round 1's kernel) walks its columns with a 200-byte stride: every warp load touches 32
// sectors, and the load unit's wavefronts -- not the histogram atomics -- bound it (32 ms for the 2.56 GB c2-sized
// matrix, unchanged when MATCH.ANY was removed).  Here a CTA reads whole rows: thread = (row lane, column) with the
// column FIXED per thread, so a warp's 32 lanes are 32 adjacent floats of the row-major matrix (fully coalesced), a
// job's rows are split over several CTAs, and the radix select runs as 4 passes of 8 bits:
//   q_hist   : shared-memory histograms [column][256 (+1 pad: adjacent columns, same bin -> different banks)] of the keys
//              that still match the column's prefix, flushed into a global [job][column][256] histogram;
//   q_select : one warp per (job, column) finds the bin holding the wanted rank, extends the prefix, clears the bins;
//   q_next   : count of values <= the selected one and the smallest value above it (per-thread registers: the column is fixed);
//   q_finish : pandas' linear interpolation in float64.
// No host synchronisation; the workspace comes from the stream-ordered allocator.
struct QState { uint32_t prefix, mask, mingt, pad; long long rank, n; unsigned long long le; };
constexpr int QH_THREADS = 1024;
constexpr int QH_MAXC = 64;                       // columns per CTA: 64 x 257 x 4 B = 66 KB of histograms

__global__ void q_init_kernel(QState* st, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { st[i].prefix = 0; st[i].mask = 0; st[i].mingt = 0xffffffffu; st[i].pad = 0; st[i].rank = 0; st[i].n = 0; st[i].le = 0; }
}

// MODE 0: histogram pass (shift = bit position of the 8-bit digit); MODE 1: the next-order-statistic pass
template <int MODE>
__global__ void __launch_bounds__(QH_THREADS)
q_scan_kernel(const int64_t* __restrict__ lo, const int64_t* __restrict__ hi, const float* __restrict__ v, int C,
              int shift, QState* __restrict__ st, unsigned int* __restrict__ ghist) {
    extern __shared__ unsigned int sh[];              // MODE 0: [Cc][257]
    const int job = blockIdx.y, c0 = blockIdx.z * QH_MAXC;
    const int Cc = min(QH_MAXC, C - c0);
    const int lanes_r = QH_THREADS / Cc;              // row lanes; threads beyond lanes_r * Cc idle
    const int tid = threadIdx.x;
    const int col = tid % Cc, rl = tid / Cc;
    const int64_t j0 = lo[job], n_rows = hi[job] - j0;
    const int64_t chunk = (n_rows + gridDim.x - 1) / gridDim.x;
    const int64_t r0 = (int64_t)blockIdx.x * chunk, r1 = min(n_rows, r0 + chunk);
    if (MODE == 0) {
        for (int i = tid; i < Cc * 257; i += QH_THREADS) sh[i] = 0;
        __syncthreads();
    }
    if (rl < lanes_r && r0 < r1) {
        const QState s = st[(size_t)job * C + c0 + col];
        const float* p = v + (j0 + r0 + rl) * C + c0 + col;
        const size_t step = (size_t)lanes_r * C;
        if (MODE == 0) {
            unsigned int* h = sh + col * 257;
            for (int64_t r = r0 + rl; r < r1; r += lanes_r, p += step) {
                const float x = *p;
                if (x == x) {
                    const uint32_t k = f2key(x);
                    if ((k & s.mask) == s.prefix) atomicAdd(&h[(k >> shift) & 255u], 1u);
                }
            }
        } else {
            unsigned long long le = 0; uint32_t mg = 0xffffffffu;
            for (int64_t r = r0 + rl; r < r1; r += lanes_r, p += step) {
                const float x = *p;
                if (x == x) {
                    const uint32_t k = f2key(x);
                    if (k <= s.prefix) ++le; else mg = min(mg, k);
                }
            }
            QState* d = st + (size_t)job * C + c0 + col;
            if (le) atomicAdd(&d->le, le);
            if (mg != 0xffffffffu) atomicMin(&d->mingt, mg);
        }
    }
    if (MODE == 0) {
        __syncthreads();
        unsigned int* g = ghist + ((size_t)job * C + c0) * 256;
        for (int i = tid; i < Cc * 256; i += QH_THREADS) {
            const unsigned int c = sh[(i >> 8) * 257 + (i & 255)];
            if (c) atomicAdd(&g[i], c);
        }
    }
}

// one warp per (job, column): locate the bin of the wanted rank, extend the prefix, clear the histogram
__global__ void q_select_kernel(int n_items, int pass, int shift, double q, QState* __restrict__ st,
                                unsigned int* __restrict__ ghist) {
    const int item = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (item >= n_items) return;
    unsigned int* h = ghist + (size_t)item * 256 + lane * 8;
    unsigned int cnt[8]; long long local = 0;
    #pragma unroll
    for (int i = 0; i < 8; ++i) { cnt[i] = h[i]; local += cnt[i]; h[i] = 0; }
    long long incl = local;
    for (int o = 1; o < 32; o <<= 1) { const long long t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
    const long long total = __shfl_sync(0xffffffffu, incl, 31);
    QState* s = st + item;
    long long rank = s->rank;
    if (pass == 0) { rank = total > 0 ? (long long)floor((double)(total - 1) * q) : 0; }
    const long long before = incl - local;
    __syncwarp();
    if (total > 0 && rank >= before && rank < before + local) {
        long long acc = before; int b = 0;
        for (;; ++b) { if (rank < acc + cnt[b]) break; acc += cnt[b]; }
        s->prefix |= (uint32_t)(lane * 8 + b) << shift;
        s->rank = rank - acc;
    }
    if (lane == 0) { s->mask |= 0xffu << shift; if (pass == 0) s->n = total; }
}

__global__ void q_finish_kernel(int n_items, double q, const QState* __restrict__ st, double* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_items) return;
    const QState s = st[i];
    double res = NAN;
    if (s.n > 0) {
        const double h = (double)(s.n - 1) * q;
        const long long k = (long long)floor(h);
        const double frac = h - (double)k;
        const double va = (double)key2f(s.prefix);
        double vb = va;
        if (frac > 0.0 && k + 1 < s.n && s.le < (unsigned long long)(k + 2)) vb = (double)key2f(s.mingt);
        res = va + (vb - va) * frac;
    }
    out[i] = res;
}
}  // namespace

int gb_launch_quantile(int n_jobs, const int64_t* lo, const int64_t* hi, const float* v, int n_cols,
                       double q, double* out, cudaStream_t stream) {
    if (n_jobs <= 0) return GB_OK;
    GB_REQUIRE(q >= 0.0 && q <= 1.0, "quantile: q must be in [0, 1]");
    const int n_items = n_jobs * n_cols;
    const int colchunks = (n_cols + QH_MAXC - 1) / QH_MAXC;
    // rows of a job are split over gx CTAs so that the launch has a few CTAs per SM without knowing the row counts
    int gx = (4 * 148 + n_jobs * colchunks - 1) / (n_jobs * colchunks);
    if (gx < 1) gx = 1; if (gx > 128) gx = 128;
    QState* st = nullptr; unsigned int* ghist = nullptr;
    GB_CUDA_CHECK(cudaMallocAsync(&st, sizeof(QState) * (size_t)n_items, stream));
    GB_CUDA_CHECK(cudaMallocAsync(&ghist, sizeof(unsigned int) * 256 * (size_t)n_items, stream));
    cudaError_t err = cudaMemsetAsync(ghist, 0, sizeof(unsigned int) * 256 * (size_t)n_items, stream);
    q_init_kernel<<<(n_items + 255) / 256, 256, 0, stream>>>(st, n_items);
    const size_t smem = (size_t)QH_MAXC * 257 * sizeof(unsigned int);
    if (err == cudaSuccess) err = cudaFuncSetAttribute(q_scan_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const dim3 grid(gx, n_jobs, colchunks);
    for (int pass = 0; pass < 4 && err == cudaSuccess; ++pass) {
        const int shift = 24 - 8 * pass;
        q_scan_kernel<0><<<grid, QH_THREADS, smem, stream>>>(lo, hi, v, n_cols, shift, st, ghist);
        q_select_kernel<<<(n_items * 32 + 255) / 256, 256, 0, stream>>>(n_items, pass, shift, q, st, ghist);
    }
    q_scan_kernel<1><<<grid, QH_THREADS, 0, stream>>>(lo, hi, v, n_cols, 0, st, ghist);
    q_finish_kernel<<<(n_items + 255) / 256, 256, 0, stream>>>(n_items, q, st, out);
    if (err == cudaSuccess) err = cudaGetLastError();
    cudaFreeAsync(st, stream); cudaFreeAsync(ghist, stream);
    GB_CUDA_CHECK(err);
    return GB_OK;
}
