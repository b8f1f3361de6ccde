// rvslice.cu — device-side bookkeeping of the population slice sampler (SURVEY.md 8f row 1: the
// vectorised proposal step on the sampler's side of the likelihood boundary; the reference
// configures UltraNest's slice step sampler at evidence/ultranest/__init__.py:175).
//
// One slice move of k walkers is three launches of this file around two or three launches of the
// likelihood (rvl_transform_loglike_dev), with no host read-back in between:
//
//   slice_begin   direction (whitened random unit vector), initial bracket, and ALL stepping-out
//                 positions of both sides (lo - j, hi + j, j < n_out) as candidate points
//   [likelihood]  u -> theta -> lnL of the k * 2 n_out candidates
//   slice_mid     length of the run of successes on each side -> final bracket; the next m
//                 shrinkage candidates, each drawn as if the ones before it had been rejected
//   [likelihood]  k * m candidates
//   slice_end     first accepted candidate -> new position, theta, lnL; walkers still pending get
//                 their shrunken bracket and m more candidates (then: likelihood, slice_end again)
//
// One warp per walker, lanes over the dimensions (ndim <= 128).  Random numbers: Philox4x32-10
// keyed by the seed, counter = (move, draw, walker, 0) -- every (seed, move, draw, walker) has its
// own stream, reproducible whatever k or the launch geometry.
// Candidates outside the unit cube are clamped before evaluation and flagged, never accepted.
// Circular coordinates (rvl_slice_phase_wrapped, the kWrap = true instantiations) are instead taken
// modulo 1 -- the candidate stores p - floor(p), with 1 -> 0 -- and never flag a candidate: the
// sampler then moves on the torus, whose uniform measure is the same as the cube's.
// An ensemble of independent runs of one model (rvl_slice_phase_runs, the kRuns = true
// instantiations) shares every launch: walker w belongs to run run_of[w], draws as walker
// walker_of[w] of that run's seed and reads that run's constraint and whitening, so a run draws
// what it would draw alone.  rvl_slice_runs_init / _whiten / _starts set up such runs on the device.
// rvl_slice_runs_radius / _travel measure, per run and round, the largest nearest-neighbour gap of
// the survivors and how many walkers moved farther than it, in the whitened metric of the moves:
// the inputs of an adaptive number of moves per run (sampler_dev, adaptive_nsteps='move-distance').
// rvl_region_runs_radius / _draw / _pick fill a round's walkers of each run by MLFriends region sampling
// instead: independent draws from the union of balls around the survivors (sampler_dev, method='mlfriends').
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <string>
#include <type_traits>

#include "../../include/rvlnl.h"

namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kMaxDim = RVL_MAX_DIM;
thread_local std::string g_slice_error;

// ---- Philox4x32-10 (Salmon et al. 2011), counter-based ---------------------------------------
struct U4 {
    uint32_t x, y, z, w;
};
__device__ __forceinline__ U4 philox(U4 c, uint32_t k0, uint32_t k1)
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = U4{hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0};
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return c;
}
// uniform strictly inside (0, 1) from two words: 52 bits, ((v >> 1) + 0.5) 2^-52 is exact and lies
// in [2^-53, 1 - 2^-53] ((2^53 - 1) + 0.5 would round to 2^53, i.e. exactly 1.0)
__device__ __forceinline__ double u01(uint32_t a, uint32_t b)
{
    const uint64_t v = ((uint64_t)a << 21) ^ (uint64_t)(b >> 11);  // 53 bits
    return ((double)(v >> 1) + 0.5) * 0x1p-52;
}

struct SliceArgs {
    int k, d, n_out, m;
    uint64_t seed;
    uint32_t move;          // index of the slice move (RNG counter)
    uint32_t shrink_round;  // index of the shrinkage round inside the move
    const double *lmin;     // device scalar: the likelihood constraint
    const double *chol;     // [d][d] lower triangular, row major
    double *u;              // [k][d] walker positions
    double *theta;          // [k][d]
    double *lcur;           // [k]  lnL of the walker (NaN until it moves)
    double *dirn;           // [k][d]
    double *lo, *hi;        // [k] bracket
    double *lo2, *hi2;      // [k] bracket after rejecting all candidates of the round
    double *tval;           // [k][m] offsets of the shrinkage candidates
    int *pending;           // [k] 1 while the move has not been accepted
    // stepping-out candidates (C = 2 n_out) and shrinkage candidates (C = m): separate buffers, so
    // that each likelihood launch covers exactly the rows of its phase
    double *cand_o;          // [k][2 n_out][d]
    uint8_t *inside_o;       // [k][2 n_out]
    const double *ll_o;      // [k][2 n_out]
    double *cand;            // [k][m][d]
    uint8_t *inside;         // [k][m]
    const double *cand_ll;   // [k][m]   likelihood of the candidates
    const double *cand_th;   // [k][m][d]
    unsigned long long *stats;  // [0] walkers left pending by a slice_end, [1] accepted moves
};
// the arguments of the kWrap = true kernels: the mask by value after the fields of SliceArgs, which
// keep their parameter offsets (and the kWrap = false kernels are exactly the unwrapped ones)
struct SliceArgsWrap : SliceArgs {
    uint32_t wrap[4];  // bit j & 31 of wrap[j >> 5]: coordinate j is circular
};
// the arguments of the kRuns = true kernels: the runs' fields after those of the kRuns = false
// instance (lmin, chol and stats then hold one entry per run: [R], [R][d][d], [R][2])
template <class Base>
struct WithRuns : Base {
    const int32_t *run_of;     // [k] run of walker w
    const int32_t *walker_of;  // [k] index of walker w inside its run
    const uint64_t *seeds;     // [R]
};
template <bool kWrap, bool kRuns = false>
using ArgsT = typename std::conditional<
    kRuns, WithRuns<typename std::conditional<kWrap, SliceArgsWrap, SliceArgs>::type>,
    typename std::conditional<kWrap, SliceArgsWrap, SliceArgs>::type>::type;

constexpr double kHiClamp = 1.0 - 0x1p-53;

// the words of counter (c0, tag, walker, 0) under a seed.  The key is the seed alone and the walker
// is a counter word: Philox is a bijection of the counter under a fixed key, so no two (seed, walker)
// pairs share a stream (a key mixing seed and walker, e.g. seed ^ walker, would repeat across seeds)
__device__ __forceinline__ U4 draw_seed(uint64_t seed, uint32_t c0, uint32_t tag, uint32_t walker)
{
    return philox(U4{c0, tag, walker, 0u}, (uint32_t)seed, (uint32_t)(seed >> 32) + 0x51CEu);
}

// who walker w of a launch is: its run r (0 without runs), its index j inside the run (the walker
// word of its counters) and the run's seed
struct Who {
    int r, j;
    uint64_t seed;
};
template <bool kWrap, bool kRuns>
__device__ __forceinline__ Who who(const ArgsT<kWrap, kRuns> &a, int w)
{
    if constexpr (kRuns) {
        const int r = a.run_of[w];
        return Who{r, a.walker_of[w], a.seeds[r]};
    } else {
        return Who{0, w, a.seed};
    }
}

// the words of draw `tag` of walker w (id) in this move
__device__ __forceinline__ U4 draw(const SliceArgs &a, uint32_t tag, int w)
{
    return draw_seed(a.seed, a.move, tag, (uint32_t)w);
}
template <bool kRuns>
__device__ __forceinline__ U4 draw(const SliceArgs &a, const Who &id, uint32_t tag, int w)
{
    if constexpr (kRuns) return draw_seed(id.seed, a.move, tag, (uint32_t)id.j);
    else return draw(a, tag, w);
}

template <bool kWrap, class A>
__device__ __forceinline__ void write_candidate(const A &a, double *cand, uint8_t *inside,
                                                int w, int slot, int C, double t, const double *ui,
                                                const double *di, int lane)
{
    bool in = true;
    double *dst = cand + ((size_t)w * C + slot) * a.d;
    for (int j = lane; j < a.d; j += 32) {
        const double p = ui[j] + t * di[j];
        if constexpr (kWrap) {
            // constant word indices: the mask stays in the parameter bank (no local copy)
            const uint32_t word = j < 32 ? a.wrap[0] : j < 64 ? a.wrap[1] : j < 96 ? a.wrap[2] : a.wrap[3];
            if ((word >> (j & 31)) & 1u) {
                // floor and the subtraction are exact; q rounds to 1.0 only for p in (-2^-54, 0),
                // where 1 is the same point as 0
                double q = p - floor(p);
                if (q >= 1.0) q = 0.0;
                dst[j] = q;
                continue;
            }
        }
        in = in && (p >= 0.0) && (p < 1.0);
        dst[j] = fmin(fmax(p, 0.0), kHiClamp);
    }
    in = __all_sync(kFull, in);
    if (lane == 0) inside[(size_t)w * C + slot] = in ? 1 : 0;
}

// the next m shrinkage candidates of walker w from bracket (lo, hi): sequential rule, speculated
template <bool kWrap, bool kRuns, class A>
__device__ __forceinline__ void propose_shrink(const A &a, const Who &id, int w, double lo, double hi,
                                               const double *ui, const double *di, int lane)
{
    const int C = a.m;
    for (int j = 0; j < a.m; ++j) {
        const U4 r = draw<kRuns>(a, id, 0x53480000u + a.shrink_round * 64u + (uint32_t)j, w);
        const double t = lo + (hi - lo) * u01(r.x, r.y);
        if (lane == 0) a.tval[(size_t)w * a.m + j] = t;
        write_candidate<kWrap>(a, a.cand, a.inside, w, j, C, t, ui, di, lane);
        if (t < 0.0) lo = t; else hi = t;
    }
    if (lane == 0) { a.lo2[w] = lo; a.hi2[w] = hi; }
}

template <bool kWrap, bool kRuns>
__global__ void __launch_bounds__(128) slice_begin_kernel(const ArgsT<kWrap, kRuns> a)
{
    const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (w >= a.k) return;
    __shared__ double sz[4][kMaxDim];
    double *z = sz[threadIdx.x >> 5];
    const Who id = who<kWrap, kRuns>(a, w);
    const double *chol = a.chol;
    if constexpr (kRuns) chol += (size_t)id.r * a.d * a.d;
    // z ~ N(0, I): Box-Muller on Philox words, two normals per counter
    double n2 = 0.0;
    for (int j = lane; j < a.d; j += 32) {
        const U4 r = draw<kRuns>(a, id, 0x44495200u + (uint32_t)(j >> 1), w);
        const double rad = sqrt(-2.0 * log(u01(r.x, r.y))), ang = 6.283185307179586 * u01(r.z, r.w);
        const double v = (j & 1) ? rad * sin(ang) : rad * cos(ang);
        z[j] = v;
        n2 += v * v;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n2 += __shfl_xor_sync(kFull, n2, o);
    __syncwarp();
    const double inv = 1.0 / sqrt(n2);
    // dirn = chol z / |z|  (the direction is uniform on the whitened unit sphere)
    double *di = a.dirn + (size_t)w * a.d;
    for (int j = lane; j < a.d; j += 32) {
        double acc = 0.0;
        for (int l = 0; l <= j; ++l) acc += chol[(size_t)j * a.d + l] * z[l];
        di[j] = acc * inv;
    }
    __syncwarp();
    const U4 r = draw<kRuns>(a, id, 0x42524B00u, w);
    const double r0 = u01(r.x, r.y);
    const double lo = -r0, hi = 1.0 - r0;
    if (lane == 0) { a.lo[w] = lo; a.hi[w] = hi; a.pending[w] = 1; }
    const int C = 2 * a.n_out;
    const double *ui = a.u + (size_t)w * a.d;
    for (int j = 0; j < a.n_out; ++j) {
        write_candidate<kWrap>(a, a.cand_o, a.inside_o, w, j, C, lo - (double)j, ui, di, lane);
        write_candidate<kWrap>(a, a.cand_o, a.inside_o, w, a.n_out + j, C, hi + (double)j, ui, di, lane);
    }
}

template <bool kWrap, bool kRuns>
__global__ void __launch_bounds__(128) slice_mid_kernel(const ArgsT<kWrap, kRuns> a)
{
    const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (w >= a.k) return;
    const Who id = who<kWrap, kRuns>(a, w);
    const int C = 2 * a.n_out;
    const double lmin = a.lmin[id.r];
    // run of successes from the bracket edge outwards, both sides
    int run_lo = 0, run_hi = 0;
    for (int j = 0; j < a.n_out; ++j) {
        const size_t s = (size_t)w * C + j;
        if (a.inside_o[s] && a.ll_o[s] > lmin && run_lo == j) run_lo = j + 1;
    }
    for (int j = 0; j < a.n_out; ++j) {
        const size_t s = (size_t)w * C + a.n_out + j;
        if (a.inside_o[s] && a.ll_o[s] > lmin && run_hi == j) run_hi = j + 1;
    }
    const double lo = a.lo[w] - (double)run_lo, hi = a.hi[w] + (double)run_hi;
    __syncwarp();
    if (lane == 0) { a.lo[w] = lo; a.hi[w] = hi; }
    propose_shrink<kWrap, kRuns>(a, id, w, lo, hi, a.u + (size_t)w * a.d, a.dirn + (size_t)w * a.d, lane);
}

template <bool kWrap, bool kRuns>
__global__ void __launch_bounds__(128) slice_end_kernel(const ArgsT<kWrap, kRuns> a, int propose_more)
{
    const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (w >= a.k) return;
    const Who id = who<kWrap, kRuns>(a, w);
    unsigned long long *stats = a.stats + 2 * id.r;
    const int C = a.m;
    const double lmin = a.lmin[id.r];
    int pend = a.pending[w];
    double *ui = a.u + (size_t)w * a.d;
    if (pend) {
        int first = -1;
        for (int j = 0; j < a.m && first < 0; ++j) {
            const size_t s = (size_t)w * C + j;
            if (a.inside[s] && a.cand_ll[s] > lmin) first = j;
        }
        if (first >= 0) {
            const size_t s = (size_t)w * C + first;
            // the accepted point is the UNclamped candidate (it was inside the cube: identical);
            // a circular coordinate is the stored value, already taken modulo 1
            for (int j = lane; j < a.d; j += 32) {
                ui[j] = a.cand[s * a.d + j];
                a.theta[(size_t)w * a.d + j] = a.cand_th[s * a.d + j];
            }
            if (lane == 0) { a.lcur[w] = a.cand_ll[s]; a.pending[w] = 0; atomicAdd(stats + 1, 1ull); }
            pend = 0;
        } else if (lane == 0) {
            a.lo[w] = a.lo2[w];
            a.hi[w] = a.hi2[w];
            if (!propose_more) atomicAdd(stats, 1ull);  // bracket not resolved: the walker stays
        }
    }
    __syncwarp();
    if (propose_more) {
        // still pending: m more candidates from the shrunken bracket; done: re-evaluate the current
        // point (keeps the launch shape fixed -- no compaction, no read-back)
        if (pend) propose_shrink<kWrap, kRuns>(a, id, w, a.lo2[w], a.hi2[w], ui, a.dirn + (size_t)w * a.d, lane);
        else
            for (int j = 0; j < a.m; ++j) {
                write_candidate<kWrap>(a, a.cand, a.inside, w, j, C, 0.0, ui, a.dirn + (size_t)w * a.d, lane);
                if (lane == 0) a.inside[(size_t)w * C + j] = 0;
            }
    }
}

// ---- ensemble set-up: initial live points, whitening and walker starts of R runs -------------------
constexpr uint32_t kTagInit = 0x494E0000u;   // + (c >> 1): coordinate c of initial live point p
constexpr uint32_t kTagStart = 0x53540000u;  // the start of walker j in a round

struct LiveArgs {
    int n_runs, nlive, d;
    uint32_t round;
    const uint64_t *seeds;  // [R]
    double *u_live;         // [R][nlive][d]
    const double *th_live;  // [R][nlive][d]
    const double *l_live;   // [R][nlive]
    const int64_t *order;   // [R][nlive] each run's live points by ascending lnL
    const int64_t *kk;      // [R] points retired this round: the survivors are order[r][kk[r]:]
};

__device__ __forceinline__ double wrap_unit(double p)
{
    const double q = p - floor(p);
    return q >= 1.0 ? 0.0 : q;
}

// u_live[r][p][c] = u01 of counter (0, kTagInit + (c >> 1), p, 0) under seeds[r]: words (x, y) for
// even c, (z, w) for odd c
__global__ void __launch_bounds__(256) runs_init_kernel(const LiveArgs a)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)a.n_runs * a.nlive * a.d) return;
    const int c = (int)(i % a.d), p = (int)(i / a.d % a.nlive), r = (int)(i / a.d / a.nlive);
    const U4 q = draw_seed(a.seeds[r], 0u, kTagInit + (uint32_t)(c >> 1), (uint32_t)p);
    a.u_live[i] = (c & 1) ? u01(q.z, q.w) : u01(q.x, q.y);
}

// One block per run: chol[r] = the lower Cholesky factor of 1e-18 I + the covariance of the surviving
// live points u_live[r][order[r][kk[r] + i]], i < n = nlive - kk[r].  A circular coordinate is first
// taken as wrap_unit(u - mu + 1/2), mu its circular mean atan2(sum sin, sum cos) / 2 pi (sums over i,
// each divided by n).  Every sum runs over i in order, so the factor of a run depends on its points
// alone.  Where a pivot is not > 0, the factor is diag(sqrt(max(cov_jj, 1e-30))).  kk[r] = 0: the run
// is skipped.
template <bool kWrap>
__global__ void __launch_bounds__(256) runs_whiten_kernel(const LiveArgs a, double *chol_all, uint32_t w0, uint32_t w1,
                                                          uint32_t w2, uint32_t w3)
{
    const int r = blockIdx.x, d = a.d;
    const int64_t kk = a.kk[r];
    if (kk <= 0) return;  // a run that takes no part in the round keeps its factor
    const int n = a.nlive - (int)kk;
    const int64_t *rows = a.order + (size_t)r * a.nlive + kk;
    const double *u = a.u_live + (size_t)r * a.nlive * d;
    double *L = chol_all + (size_t)r * d * d;
    __shared__ double mu[kMaxDim], mean[kMaxDim], diag[kMaxDim];
    __shared__ int failed;
    auto circular = [&](int c) {
        if constexpr (kWrap) {
            const uint32_t word = c < 32 ? w0 : c < 64 ? w1 : c < 96 ? w2 : w3;
            return ((word >> (c & 31)) & 1u) != 0u;
        } else {
            return false;
        }
    };
    auto value = [&](int64_t row, int c) {
        const double x = u[(size_t)row * d + c];
        return circular(c) ? wrap_unit(x - mu[c] + 0.5) : x;
    };
    if (threadIdx.x == 0) failed = 0;
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
        double m = 0.0;
        if (circular(c)) {
            double ss = 0.0, cs = 0.0;
            for (int i = 0; i < n; ++i) {
                const double ang = 6.283185307179586 * u[(size_t)rows[i] * d + c];
                ss += sin(ang);
                cs += cos(ang);
            }
            m = atan2(ss / n, cs / n) / 6.283185307179586;
        }
        mu[c] = m;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
        double acc = 0.0;
        for (int i = 0; i < n; ++i) acc += value(rows[i], c);
        mean[c] = acc / n;
    }
    __syncthreads();
    // the covariance into the lower triangle of L (upper triangle: 0)
    for (int e = threadIdx.x; e < d * d; e += blockDim.x) {
        const int p = e / d, q = e % d;
        if (q > p) {
            L[e] = 0.0;
            continue;
        }
        double acc = 0.0;
        for (int i = 0; i < n; ++i) acc += (value(rows[i], p) - mean[p]) * (value(rows[i], q) - mean[q]);
        double cv = acc / (n - 1);
        if (p == q) {
            cv += 1e-18;
            diag[p] = cv;
        }
        L[e] = cv;
    }
    __syncthreads();
    // Cholesky, column by column in place: pivot by thread 0, then the column below it
    for (int j = 0; j < d; ++j) {
        if (threadIdx.x == 0) {
            double s = L[(size_t)j * d + j];
            for (int l = 0; l < j; ++l) s -= L[(size_t)j * d + l] * L[(size_t)j * d + l];
            if (s > 0.0) L[(size_t)j * d + j] = sqrt(s);
            else failed = 1;
        }
        __syncthreads();
        if (failed) break;
        const double piv = L[(size_t)j * d + j];
        for (int i = j + 1 + threadIdx.x; i < d; i += blockDim.x) {
            double s = L[(size_t)i * d + j];
            for (int l = 0; l < j; ++l) s -= L[(size_t)i * d + l] * L[(size_t)j * d + l];
            L[(size_t)i * d + j] = s / piv;
        }
        __syncthreads();
    }
    if (failed)
        for (int e = threadIdx.x; e < d * d; e += blockDim.x) {
            const int p = e / d, q = e % d;
            L[e] = p == q ? sqrt(fmax(diag[p], 1e-30)) : 0.0;
        }
}

// One warp per walker w (run r = run_of[w], walker j = walker_of[w] of that run): a start drawn
// uniformly among the run's survivors -- survivor __umulhi(x, n) of counter (round, kTagStart, j, 0)
// under seeds[r], n = nlive - kk[r] -- copied into u[w], theta[w]; lcur[w] = NaN; start[w] = its slot,
// lstart[w] = its lnL
__global__ void __launch_bounds__(128) runs_starts_kernel(const LiveArgs a, int k, const int32_t *run_of,
                                                          const int32_t *walker_of, double *u,
                                                          double *theta, double *lcur, int64_t *start,
                                                          double *lstart)
{
    const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (w >= k) return;
    const int r = run_of[w];
    const int64_t kk = a.kk[r];
    const U4 q = draw_seed(a.seeds[r], a.round, kTagStart, (uint32_t)walker_of[w]);
    const int64_t slot = a.order[(size_t)r * a.nlive + kk + __umulhi(q.x, (uint32_t)(a.nlive - kk))];
    const size_t src = (size_t)r * a.nlive + slot;
    for (int c = lane; c < a.d; c += 32) {
        u[(size_t)w * a.d + c] = a.u_live[src * a.d + c];
        theta[(size_t)w * a.d + c] = a.th_live[src * a.d + c];
    }
    if (lane == 0) {
        lcur[w] = __longlong_as_double(0x7ff8000000000000ll);
        start[w] = slot;
        lstart[w] = a.l_live[src];
    }
}

// ---- adaptive number of moves: the spacing of each run's survivors and how far its walkers went ------
// The distance of two unit-cube points a, b under run r's whitening factor L = chol[r]:
//   D(a, b) = |y|^2,  y = L^-1 delta,  delta = a - b, and delta_c - rint(delta_c) (half to even) in a
//   circular coordinate.
// Every value is formed in a fixed order with one rounding per operation (the library is built with
// -fmad=false and IEEE division), so a host restatement reproduces it bit for bit and a run's values
// depend on its own points alone, whatever the number of runs:
//   Linv = L^-1, lower triangular, by forward substitution column by column (thread c forms column c):
//          Linv_cc = 1 / L_cc;  for i = c + 1 .. d - 1:  s = 0, s = s + L_il Linv_lc for l = c .. i - 1,
//          Linv_ic = -(s / L_ii)
//   y_i  = 0, y_i = y_i + Linv_il delta_l for l = 0 .. i
//   D    = 0, D = D + y_i y_i for i = 0 .. d - 1
// Linv sits in shared memory, packed by rows (row i at i (i + 1) / 2), and each thread keeps its
// delta in a shared column (delta_l at l * blockDim.x + threadIdx.x): d <= 128 doubles do not fit in
// registers.  Minima, maxima and the integer counts are exact, so their order is free.
constexpr int kAdaptThreads = 128;

struct Wrap4 {
    uint32_t w[4];  // bit c & 31 of w[c >> 5]: coordinate c is circular
};

size_t adapt_smem(int d)
{
    return ((size_t)d * (d + 1) / 2 + (size_t)kAdaptThreads * d) * sizeof(double);
}

__device__ __forceinline__ bool circular(const Wrap4 &wr, int c)
{
    const uint32_t word = c < 32 ? wr.w[0] : c < 64 ? wr.w[1] : c < 96 ? wr.w[2] : wr.w[3];
    return ((word >> (c & 31)) & 1u) != 0u;
}

// Linv of the lower factor L [d][d] (row major) into shared memory; ends with a barrier
__device__ void form_linv(const double *L, int d, double *Linv)
{
    for (int c = threadIdx.x; c < d; c += blockDim.x) {
        Linv[c * (c + 1) / 2 + c] = 1.0 / L[(size_t)c * d + c];
        for (int i = c + 1; i < d; ++i) {
            double s = 0.0;
            for (int l = c; l < i; ++l) s = s + L[(size_t)i * d + l] * Linv[l * (l + 1) / 2 + c];
            Linv[i * (i + 1) / 2 + c] = -(s / L[(size_t)i * d + i]);
        }
    }
    __syncthreads();
}

// D(a, b); dl: this thread's delta column (stride blockDim.x)
__device__ __forceinline__ double whitened_dist2(const double *a, const double *b, int d, const double *Linv,
                                                 double *dl, const Wrap4 &wr)
{
    const int T = blockDim.x;
    for (int c = 0; c < d; ++c) {
        double x = a[c] - b[c];
        if (circular(wr, c)) x = x - rint(x);
        dl[c * T] = x;
    }
    double D = 0.0;
    for (int i = 0; i < d; ++i) {
        const double *row = Linv + i * (i + 1) / 2;
        double y = 0.0;
        for (int l = 0; l <= i; ++l) y = y + row[l] * dl[l * T];
        D = D + y * y;
    }
    return D;
}

// One block per run r with kk[r] > 0 (others are skipped: rad2[r] is left as it is): rad2[r] = the
// largest nearest-neighbour distance among the survivors u_live[r][order[r][kk[r] + i]], i < n =
// nlive - kk[r]: max over i of min over j != i of D(u_i, u_j).  Thread t takes i = t, t + T, ..;
// n < 2: 0.
__global__ void __launch_bounds__(kAdaptThreads) runs_radius_kernel(const LiveArgs a, const double *chol_all,
                                                                    const Wrap4 wr, double *rad2)
{
    const int r = blockIdx.x, d = a.d;
    const int64_t kk = a.kk[r];
    if (kk <= 0) return;
    extern __shared__ double smem[];
    __shared__ double wmax[kAdaptThreads / 32];
    double *Linv = smem, *dl = smem + d * (d + 1) / 2 + threadIdx.x;
    form_linv(chol_all + (size_t)r * d * d, d, Linv);
    const int n = a.nlive - (int)kk;
    const int64_t *rows = a.order + (size_t)r * a.nlive + kk;
    const double *u = a.u_live + (size_t)r * a.nlive * d;
    double mx = 0.0;
    for (int i = threadIdx.x; i < n && n > 1; i += blockDim.x) {
        const double *ui = u + (size_t)rows[i] * d;
        double mn = INFINITY;
        for (int j = 0; j < n; ++j)
            if (j != i) mn = fmin(mn, whitened_dist2(ui, u + (size_t)rows[j] * d, d, Linv, dl, wr));
        mx = fmax(mx, mn);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(kFull, mx, o));
    if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x == 0) {
        double m = wmax[0];
        for (int i = 1; i < (int)(blockDim.x >> 5); ++i) m = fmax(m, wmax[i]);
        rad2[r] = m;
    }
}

// One block per run r with kk[r] > 0 (others are skipped: far[r] is left as it is), one thread per
// walker w of the launch with run_of[w] == r: far[r] = the number of those with D(u_end[w], u_start[w])
// > rad2[r], u_end[w] = u[w], u_start[w] = u_live[r][start[w]] (a walker that did not move: D = 0).
__global__ void __launch_bounds__(kAdaptThreads) runs_travel_kernel(const LiveArgs a, int k, const int32_t *run_of,
                                                                    const int64_t *start, const double *u,
                                                                    const double *chol_all, const Wrap4 wr,
                                                                    const double *rad2, int32_t *far)
{
    const int r = blockIdx.x, d = a.d;
    if (a.kk[r] <= 0) return;
    extern __shared__ double smem[];
    __shared__ int count;
    double *Linv = smem, *dl = smem + d * (d + 1) / 2 + threadIdx.x;
    if (threadIdx.x == 0) count = 0;
    form_linv(chol_all + (size_t)r * d * d, d, Linv);
    const double lim = rad2[r];
    for (int w = threadIdx.x; w < k; w += blockDim.x) {
        if (run_of[w] != r) continue;
        const double *b = a.u_live + ((size_t)r * a.nlive + start[w]) * d;
        if (whitened_dist2(u + (size_t)w * d, b, d, Linv, dl, wr) > lim) atomicAdd(&count, 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) far[r] = count;
}

// ---- MLFriends region sampling of an ensemble: independent draws from the constrained prior ------
// The region of run r is the union of the balls D(x, u_i) <= rho2[r] around its survivors u_i
// (order[r][kk[r] + i], i < n), D the distance of whitened_dist2 under chol[r].  Counter layout (the
// c0 word is the round, live->round, as for the starts; every tag below is used by no other kernel):
//   (round, kTagBoot + b, q, 0)                 bootstrap b: survivor indices 4q .. 4q + 3 of the draw
//                                               with replacement, floor(word n / 2^32) of words x, y, z, w
//   (round, kTagRegion + (batch << 8), s, 0)    candidate slot s of a batch: survivor floor(x n / 2^32)
//                                               and v = u01(z, w)
//   (round, kTagRegion + (batch << 8) + 1 + (c >> 1), s, 0)
//                                               its Gaussian coordinate c: Box-Muller of u01(x, y),
//                                               u01(z, w) -- cos for even c, sin for odd c
constexpr uint32_t kTagBoot = 0x42540000u;
constexpr uint32_t kTagRegion = 0x52000000u;
constexpr int kCompactThreads = 256;

// bytes of dynamic shared memory of the radius kernel: Linv and the delta columns, then one flag per
// survivor
size_t boot_smem(int d, int nlive)
{
    return adapt_smem(d) + (size_t)nlive;
}

// the exclusive prefix of flag f among the threads of the block and the block's total (every thread
// of the block calls it; wsum: shared, one int per warp)
__device__ __forceinline__ int block_prefix(bool f, int *wsum, int &total)
{
    const unsigned bal = __ballot_sync(kFull, f);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) wsum[wid] = __popc(bal);
    __syncthreads();
    int pre = __popc(bal & ((1u << lane) - 1u));
    total = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
        if (w < wid) pre += wsum[w];
        total += wsum[w];
    }
    __syncthreads();
    return pre;
}

// rad2[r] = 0 for the runs taking part in the round, before the bootstraps take their maximum
__global__ void region_clear_kernel(const LiveArgs a, double *rad2)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < a.n_runs && a.kk[r] > 0) rad2[r] = 0.0;
}

// One block per (bootstrap b, run r) with kk[r] > 0: the survivors drawn with replacement (n draws)
// are the selected ones; rho2_b = max over the survivors never drawn of min over the selected ones
// of D (0 when every survivor was drawn), merged into rad2[r] by an integer atomicMax of its bits
// (non-negative doubles order as their bit patterns): exact, whatever the order of the blocks.
__global__ void __launch_bounds__(kAdaptThreads) region_radius_kernel(const LiveArgs a, const double *chol_all,
                                                                      const Wrap4 wr, double *rad2)
{
    const int b = blockIdx.x, r = blockIdx.y, d = a.d;
    const int64_t kk = a.kk[r];
    if (kk <= 0) return;
    extern __shared__ double smem[];
    __shared__ double wmax[kAdaptThreads / 32];
    double *Linv = smem, *dl = smem + d * (d + 1) / 2 + threadIdx.x;
    uint8_t *chosen = (uint8_t *)(smem + d * (d + 1) / 2 + kAdaptThreads * d);
    const int n = a.nlive - (int)kk;
    for (int i = threadIdx.x; i < n; i += blockDim.x) chosen[i] = 0;
    form_linv(chol_all + (size_t)r * d * d, d, Linv);  // (ends with a barrier)
    const uint64_t seed = a.seeds[r];
    for (int q = threadIdx.x; 4 * q < n; q += blockDim.x) {
        const U4 w = draw_seed(seed, a.round, kTagBoot + (uint32_t)b, (uint32_t)q);
        const uint32_t words[4] = {w.x, w.y, w.z, w.w};
        for (int t = 0; t < 4 && 4 * q + t < n; ++t) chosen[__umulhi(words[t], (uint32_t)n)] = 1;
    }
    __syncthreads();
    const int64_t *rows = a.order + (size_t)r * a.nlive + kk;
    const double *u = a.u_live + (size_t)r * a.nlive * d;
    double mx = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        if (chosen[i]) continue;
        const double *ui = u + (size_t)rows[i] * d;
        double mn = INFINITY;
        for (int j = 0; j < n; ++j)
            if (chosen[j]) mn = fmin(mn, whitened_dist2(ui, u + (size_t)rows[j] * d, d, Linv, dl, wr));
        mx = fmax(mx, mn);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(kFull, mx, o));
    if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x == 0) {
        double m = wmax[0];
        for (int i = 1; i < (int)(blockDim.x >> 5); ++i) m = fmax(m, wmax[i]);
        atomicMax((unsigned long long *)(rad2 + r), (unsigned long long)__double_as_longlong(m));
    }
}

// Block (x, r), thread t: candidate slot s = x blockDim.x + t < ns of run r (its slots are the rows
// slot_base[r] .. slot_base[r + 1] - 1 of stage / flag).  Survivor i and a point y uniform in the unit
// ball (z / |z| v^(1/d), z Gaussian); delta = (rho v^(1/d) / |z|) L z; rejected where a circular
// |delta_c| > 1/2 (each ball is then its nearest-image ball on the torus); x = u_i + delta, a circular
// coordinate wrapped as the slice candidates are, a non-circular one outside [0, 1) rejected; rejected
// where a survivor j < i has D(x, u_j) <= rho2[r] (x belongs to the first ball that holds it).  flag =
// accepted, count[r] += the run's accepted slots.
__global__ void __launch_bounds__(kAdaptThreads) region_draw_kernel(const LiveArgs a, const double *chol_all,
                                                                    const Wrap4 wr, const double *rad2,
                                                                    uint32_t batch, const int32_t *slot_base,
                                                                    double *stage, uint8_t *flag, int32_t *count)
{
    const int r = blockIdx.y, d = a.d, T = blockDim.x;
    const int64_t kk = a.kk[r];
    const int s0 = slot_base[r], ns = slot_base[r + 1] - s0;
    if (kk <= 0 || (int)(blockIdx.x * blockDim.x) >= ns) return;  // the whole block
    extern __shared__ double smem[];
    double *Linv = smem, *dl = smem + d * (d + 1) / 2 + threadIdx.x;
    const double *L = chol_all + (size_t)r * d * d;
    form_linv(L, d, Linv);
    const int n = a.nlive - (int)kk, s = blockIdx.x * blockDim.x + threadIdx.x;
    bool ok = s < ns;
    if (ok) {
        const int64_t *rows = a.order + (size_t)r * a.nlive + kk;
        const double *u = a.u_live + (size_t)r * a.nlive * d;
        const uint64_t seed = a.seeds[r];
        const uint32_t tag = kTagRegion + (batch << 8);
        const U4 q0 = draw_seed(seed, a.round, tag, (uint32_t)s);
        const int i = (int)__umulhi(q0.x, (uint32_t)n);
        const double v = u01(q0.z, q0.w);
        double n2 = 0.0;
        for (int c = 0; c < d; ++c) {
            const U4 q = draw_seed(seed, a.round, tag + 1u + (uint32_t)(c >> 1), (uint32_t)s);
            const double rad = sqrt(-2.0 * log(u01(q.x, q.y))), ang = 6.283185307179586 * u01(q.z, q.w);
            const double z = (c & 1) ? rad * sin(ang) : rad * cos(ang);
            dl[c * T] = z;
            n2 = n2 + z * z;
        }
        const double scale = sqrt(rad2[r]) * (pow(v, 1.0 / d) / sqrt(n2));
        const double *ui = u + (size_t)rows[i] * d;
        double *x = stage + (size_t)(s0 + s) * d;
        for (int c = 0; c < d && ok; ++c) {
            double acc = 0.0;
            for (int l = 0; l <= c; ++l) acc = acc + L[(size_t)c * d + l] * dl[l * T];
            const double dc = scale * acc, p = ui[c] + dc;
            if (circular(wr, c)) {
                ok = fabs(dc) <= 0.5;
                x[c] = wrap_unit(p);
            } else {
                ok = p >= 0.0 && p < 1.0;
                x[c] = p;
            }
        }
        const double lim = rad2[r];
        for (int j = 0; j < i && ok; ++j)
            if (whitened_dist2(x, u + (size_t)rows[j] * d, d, Linv, dl, wr) <= lim) ok = false;
    }
    if (s < ns) flag[s0 + s] = ok ? 1 : 0;
    const int acc = __syncthreads_count(ok);
    if (threadIdx.x == 0 && acc) atomicAdd(count + r, acc);
}

// One block per run: offs[r] = count[0] + .. + count[r - 1] (offs[R] = the total), and the accepted
// slots of run r, in slot order, copied to the rows offs[r] .. offs[r + 1] - 1 of cand (none for a run
// with kk[r] = 0: the draw kernel left its flags as they were)
__global__ void __launch_bounds__(kCompactThreads) region_compact_kernel(int n_runs, int d, const int64_t *kk,
                                                                         const int32_t *slot_base,
                                                                         const double *stage, const uint8_t *flag,
                                                                         const int32_t *count, int32_t *offs,
                                                                         double *cand)
{
    const int r = blockIdx.x;
    __shared__ int wsum[kCompactThreads / 32];
    int base = 0;
    for (int q = 0; q < r; ++q) base += count[q];
    if (threadIdx.x == 0) {
        offs[r] = base;
        if (r == n_runs - 1) offs[n_runs] = base + count[r];
    }
    if (kk[r] <= 0) return;
    const int s0 = slot_base[r], ns = slot_base[r + 1] - s0;
    for (int c0 = 0; c0 < ns; c0 += blockDim.x) {
        const int s = c0 + threadIdx.x;
        const bool f = s < ns && flag[s0 + s];
        int total;
        const int pre = block_prefix(f, wsum, total);
        if (f)
            for (int c = 0; c < d; ++c) cand[(size_t)(base + pre) * d + c] = stage[(size_t)(s0 + s) * d + c];
        base += total;
    }
}

// One block per run r with kk[r] > 0: its rows offs[r] .. offs[r + 1] - 1 with cand_ll > lmin[r], in
// row order, fill its walkers filled[r], filled[r] + 1, .. < kk[r] (walker j of run r: the walker w of
// the launch with run_of[w] = r, walker_of[w] = j): u, theta, lcur from the row.  filled[r] grows by
// what was taken, above[r] = the rows above lmin[r].  sel: scratch, one int per row.
__global__ void __launch_bounds__(kCompactThreads) region_pick_kernel(int k, int d, const int64_t *kk_all,
                                                                      const double *lmin, const int32_t *offs,
                                                                      const double *cand, const double *cand_th,
                                                                      const double *cand_ll, int32_t *sel,
                                                                      const int32_t *run_of, const int32_t *walker_of,
                                                                      double *u, double *theta, double *lcur,
                                                                      int32_t *filled, int32_t *above)
{
    const int r = blockIdx.x;
    const int64_t need = kk_all[r];
    if (need <= 0) return;
    __shared__ int wsum[kCompactThreads / 32];
    const int o0 = offs[r], nr = offs[r + 1] - o0, f0 = filled[r];
    const double lm = lmin[r];
    int cnt = 0;
    for (int c0 = 0; c0 < nr; c0 += blockDim.x) {
        const int s = c0 + threadIdx.x;
        const bool f = s < nr && cand_ll[o0 + s] > lm;
        int total;
        const int pre = block_prefix(f, wsum, total);
        if (f) sel[o0 + cnt + pre] = o0 + s;
        cnt += total;
    }
    __syncthreads();
    for (int w = threadIdx.x; w < k; w += blockDim.x) {
        if (run_of[w] != r) continue;
        const int t = walker_of[w] - f0;
        if (t < 0 || t >= cnt || walker_of[w] >= need) continue;
        const int row = sel[o0 + t];
        for (int c = 0; c < d; ++c) {
            u[(size_t)w * d + c] = cand[(size_t)row * d + c];
            theta[(size_t)w * d + c] = cand_th[(size_t)row * d + c];
        }
        lcur[w] = cand_ll[row];
    }
    if (threadIdx.x == 0) {
        filled[r] = (int32_t)(f0 + cnt < need ? f0 + cnt : need);
        above[r] = cnt;
    }
}

int sfail(const std::string &m)
{
    g_slice_error = m;
    return RVL_EINVAL;
}

// the mask of rvl_slice_phase_wrapped (NULL: none) into out[4]; any = some bit set
int read_wrap(const uint32_t *wrap_bits, int d, uint32_t *out, bool &any)
{
    any = false;
    if (!wrap_bits) return RVL_OK;
    for (int i = 0; i < 4; ++i) {
        // the bits at or above d of word i (word i holds coordinates 32 i .. 32 i + 31)
        const int lo = d - 32 * i;
        const uint32_t beyond = lo <= 0 ? 0xffffffffu : lo >= 32 ? 0u : ~((1u << lo) - 1u);
        if (wrap_bits[i] & beyond)
            return sfail("wrap_bits: bit " + std::to_string(32 * i + __builtin_ctz(wrap_bits[i] & beyond)) +
                         " set, but d = " + std::to_string(d));
        out[i] = wrap_bits[i];
        any = any || wrap_bits[i] != 0u;
    }
    return RVL_OK;
}

int check_runs(const rvl_slice_runs *runs)
{
    if (!runs) return sfail("runs is NULL");
    if (runs->n_runs < 1) return sfail("runs: n_runs must be >= 1");
    if (!runs->run_of || !runs->walker_of || !runs->seeds || !runs->lmin || !runs->chol || !runs->stats)
        return sfail("runs: run_of, walker_of, seeds, lmin, chol and stats must all be set");
    return RVL_OK;
}

template <bool kWrap, bool kRuns>
void launch_phase(int32_t phase, const ArgsT<kWrap, kRuns> &a, unsigned grid, unsigned threads,
                  cudaStream_t st)
{
    if (phase == 0) slice_begin_kernel<kWrap, kRuns><<<grid, threads, 0, st>>>(a);
    else if (phase == 1) slice_mid_kernel<kWrap, kRuns><<<grid, threads, 0, st>>>(a);
    else slice_end_kernel<kWrap, kRuns><<<grid, threads, 0, st>>>(a, phase == 2 ? 1 : 0);
}

int launched()
{
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        g_slice_error = cudaGetErrorString(e);
        return RVL_ECUDA;
    }
    return RVL_OK;
}

int slice_phase(int32_t phase, const rvl_slice_args *s, const rvl_slice_runs *runs,
                const uint32_t *wrap_bits, void *stream)
{
    if (!s) return sfail("args is NULL");
    if (s->k <= 0 || s->d <= 0 || s->d > kMaxDim || s->n_out < 1 || s->m < 1 || s->m > 64)
        return sfail("bad sizes (k > 0, 0 < d <= 128, n_out >= 1, 1 <= m <= 64)");
    SliceArgsWrap a{};
    bool wrap = false;
    if (const int rc = read_wrap(wrap_bits, s->d, a.wrap, wrap)) return rc;
    a.k = s->k; a.d = s->d; a.n_out = s->n_out; a.m = s->m; a.seed = s->seed; a.move = s->move;
    a.shrink_round = s->shrink_round;
    a.lmin = (const double *)s->lmin; a.chol = (const double *)s->chol; a.u = (double *)s->u;
    a.theta = (double *)s->theta; a.lcur = (double *)s->lcur; a.dirn = (double *)s->dirn;
    a.lo = (double *)s->lo; a.hi = (double *)s->hi; a.lo2 = (double *)s->lo2; a.hi2 = (double *)s->hi2;
    a.tval = (double *)s->tval; a.pending = (int *)s->pending;
    a.cand_o = (double *)s->cand_out; a.inside_o = (uint8_t *)s->inside_out; a.ll_o = (const double *)s->ll_out;
    a.cand = (double *)s->cand; a.inside = (uint8_t *)s->inside; a.cand_ll = (const double *)s->cand_ll;
    a.cand_th = (const double *)s->cand_th; a.stats = (unsigned long long *)s->stats;
    const int wpb = 4;
    const unsigned grid = (unsigned)((s->k + wpb - 1) / wpb);
    cudaStream_t st = (cudaStream_t)stream;
    if (phase < 0 || phase > 3)
        return sfail("phase must be 0 (begin), 1 (mid), 2 (end + more candidates) or 3 (end)");
    if (runs) {
        if (const int rc = check_runs(runs)) return rc;
        a.seed = 0;
        a.lmin = (const double *)runs->lmin; a.chol = (const double *)runs->chol;
        a.stats = (unsigned long long *)runs->stats;
        const int32_t *run_of = (const int32_t *)runs->run_of, *walker_of = (const int32_t *)runs->walker_of;
        const uint64_t *seeds = (const uint64_t *)runs->seeds;
        if (wrap) {
            WithRuns<SliceArgsWrap> b{};
            static_cast<SliceArgsWrap &>(b) = a;
            b.run_of = run_of; b.walker_of = walker_of; b.seeds = seeds;
            launch_phase<true, true>(phase, b, grid, wpb * 32, st);
        } else {
            WithRuns<SliceArgs> b{};
            static_cast<SliceArgs &>(b) = a;
            b.run_of = run_of; b.walker_of = walker_of; b.seeds = seeds;
            launch_phase<false, true>(phase, b, grid, wpb * 32, st);
        }
    } else if (wrap) {
        launch_phase<true, false>(phase, a, grid, wpb * 32, st);
    } else {
        launch_phase<false, false>(phase, a, grid, wpb * 32, st);
    }
    return launched();
}

int live_args(const rvl_slice_runs *runs, const rvl_slice_live *l, LiveArgs &a)
{
    if (!runs) return sfail("runs is NULL");
    if (!l) return sfail("live is NULL");
    if (runs->n_runs < 1 || l->nlive < 3 || l->d <= 0 || l->d > kMaxDim)
        return sfail("bad sizes (n_runs >= 1, nlive >= 3, 0 < d <= 128)");
    if (!runs->seeds || !l->u_live) return sfail("runs->seeds and live->u_live must be set");
    a.n_runs = runs->n_runs; a.nlive = l->nlive; a.d = l->d; a.round = l->round;
    a.seeds = (const uint64_t *)runs->seeds; a.u_live = (double *)l->u_live;
    a.th_live = (const double *)l->th_live; a.l_live = (const double *)l->l_live;
    a.order = (const int64_t *)l->order; a.kk = (const int64_t *)l->kk;
    return RVL_OK;
}

// the common checks of rvl_slice_runs_radius / _travel (seeds are not needed)
int adapt_args(const rvl_slice_runs *runs, const rvl_slice_live *l, const uint32_t *wrap_bits, const void *rad2,
               LiveArgs &a, Wrap4 &wr)
{
    if (!runs) return sfail("runs is NULL");
    if (!l) return sfail("live is NULL");
    if (runs->n_runs < 1 || l->nlive < 3 || l->d <= 0 || l->d > kMaxDim)
        return sfail("bad sizes (n_runs >= 1, nlive >= 3, 0 < d <= 128)");
    if (!l->u_live || !l->kk || !runs->chol || !rad2)
        return sfail("live->u_live, live->kk, runs->chol and rad2 must be set");
    bool any = false;
    if (const int rc = read_wrap(wrap_bits, l->d, wr.w, any)) return rc;
    a.n_runs = runs->n_runs; a.nlive = l->nlive; a.d = l->d; a.round = l->round;
    a.u_live = (double *)l->u_live; a.order = (const int64_t *)l->order; a.kk = (const int64_t *)l->kk;
    return RVL_OK;
}

// lets `kernel` take `smem` bytes of dynamic shared memory
template <class K>
int allow_bytes(K kernel, size_t smem)
{
    if (smem <= 48 * 1024) return RVL_OK;
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
        g_slice_error = cudaGetErrorString(e);
        return RVL_ECUDA;
    }
    return RVL_OK;
}

// lets `kernel` take adapt_smem(d) bytes of dynamic shared memory (up to 197 KB at d = 128)
template <class K>
int allow_smem(K kernel, int d)
{
    return allow_bytes(kernel, adapt_smem(d));
}

// the common checks of the region entry points: runs, live and their sizes, the mask, seeds / chol /
// u_live / order / kk of the runs and live points
int region_args(const rvl_region_args *g, const rvl_slice_runs *runs, const rvl_slice_live *l,
                const uint32_t *wrap_bits, LiveArgs &a, Wrap4 &wr)
{
    if (!g) return sfail("region is NULL");
    if (!runs) return sfail("runs is NULL");
    if (!l) return sfail("live is NULL");
    if (runs->n_runs < 1 || l->nlive < 3 || l->d <= 0 || l->d > kMaxDim)
        return sfail("bad sizes (n_runs >= 1, nlive >= 3, 0 < d <= 128)");
    if (!runs->seeds || !runs->chol || !l->u_live || !l->order || !l->kk)
        return sfail("runs->seeds, runs->chol, live->u_live, live->order and live->kk must be set");
    bool any = false;
    if (const int rc = read_wrap(wrap_bits, l->d, wr.w, any)) return rc;
    a.n_runs = runs->n_runs; a.nlive = l->nlive; a.d = l->d; a.round = l->round;
    a.seeds = (const uint64_t *)runs->seeds; a.u_live = (double *)l->u_live;
    a.order = (const int64_t *)l->order; a.kk = (const int64_t *)l->kk;
    return RVL_OK;
}

}  // namespace

extern "C" {

const char *rvl_slice_last_error(void) { return g_slice_error.c_str(); }

/* One phase of a slice move (see the header).  p: 16 device pointers in the order of
 * rvl_slice_args; all launches go to `stream`. */
int rvl_slice_phase(int32_t phase, const rvl_slice_args *s, void *stream)
{
    return slice_phase(phase, s, nullptr, nullptr, stream);
}

/* The same with circular coordinates: bit j & 31 of wrap_bits[j >> 5] set = coordinate j is taken
 * modulo 1 (see the header).  NULL or no bit set: exactly the launches of rvl_slice_phase. */
int rvl_slice_phase_wrapped(int32_t phase, const rvl_slice_args *s, const uint32_t wrap_bits[4],
                            void *stream)
{
    return slice_phase(phase, s, nullptr, wrap_bits, stream);
}

/* One phase for the walkers of several runs (see the header). */
int rvl_slice_phase_runs(int32_t phase, const rvl_slice_args *s, const rvl_slice_runs *runs,
                         const uint32_t wrap_bits[4], void *stream)
{
    if (!runs) return sfail("runs is NULL");
    return slice_phase(phase, s, runs, wrap_bits, stream);
}

int rvl_slice_runs_init(const rvl_slice_runs *runs, const rvl_slice_live *live, void *stream)
{
    LiveArgs a{};
    if (const int rc = live_args(runs, live, a)) return rc;
    const size_t n = (size_t)a.n_runs * a.nlive * a.d;
    runs_init_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a);
    return launched();
}

int rvl_slice_runs_whiten(const rvl_slice_runs *runs, const rvl_slice_live *live,
                          const uint32_t wrap_bits[4], void *stream)
{
    LiveArgs a{};
    if (const int rc = live_args(runs, live, a)) return rc;
    if (!live->order || !live->kk || !runs->chol) return sfail("live->order, live->kk and runs->chol must be set");
    uint32_t w[4] = {0u, 0u, 0u, 0u};
    bool wrap = false;
    if (const int rc = read_wrap(wrap_bits, a.d, w, wrap)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    double *chol = (double *)runs->chol;
    if (wrap) runs_whiten_kernel<true><<<a.n_runs, 256, 0, st>>>(a, chol, w[0], w[1], w[2], w[3]);
    else runs_whiten_kernel<false><<<a.n_runs, 256, 0, st>>>(a, chol, 0u, 0u, 0u, 0u);
    return launched();
}

int rvl_slice_runs_starts(const rvl_slice_args *s, const rvl_slice_runs *runs, const rvl_slice_live *live,
                          void *stream)
{
    LiveArgs a{};
    if (const int rc = live_args(runs, live, a)) return rc;
    if (!s) return sfail("args is NULL");
    if (s->k <= 0 || s->d != a.d) return sfail("bad sizes (args->k > 0, args->d == live->d)");
    if (!live->th_live || !live->l_live || !live->order || !live->kk || !live->start || !live->lstart ||
        !runs->run_of || !runs->walker_of || !s->u || !s->theta || !s->lcur)
        return sfail("starts: a device address is missing");
    const int wpb = 4;
    runs_starts_kernel<<<(unsigned)((s->k + wpb - 1) / wpb), wpb * 32, 0, (cudaStream_t)stream>>>(
        a, s->k, (const int32_t *)runs->run_of, (const int32_t *)runs->walker_of, (double *)s->u,
        (double *)s->theta, (double *)s->lcur, (int64_t *)live->start, (double *)live->lstart);
    return launched();
}

int rvl_slice_runs_radius(const rvl_slice_runs *runs, const rvl_slice_live *live, const uint32_t wrap_bits[4],
                          double *rad2, void *stream)
{
    LiveArgs a{};
    Wrap4 wr{};
    if (const int rc = adapt_args(runs, live, wrap_bits, rad2, a, wr)) return rc;
    if (!live->order) return sfail("live->order must be set");
    if (const int rc = allow_smem(runs_radius_kernel, a.d)) return rc;
    runs_radius_kernel<<<a.n_runs, kAdaptThreads, adapt_smem(a.d), (cudaStream_t)stream>>>(
        a, (const double *)runs->chol, wr, rad2);
    return launched();
}

int rvl_slice_runs_travel(const rvl_slice_args *s, const rvl_slice_runs *runs, const rvl_slice_live *live,
                          const uint32_t wrap_bits[4], const double *rad2, int32_t *far, void *stream)
{
    LiveArgs a{};
    Wrap4 wr{};
    if (const int rc = adapt_args(runs, live, wrap_bits, rad2, a, wr)) return rc;
    if (!s) return sfail("args is NULL");
    if (s->k <= 0 || s->d != a.d) return sfail("bad sizes (args->k > 0, args->d == live->d)");
    if (!s->u || !runs->run_of || !live->start || !far)
        return sfail("travel: args->u, runs->run_of, live->start and far must be set");
    if (const int rc = allow_smem(runs_travel_kernel, a.d)) return rc;
    runs_travel_kernel<<<a.n_runs, kAdaptThreads, adapt_smem(a.d), (cudaStream_t)stream>>>(
        a, s->k, (const int32_t *)runs->run_of, (const int64_t *)live->start, (const double *)s->u,
        (const double *)runs->chol, wr, rad2, far);
    return launched();
}

int rvl_region_runs_radius(const rvl_region_args *g, const rvl_slice_runs *runs, const rvl_slice_live *live,
                           const uint32_t wrap_bits[4], void *stream)
{
    LiveArgs a{};
    Wrap4 wr{};
    if (const int rc = region_args(g, runs, live, wrap_bits, a, wr)) return rc;
    if (g->num_bootstraps < 1 || g->num_bootstraps > 65536) return sfail("num_bootstraps must be in [1, 65536]");
    if (!g->rad2) return sfail("region->rad2 must be set");
    const size_t smem = boot_smem(a.d, a.nlive);
    if (smem > 227 * 1024) return sfail("nlive too large: the bootstrap's flags do not fit in shared memory");
    if (const int rc = allow_bytes(region_radius_kernel, smem)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    double *rad2 = (double *)g->rad2;
    region_clear_kernel<<<(unsigned)((a.n_runs + 127) / 128), 128, 0, st>>>(a, rad2);
    region_radius_kernel<<<dim3((unsigned)g->num_bootstraps, (unsigned)a.n_runs), kAdaptThreads, smem, st>>>(
        a, (const double *)runs->chol, wr, rad2);
    return launched();
}

int rvl_region_runs_draw(const rvl_region_args *g, const rvl_slice_runs *runs, const rvl_slice_live *live,
                         const uint32_t wrap_bits[4], void *stream)
{
    LiveArgs a{};
    Wrap4 wr{};
    if (const int rc = region_args(g, runs, live, wrap_bits, a, wr)) return rc;
    if (g->batch > 0xFFFFu) return sfail("region->batch must be below 65536");
    if (g->max_slots < 0) return sfail("region->max_slots must be >= 0");
    if (!g->rad2 || !g->slot_base || !g->stage || !g->flag || !g->count || !g->offs || !g->cand)
        return sfail("draw: region->rad2, slot_base, stage, flag, count, offs and cand must be set");
    if (const int rc = allow_smem(region_draw_kernel, a.d)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    int32_t *count = (int32_t *)g->count;
    const int32_t *slot_base = (const int32_t *)g->slot_base;
    if (cudaMemsetAsync(count, 0, sizeof(int32_t) * a.n_runs, st) != cudaSuccess) return launched();
    if (g->max_slots > 0)
        region_draw_kernel<<<dim3((unsigned)((g->max_slots + kAdaptThreads - 1) / kAdaptThreads), (unsigned)a.n_runs),
                             kAdaptThreads, adapt_smem(a.d), st>>>(a, (const double *)runs->chol, wr,
                                                                   (const double *)g->rad2, g->batch, slot_base,
                                                                   (double *)g->stage, (uint8_t *)g->flag, count);
    region_compact_kernel<<<a.n_runs, kCompactThreads, 0, st>>>(a.n_runs, a.d, a.kk, slot_base, (const double *)g->stage,
                                                                (const uint8_t *)g->flag, count,
                                                                (int32_t *)g->offs, (double *)g->cand);
    return launched();
}

int rvl_region_runs_pick(const rvl_region_args *g, const rvl_slice_args *s, const rvl_slice_runs *runs,
                         const rvl_slice_live *live, void *stream)
{
    if (!g) return sfail("region is NULL");
    if (!s) return sfail("args is NULL");
    if (!runs) return sfail("runs is NULL");
    if (!live) return sfail("live is NULL");
    if (runs->n_runs < 1 || s->k <= 0 || s->d <= 0 || s->d > kMaxDim || s->d != live->d)
        return sfail("bad sizes (n_runs >= 1, args->k > 0, 0 < d <= 128, args->d == live->d)");
    if (!g->offs || !g->cand || !g->cand_th || !g->cand_ll || !g->sel || !g->filled || !g->above ||
        !s->u || !s->theta || !s->lcur || !runs->run_of || !runs->walker_of || !runs->lmin || !live->kk)
        return sfail("pick: a device address is missing");
    region_pick_kernel<<<runs->n_runs, kCompactThreads, 0, (cudaStream_t)stream>>>(
        s->k, s->d, (const int64_t *)live->kk, (const double *)runs->lmin, (const int32_t *)g->offs,
        (const double *)g->cand, (const double *)g->cand_th, (const double *)g->cand_ll, (int32_t *)g->sel,
        (const int32_t *)runs->run_of, (const int32_t *)runs->walker_of, (double *)s->u, (double *)s->theta,
        (double *)s->lcur, (int32_t *)g->filled, (int32_t *)g->above);
    return launched();
}

}  // extern "C"
