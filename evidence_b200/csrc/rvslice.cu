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
template <bool kWrap>
using ArgsT = typename std::conditional<kWrap, SliceArgsWrap, SliceArgs>::type;

constexpr double kHiClamp = 1.0 - 0x1p-53;

// the words of draw `tag` of walker w in this move.  The key is the seed alone and the walker is a
// counter word: Philox is a bijection of the counter under a fixed key, so no two (seed, walker)
// pairs share a stream (a key mixing seed and walker, e.g. seed ^ walker, would repeat across seeds)
__device__ __forceinline__ U4 draw(const SliceArgs &a, uint32_t tag, int w)
{
    return philox(U4{a.move, tag, (uint32_t)w, 0u}, (uint32_t)a.seed,
                  (uint32_t)(a.seed >> 32) + 0x51CEu);
}

template <bool kWrap>
__device__ __forceinline__ void write_candidate(const ArgsT<kWrap> &a, double *cand, uint8_t *inside,
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
template <bool kWrap>
__device__ __forceinline__ void propose_shrink(const ArgsT<kWrap> &a, int w, double lo, double hi,
                                               const double *ui, const double *di, int lane)
{
    const int C = a.m;
    for (int j = 0; j < a.m; ++j) {
        const U4 r = draw(a, 0x53480000u + a.shrink_round * 64u + (uint32_t)j, w);
        const double t = lo + (hi - lo) * u01(r.x, r.y);
        if (lane == 0) a.tval[(size_t)w * a.m + j] = t;
        write_candidate<kWrap>(a, a.cand, a.inside, w, j, C, t, ui, di, lane);
        if (t < 0.0) lo = t; else hi = t;
    }
    if (lane == 0) { a.lo2[w] = lo; a.hi2[w] = hi; }
}

template <bool kWrap>
__global__ void __launch_bounds__(128) slice_begin_kernel(const ArgsT<kWrap> a)
{
    const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (w >= a.k) return;
    __shared__ double sz[4][kMaxDim];
    double *z = sz[threadIdx.x >> 5];
    // z ~ N(0, I): Box-Muller on Philox words, two normals per counter
    double n2 = 0.0;
    for (int j = lane; j < a.d; j += 32) {
        const U4 r = draw(a, 0x44495200u + (uint32_t)(j >> 1), w);
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
        for (int l = 0; l <= j; ++l) acc += a.chol[(size_t)j * a.d + l] * z[l];
        di[j] = acc * inv;
    }
    __syncwarp();
    const U4 r = draw(a, 0x42524B00u, w);
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

template <bool kWrap>
__global__ void __launch_bounds__(128) slice_mid_kernel(const ArgsT<kWrap> a)
{
    const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (w >= a.k) return;
    const int C = 2 * a.n_out;
    const double lmin = *a.lmin;
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
    propose_shrink<kWrap>(a, w, lo, hi, a.u + (size_t)w * a.d, a.dirn + (size_t)w * a.d, lane);
}

template <bool kWrap>
__global__ void __launch_bounds__(128) slice_end_kernel(const ArgsT<kWrap> a, int propose_more)
{
    const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (w >= a.k) return;
    const int C = a.m;
    const double lmin = *a.lmin;
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
            if (lane == 0) { a.lcur[w] = a.cand_ll[s]; a.pending[w] = 0; atomicAdd(a.stats + 1, 1ull); }
            pend = 0;
        } else if (lane == 0) {
            a.lo[w] = a.lo2[w];
            a.hi[w] = a.hi2[w];
            if (!propose_more) atomicAdd(a.stats, 1ull);  // bracket not resolved: the walker stays
        }
    }
    __syncwarp();
    if (propose_more) {
        // still pending: m more candidates from the shrunken bracket; done: re-evaluate the current
        // point (keeps the launch shape fixed -- no compaction, no read-back)
        if (pend) propose_shrink<kWrap>(a, w, a.lo2[w], a.hi2[w], ui, a.dirn + (size_t)w * a.d, lane);
        else
            for (int j = 0; j < a.m; ++j) {
                write_candidate<kWrap>(a, a.cand, a.inside, w, j, C, 0.0, ui, a.dirn + (size_t)w * a.d, lane);
                if (lane == 0) a.inside[(size_t)w * C + j] = 0;
            }
    }
}

int sfail(const std::string &m)
{
    g_slice_error = m;
    return RVL_EINVAL;
}

int slice_phase(int32_t phase, const rvl_slice_args *s, const uint32_t *wrap_bits, void *stream)
{
    if (!s) return sfail("args is NULL");
    if (s->k <= 0 || s->d <= 0 || s->d > kMaxDim || s->n_out < 1 || s->m < 1 || s->m > 64)
        return sfail("bad sizes (k > 0, 0 < d <= 128, n_out >= 1, 1 <= m <= 64)");
    SliceArgsWrap a{};
    bool wrap = false;
    if (wrap_bits) {
        for (int i = 0; i < 4; ++i) {
            // the bits at or above d of word i (word i holds coordinates 32 i .. 32 i + 31)
            const int lo = s->d - 32 * i;
            const uint32_t beyond = lo <= 0 ? 0xffffffffu : lo >= 32 ? 0u : ~((1u << lo) - 1u);
            if (wrap_bits[i] & beyond)
                return sfail("wrap_bits: bit " + std::to_string(32 * i + __builtin_ctz(wrap_bits[i] & beyond)) +
                             " set, but d = " + std::to_string(s->d));
            a.wrap[i] = wrap_bits[i];
            wrap = wrap || wrap_bits[i] != 0u;
        }
    }
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
    if (wrap) {
        if (phase == 0) slice_begin_kernel<true><<<grid, wpb * 32, 0, st>>>(a);
        else if (phase == 1) slice_mid_kernel<true><<<grid, wpb * 32, 0, st>>>(a);
        else slice_end_kernel<true><<<grid, wpb * 32, 0, st>>>(a, phase == 2 ? 1 : 0);
    } else {
        const SliceArgs &b = a;
        if (phase == 0) slice_begin_kernel<false><<<grid, wpb * 32, 0, st>>>(b);
        else if (phase == 1) slice_mid_kernel<false><<<grid, wpb * 32, 0, st>>>(b);
        else slice_end_kernel<false><<<grid, wpb * 32, 0, st>>>(b, phase == 2 ? 1 : 0);
    }
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        g_slice_error = cudaGetErrorString(e);
        return RVL_ECUDA;
    }
    return RVL_OK;
}

}  // namespace

extern "C" {

const char *rvl_slice_last_error(void) { return g_slice_error.c_str(); }

/* One phase of a slice move (see the header).  p: 16 device pointers in the order of
 * rvl_slice_args; all launches go to `stream`. */
int rvl_slice_phase(int32_t phase, const rvl_slice_args *s, void *stream)
{
    return slice_phase(phase, s, nullptr, stream);
}

/* The same with circular coordinates: bit j & 31 of wrap_bits[j >> 5] set = coordinate j is taken
 * modulo 1 (see the header).  NULL or no bit set: exactly the launches of rvl_slice_phase. */
int rvl_slice_phase_wrapped(int32_t phase, const rvl_slice_args *s, const uint32_t wrap_bits[4],
                            void *stream)
{
    return slice_phase(phase, s, wrap_bits, stream);
}

}  // extern "C"
