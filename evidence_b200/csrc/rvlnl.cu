// rvlnl.cu — librvlnl.so: B200 (sm_100a) batched Keplerian RV log-likelihood + prior transform
// behind the C-ABI of include/rvlnl.h.  No CPU fallback, no dispatch: sm_100a only.
//
// Reference path replaced (paths relative to the reference checkout):
//   evidence/rvmodel/__init__.py:157-219  RVModel.log_likelihood      -> rv_lnl_kernel
//   evidence/rvmodel/__init__.py:343-463  kep_rv / modelk             -> point_setup + solve_planet;
//                                                                       at caller times: kepler_rv_kernel
//   evidence/rvmodel/trueanomaly.c:8-41   trueanomaly()               -> solve_planet / trueanomaly_kernel
//   evidence/rvmodel/__init__.py:222-273  drift                       -> epoch term of rv_lnl_kernel
//   evidence/rvmodel/__init__.py:59-80    BaseModel.logL              -> epoch term + slice reduce
//   evidence/ultranest/__init__.py:125-137 prior(hypercube)           -> prior_transform_kernel / point_prepare_kernel
//
// Layout.  Epoch data lives in HBM as columns [ncol][Npad] of doubles (t, vrad, svrad^2, then
// (t-tref)/365.25 when the model has a drift, then the linear-parameter columns) followed by
// Npad instrument ids (uint8); Npad = N rounded up to whole groups of four 32-epoch chunks (the last
// epoch repeated, masked).  The epoch axis is cut into Sm resident ranges of whole chunks -- the
// fewest that fit shared memory; block b serves range b % Sm and brings that range of every column
// into shared memory ONCE with 1-D TMA bulk copies (cp.async.bulk + mbarrier), then stays resident:
// its warps pull work items -- (point, sub-slice of the range) in phases from coarse to fine, see
// Phase below -- from a per-range work counter.  warp <-> one item, lanes <-> 32 epochs (x U = 2 or 4
// chunks in flight): all lanes of a warp share the eccentricity, so Newton iteration counts are
// nearly uniform and the loop exit / sin-cos path choice come from one warp redux per trip.  chi^2
// and log-det sums are reduced with warp shuffles.  A point that is cut into several items has its
// per-point constants derived once by a setup item at the head of the list (or by the prepare pass
// of the fused prior transform); every item writes its partial sums and the LAST item of the point
// to arrive adds them in slice order (deterministic) -- one launch per likelihood call.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <string>
#include <vector>

#include "../../include/rvlnl.h"
#include "rvl_lean.h"
#include "rvl_math.h"

namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kPlanetStride = 8;  // doubles per planet in the per-warp constant block
constexpr int kModelBytes = (int)((sizeof(rvl_model_desc) + 127) / 128 * 128);
// per-planet constants: 0 nmot, 1 M0, 2 ec, 3 A, 4 Bs, 5 Ce, 6 epoch, 7 -(A ec)


// Peer buffers of the fused all-gather: device pointers into the other ranks' (and our own)
// gathered lnL vectors (NVLink peer / symmetric memory).  Passed by value.
struct PeerOut {
    double *ptr[RVL_MAX_PEERS];
    int n;
    long long offset;  // element offset of this rank's block inside every gathered vector
    // completion signal (seq != 0): when the whole launch is done, slot flag_off + rank of every
    // peer buffer receives seq (64-bit, release at system scope) -- the consumer side waits for
    // all ranks' slots of its own buffer instead of running a barrier or a collective
    long long flag_off;
    unsigned long long seq;
    int rank;
};

// One phase of the work list of a queue.  Items idx0 .. (next phase's idx0 - 1) cover points
// pt0, pt0+1, ... ; every point is cut into S sub-slices of cps chunks (of the block's resident
// epoch range), one item each.  Phases run from coarse (whole points) to fine (a pair of chunks),
// so the items handed out last are the short ones: guided self-scheduling against the tail.
struct Phase {
    unsigned idx0;
    int S, cps;
    int shift;  // log2(S) when S is a power of two (the usual case), else -1
    long long pt0;
    long long part0;  // offset (in doubles) of this phase's partial sums
};
constexpr int kMaxPhases = 8;

struct KArgs {
    const rvl_model_desc *model;  // device copy
    const double *cols;           // [ncol][Npad]
    const uint8_t *inst;          // [Npad]
    const double *theta;          // [B][ndim]
    double *lnl;                  // [B]
    double *partial;              // per phase: [points][Sm*S][2] partial sums of the split points
    int *arrive;                  // [split points] items of the point finished so far (self-resetting)
    int *flags;                   // [B] 1 = invalid Keplerian (written by the prepare pass)
    const double *consts;         // [B][wstride] per-point constants from point_prepare_kernel, or NULL
    unsigned long long *counters; // 0 newton iters, 1 cap hits, 2 invalid points
    unsigned int *work;           // [Sm] dynamic work counters, [Sm] = blocks finished (self-resetting)
    long long B;
    long long ptS0;  // first point that is split into more than one item
    double cte;      // -0.5 N ln(2 pi)
    double tlo, thi; // range of the epochs (point_setup: is every mean anomaly in the fast range?)
    int N, Npad, ncol;
    int Sm, cpm;     // resident epoch ranges ("memory slices": block b holds range b % Sm), chunks each
    unsigned nitems; // compute items per queue
    unsigned n_setup; // setup items that precede them in the queue (one split point each), or 0
    unsigned seq;     // launch stamp of the `ready` flags
    double *gconsts;  // [n_setup][wstride] constants of the split points, written by the setup items
    unsigned *ready;  // [n_setup] seq*2 + invalid once the constants of the point are in gconsts
    int nph;
    int wstride;     // doubles of per-point constants
    int wblock;      // doubles per warp in shared memory: the constants + a staged theta row
    Phase ph[kMaxPhases];
    PeerOut peers;
    unsigned long long *trace;  // optional [grid*warps][4]: t_enter, t_ready, t_done (ns), items
};

// ---- shared-memory / TMA helpers (sm_90+ PTX) --------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, unsigned parity)
{
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity)
{
    while (!mbar_try_wait(bar, parity)) {
    }
}
// 1-D TMA: global -> shared, completion counted in bytes on the mbarrier.  bytes % 16 == 0.
__device__ __forceinline__ void tma_load_1d(void *dst, const void *src, unsigned bytes,
                                            uint64_t *bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
            "r"(smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u32(unsigned *p, unsigned v)
{
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int atom_add_acq_rel(int *p, int v)
{
    int o;
    asm volatile("atom.acq_rel.gpu.global.add.s32 %0, [%1], %2;" : "=r"(o) : "l"(p), "r"(v) : "memory");
    return o;
}

__device__ __forceinline__ double par_of(const rvl_param &p, const double *row)
{
    return p.slot >= 0 ? row[p.slot] : p.value;
}

// shared-memory loads through a 32-bit shared-window address (one live register per base
// pointer; stops the compiler from re-deriving generic addresses inside the hot loops)
__device__ __forceinline__ double lds_f64(uint32_t addr)
{
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ int lds_u8(uint32_t addr)
{
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return (int)v;
}

// ---- the sin/cos table of rvl::sincos_tab and the path thresholds (rvl_lean.h) ------------------
using rvl::g_sintab_hi;
using rvl::g_sintab_lo;
using rvl::SmemSinTab;
using rvl::kHiTrigMax;
using rvl::kHiTiny;
using rvl::kHiSmall;
using rvl::kHiMid;
using rvl::kHiMedium;
constexpr unsigned kSinTabHiBytes = rvl::kSinTabN * sizeof(double2);
constexpr unsigned kSinTabBytes = 2 * kSinTabHiBytes;
static_assert(kSinTabBytes % 128 == 0, "the epoch columns behind the table stay 128-byte aligned");

// huge / non-finite arguments: CUDA libdevice (Payne-Hanek), out of line and returned by value
__device__ __noinline__ double2 sincos_slow(double x)
{
    double s, c;
    sincos(x, &s, &c);
    return make_double2(s, c);
}
// high word of |x| as an integer: orders like |x| itself (positive doubles sort as integers)
__device__ __forceinline__ int abs_hi(double x) { return __double2hiint(x) & 0x7fffffff; }
#ifndef RVL_MEDIUM
#define RVL_MEDIUM 1
#endif

template <int U>
__device__ __forceinline__ bool any_big(const double (&E)[U])
{
    int emax = 0;
#pragma unroll
    for (int u = 0; u < U; ++u) emax = max(emax, abs_hi(E[u]));
    return __any_sync(kFull, !(emax < kHiTrigMax));
}

// ---- U epochs per lane x one planet: Kepler solves + RV terms -------------------------------
// Lanes freeze individually (trueanomaly.c:21: per-element stop): a frozen lane's step is exactly
// 0, so its E never moves again and `|d| > tol` keeps it inactive without a separate flag.
// iters[u] counts the Newton steps BEYOND the first (every solve takes at least one: the caller
// adds one per planet and live epoch).
//
// solve_planet_ref: the plain statement of the loop -- any tolerance, any |M| (libdevice sin/cos
// when an argument is >= 1e5 or not finite), VARIANT 1 = IEEE division + full sin/cos every step.
// It is the conservative kernel build (rvl_set_option("variant", 1), the in-product cross-check)
// and the fallback of the lean loop below.
template <int VARIANT, int U>
__device__ __forceinline__ void solve_planet_ref(const rvl::KTab &kt, const double (&t)[U], uint32_t pc, double tol,
                                                 int itmax, double (&rv)[U], int (&iters)[U],
                                                 int &caps, int done = 1)
{
    // `done`: Newton steps whose iteration counts the caller has already added (the lean loop
    // hands over after `done` steps; a lane is active in steps 1..last, so what is left to add is
    // max(last - done, 0)); 1 = only the first step, which the caller of solve_planet counts
    const double nmot = lds_f64(pc), M0 = lds_f64(pc + 8), ec = lds_f64(pc + 16),
                 epoch = lds_f64(pc + 48);
    double M[U], E[U], s[U], c[U], d[U];
    int last[U];
    bool big = false;
#pragma unroll
    for (int u = 0; u < U; ++u) {
        M[u] = rvl::mean_anomaly(nmot, t[u], epoch, M0);
        E[u] = M[u];
        big = big || !(abs_hi(M[u]) < kHiTrigMax);
        d[u] = 1e300;  // "no step taken yet": forces the full sin/cos on the first pass
        s[u] = 0.0;
        c[u] = 1.0;
        last[u] = 0;
    }
    // slow: some |M| >= 1e5 (or non-finite), or an eccentricity outside [-0.99, 0.99] (only
    // reachable with a nonsensical direct `ecc`): every sin/cos of this solve goes through
    // libdevice, which is valid for any argument
    const bool slow = __any_sync(kFull, big || !(ec >= -0.99));
    int trip = 0;  // warp-uniform number of Newton steps taken so far
    const int tol_hi = __double2hiint(tol);
    for (;;) {
        int hmax = 0;
#pragma unroll
        for (int u = 0; u < U; ++u) hmax = max(hmax, abs_hi(d[u]));
        const int wmax = (int)__reduce_max_sync(kFull, (unsigned)hmax);
        // (1) bring (sin E, cos E) up to date with the step d just taken
        if (VARIANT == 0 && wmax < kHiTiny) {
#pragma unroll
            for (int u = 0; u < U; ++u) rvl::advance_tiny(kt, d[u], s[u], c[u]);
        } else if (VARIANT == 0 && wmax < kHiSmall) {
#pragma unroll
            for (int u = 0; u < U; ++u) rvl::advance_small(kt, d[u], s[u], c[u]);
        } else if (VARIANT == 0 && !slow && wmax < kHiMid) {
#pragma unroll
            for (int u = 0; u < U; ++u) rvl::advance_mid(kt, d[u], s[u], c[u]);
        } else if (VARIANT == 0 && !slow && wmax < kHiMedium) {
#pragma unroll
            for (int u = 0; u < U; ++u) rvl::advance_medium(kt, d[u], s[u], c[u]);
        } else if (slow || (trip > 2 && any_big<U>(E))) {
            // |E| can only leave the fast range after >= 3 Newton steps (|step| <= 100 |f|)
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const double2 r = sincos_slow(E[u]);
                s[u] = r.x;
                c[u] = r.y;
            }
        } else {
#pragma unroll
            for (int u = 0; u < U; ++u) rvl::sincos_fast(kt, E[u], s[u], c[u]);
        }
        // (2) which lanes still iterate (trueanomaly.c:21); the cap (:32-33) bounds the loop
        bool pa[U];
#pragma unroll
        for (int u = 0; u < U; ++u) pa[u] = fabs(d[u]) > tol;
        if (trip >= itmax || wmax < tol_hi) break;  // high word below tol's: every |d| < tol
        if (wmax == tol_hi) {                       // rare tie on the high word: exact vote
            bool any_left = false;
#pragma unroll
            for (int u = 0; u < U; ++u) any_left = any_left || pa[u];
            if (!__any_sync(kFull, any_left)) break;
        }
        ++trip;
        // (3) one Newton step for the active lanes; a frozen lane's step is exactly 0
#pragma unroll
        for (int u = 0; u < U; ++u) {
            double En;
            if (VARIANT == 0) {
                rvl::newton_step(E[u], s[u], c[u], M[u], ec, En);
            } else {
                const double f = rvl::sub(rvl::sub(E[u], rvl::mul(ec, s[u])), M[u]);
                const double fp = rvl::sub(1.0, rvl::mul(ec, c[u]));
                En = rvl::sub(E[u], __ddiv_rn(f, fp));
            }
            En = pa[u] ? En : E[u];
            d[u] = rvl::sub(En, E[u]);  // exact
            E[u] = En;
            last[u] = pa[u] ? trip : last[u];
        }
    }
    const double A = lds_f64(pc + 24), Bs = lds_f64(pc + 32), Ce = lds_f64(pc + 40);
    const double mAec = lds_f64(pc + 56);
#pragma unroll
    for (int u = 0; u < U; ++u) {
        iters[u] += max(last[u] - done, 0);
        caps += (fabs(d[u]) > tol) ? 1 : 0;
        rv[u] = rvl::add(rv[u], VARIANT == 0 ? rvl::kepler_rv2(s[u], c[u], ec, A, Bs, Ce, mAec)
                                             : rvl::kepler_rv(s[u], c[u], ec, A, Bs, Ce));
    }
}

// The lean loop (VARIANT 0), for the reference tolerance and |M| < 1e5 -- everything a sampler
// ever asks for; anything else restarts in solve_planet_ref above (a cold, warp-uniform branch), so
// that the hot loop holds no call and no libdevice code.
// The cost of this loop is its TOTAL instruction count, not only its FP64 count: measured on B200
// (profiles/r2_*), cycles per solve = 2.0 x FP64 instructions + 0.84 x all other instructions.
// So, beyond the arithmetic of rvl_math.h:
//   * pass 1 (full sin/cos of M, every lane active) is peeled: no path selection, no freeze;
//   * the warp-wide maximum of |d| comes from ONE FMNMX with |.| modifiers on the high words read
//     as floats (they order like the doubles) and ONE redux to a uniform register;
//   * path selection is a two-level tree ordered by frequency; `wmax < tol` picks the short last
//     pass and leaves (a tie of the high words just runs one more, idle, pass);
//   * a lane freezes by zeroing the 20-bit seed of its reciprocal (ONE select on the high word):
//     r = 0 -> E' = fma(-f, 0, E) = E, d = 0, with no 64-bit select on E;
//   * iteration counts: one predicated add per step; cap hits are only looked for when the cap
//     was reached;
//   * whether the solves may run here at all (|M| inside the fast sin/cos range, e >= -0.99, the
//     reference tolerance) is decided once per point (point_setup, item_epochs), not per planet
//     and epoch group;
//   * each solve ADDS its velocity to rv[], and the cap exit finishes on the spot: the common
//     exit is then reached from the last pass alone and takes (sin E, cos E) from the registers
//     that pass left them in (a join in front of the velocity formula cost 16 moves per 4 solves).
template <int VARIANT, int U>
__device__ __forceinline__ void solve_planet(const rvl::KTab &kt, SmemSinTab tab, const double (&t)[U],
                                             uint32_t pc, double tol, int itmax, double (&rv)[U],
                                             int (&iters)[U], int &caps, bool lean)
{
    if (VARIANT != 0) {
        solve_planet_ref<VARIANT, U>(kt, t, pc, tol, itmax, rv, iters, caps);
        return;
    }
    const double nmot = lds_f64(pc), M0 = lds_f64(pc + 8), ec = lds_f64(pc + 16),
                 epoch = lds_f64(pc + 48);
    const int tol_hi = __double2hiint(tol);
    double M[U], E[U], s[U], c[U], d[U];
#pragma unroll
    for (int u = 0; u < U; ++u) M[u] = rvl::mean_anomaly(nmot, t[u], epoch, M0);
    // `lean` (warp-uniform, decided once per point by point_setup and item_epochs): every |M| of
    // the point is inside the fast sin/cos range, e >= -0.99, the reference tolerance, itmax >= 2
    bool fallback = !lean;
    int trip = 1;
    if (!fallback) {
        // pass 1 + step 1: E0 = M, every lane active (trueanomaly.c:19-29)
#pragma unroll
        for (int u = 0; u < U; ++u) {
            rvl::sincos_tab(kt, tab, M[u], s[u], c[u]);
            double En;
            rvl::newton_step(M[u], s[u], c[u], M[u], ec, En);
            d[u] = rvl::sub(En, M[u]);  // exact
            E[u] = En;
        }
#pragma unroll 2
        for (;;) {
            float hm = 0.0f;
#pragma unroll
            for (int u = 0; u < U; ++u) hm = fmaxf(hm, fabsf(__int_as_float(__double2hiint(d[u]))));
            const int wmax = (int)__reduce_max_sync(kFull, __float_as_uint(hm));
            // (1) bring (sin E, cos E) up to date with the step d just taken
            if (wmax < kHiSmall) {
                if (wmax < tol_hi) {  // every |d| < tol: the last pass
#pragma unroll
                    for (int u = 0; u < U; ++u) rvl::advance_final(kt, d[u], s[u], c[u]);
                    break;
                }
                if (wmax < kHiTiny) {
#pragma unroll
                    for (int u = 0; u < U; ++u) rvl::advance_tiny(kt, d[u], s[u], c[u]);
                } else {
#pragma unroll
                    for (int u = 0; u < U; ++u) rvl::advance_small(kt, d[u], s[u], c[u]);
                }
            } else if (wmax < kHiMedium) {
                if (wmax < kHiMid) {
#pragma unroll
                    for (int u = 0; u < U; ++u) rvl::advance_mid(kt, d[u], s[u], c[u]);
                } else {  // (a fresh sincos_tab here has fewer instructions, but measured slower:
                          // its two table loads per solve cost more than the five FP64 saved)
#pragma unroll
                    for (int u = 0; u < U; ++u) rvl::advance_medium(kt, d[u], s[u], c[u]);
                }
            } else {
                // |E| can only leave the fast range after >= 3 Newton steps (|step| <= 100 |f|)
                if (trip > 2 && any_big<U>(E)) { fallback = true; break; }
#pragma unroll
                for (int u = 0; u < U; ++u) rvl::sincos_tab(kt, tab, E[u], s[u], c[u]);
            }
            if (trip >= itmax) {  // the cap (trueanomaly.c:32-33): rare, finished on the spot so that
                                  // the common exit below is reached from the last pass alone and
                                  // takes (sin E, cos E) from where that pass left them (no moves)
                const double A = lds_f64(pc + 24), Bs = lds_f64(pc + 32), Ce = lds_f64(pc + 40);
                const double mAec = lds_f64(pc + 56);
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    caps += (fabs(d[u]) > tol) ? 1 : 0;
                    rv[u] = rvl::add(rv[u], rvl::kepler_rv2(s[u], c[u], ec, A, Bs, Ce, mAec));
                }
                return;
            }
            ++trip;
            // (2) one Newton step (trueanomaly.c:25-29); frozen lanes (|d| <= tol, :21) get r = 0
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const double x = rvl::fma_(-ec, c[u], 1.0);
                const double y0 = rvl::rcp_seed(x);
                // pa = |d| > tol (false for NaN, like the reference's test): the seed's high word
                // or 0, and the iteration count as ONE predicated add (a lane is active in steps
                // 1..k, so the count is k; the compiler's own form is an add plus a select)
                int yh;
                asm("{\n\t.reg .pred p;\n\t.reg .f64 a;\n\t"
                    "abs.f64 a, %3;\n\t"
                    "setp.gt.f64 p, a, %4;\n\t"
                    "selp.b32 %0, %2, 0, p;\n\t"
                    "@p add.s32 %1, %1, 1;\n\t}"
                    : "=r"(yh), "+r"(iters[u])
                    : "r"(__double2hiint(y0)), "d"(d[u]), "d"(tol));
                const double y = __hiloint2double(yh, 0);
                const double e = rvl::fma_(-x, y, 1.0);
                const double r = rvl::fma_(y, rvl::fma_(e, e, e), y);
#if RVL_FMA_F
                const double f = rvl::sub(rvl::fma_(-ec, s[u], E[u]), M[u]);
#else
                const double f = rvl::sub(rvl::sub(E[u], rvl::mul(ec, s[u])), M[u]);
#endif
                const double En = rvl::fma_(-f, r, E[u]);
                d[u] = rvl::sub(En, E[u]);  // exact; 0 for a frozen lane
                E[u] = En;
            }
        }
    }
    if (fallback) {  // (warp-uniform) restart in the general loop: same arithmetic, same trajectory
        solve_planet_ref<0, U>(kt, t, pc, tol, itmax, rv, iters, caps, trip);
        return;
    }
    const double A = lds_f64(pc + 24), Bs = lds_f64(pc + 32), Ce = lds_f64(pc + 40);
    const double mAec = lds_f64(pc + 56);
#pragma unroll
    for (int u = 0; u < U; ++u) rv[u] = rvl::add(rv[u], rvl::kepler_rv2(s[u], c[u], ec, A, Bs, Ce, mAec));
}

// ---- per-point setup: theta row -> per-warp constants (modelk :411-457, :181-192) ---------
// lane p < K handles planet p; lane i < n_inst handles instrument i; lane 0 the drift/linpar
// coefficients.  Returns (warp-uniform) whether the point is a valid Keplerian.
#ifndef RVL_SETUP_OUTLINE
#define RVL_SETUP_OUTLINE 1
#endif
#if RVL_SETUP_OUTLINE
#define RVL_SETUP_INLINE __noinline__
#else
#define RVL_SETUP_INLINE __forceinline__
#endif
__device__ RVL_SETUP_INLINE bool point_setup(const rvl_model_desc &m, const double *row,
                                            double *wc, int lane, double tlo, double thi)
{
    const int K = m.n_planets;
    bool bad = false;
    bool lean = true;  // this planet's solves may take the lean Newton loop (see solve_planet)
    const rvl::KTab kt = rvl::load_ktab();
    if (lane < K) {
        const rvl_planet_desc &pl = m.planet[lane];
        double amp = par_of(pl.amp, row);
        if (pl.amp_is_log) amp = rvl::exp_cr(amp);
        double per = par_of(pl.period, row);
        if (pl.period_is_log) per = rvl::exp_cr(per);  // THE nearest double (see rvl_math.h)
        const double a = par_of(pl.e1, row), b = par_of(pl.e2, row);
        double ecc, omega;
        if (pl.ecc_mode == RVL_ECC_SECOS_SESIN) {
            ecc = rvl::add(rvl::mul(a, a), rvl::mul(b, b));
            omega = atan2(b, a);
            bad = ecc > 1.0;
        } else if (pl.ecc_mode == RVL_ECC_ECOS_ESIN) {
            ecc = sqrt(rvl::add(rvl::mul(a, a), rvl::mul(b, b)));
            omega = atan2(b, a);
            bad = ecc > 1.0;
        } else {
            ecc = a;
            omega = b;
        }
        double M0 = par_of(pl.phase, row);
        if (pl.phase_mode == RVL_PHASE_ML0) M0 = rvl::sub(M0, omega);
        const double ec = ecc > 0.99 ? 0.99 : ecc;  // trueanomaly.c:11-12
        double sw, cw;
        if (abs_hi(omega) < kHiTrigMax) {
            rvl::sincos_fast(kt, omega, sw, cw);
        } else {
            const double2 r = sincos_slow(omega);
            sw = r.x;
            cw = r.y;
        }
        const double root = sqrt(rvl::mul(rvl::sub(1.0, ec), rvl::add(1.0, ec)));
        double *pc = wc + lane * kPlanetStride;
        pc[0] = __ddiv_rn(6.283185307179586, per);  // 2*np.pi/P_day (:459)
        pc[1] = M0;
        pc[2] = ec;
        pc[3] = rvl::mul(amp, cw);
        pc[4] = -rvl::mul(rvl::mul(amp, sw), root);
        pc[5] = rvl::mul(amp, rvl::mul(ecc, cw));
        pc[6] = par_of(pl.epoch, row);
        pc[7] = -rvl::mul(pc[3], ec);
        // |M| <= |n| max|t - epoch| + |M0| over the data set's epochs (padding repeats an epoch):
        // below the fast sin/cos range for every epoch, or the point takes the general loop.
        // NaN / Inf anywhere compares false.
        const double span = fmax(fabs(rvl::sub(tlo, pc[6])), fabs(rvl::sub(thi, pc[6])));
        lean = rvl::add(rvl::mul(fabs(pc[0]), span), fabs(M0)) < 0.99 * rvl::kTrigFastMax && ec >= -0.99;
    }
    double *ic = wc + K * kPlanetStride;
    if (lane < m.n_inst) {
        ic[2 * lane] = par_of(m.offset[lane], row);
        double j2 = 0.0;
        if (m.jitter_in_model) {
            const double j = par_of(m.jitter[lane], row);
            j2 = rvl::mul(j, j);
        }
        ic[2 * lane + 1] = j2;
    }
    double *dc = ic + 2 * m.n_inst;
    if (lane < 4) dc[lane] = m.drift_in_model ? par_of(m.drift[lane], row) : 0.0;
    if (lane < m.n_linpar) dc[4 + lane] = par_of(m.linpar[lane], row);
    lean = __all_sync(kFull, lean);
    if (lane == 0) dc[4 + m.n_linpar] = lean ? 1.0 : 0.0;
    __syncwarp();
    return !__any_sync(kFull, bad);
}

// ---- the epochs [c_lo, c_hi) x 32 of one work item, for the warp's current point ---------------
// Code generation note: the instruction selection of the Newton loop (coefficients as direct
// constant-bank operands, branches on uniform registers) is sensitive to what is inlined around
// it; with the setup-item consumer inlined next to it ptxas switched to LDCU-staged coefficients
// and convergence barriers inside the loop (+10% instructions per trip, -5% on the whole
// kernel).  point_setup and take_point_consts are therefore out of line; this function is
// inlined by default (RVL_OUTLINE=1 moves it out of line too, at the price of spills around it).
// The block-wide constants come from shared memory (HotCtx), the per-point constants from the
// warp's block at a_wc.
struct HotCtx {
    double tol;
    uint32_t a_t0, colb, a_inst0, lin0;  // shared-window addresses / strides of the epoch columns
    int K, itmax, has_drift, drift_hi, nlin, n_inst, e_base0, N;
};
struct ItemSums {
    double chi, prod;
    int esum, iters, caps, ok;
};

#ifndef RVL_OUTLINE
#define RVL_OUTLINE 0
#endif
#ifndef RVL_PIN_WC
#define RVL_PIN_WC 1
#endif
#if RVL_OUTLINE
#define RVL_ITEM_INLINE __noinline__
#else
#define RVL_ITEM_INLINE __forceinline__
#endif
template <int VARIANT, int U>
__device__ RVL_ITEM_INLINE ItemSums item_epochs(const rvl::KTab &kt, SmemSinTab tab, const HotCtx *hc,
                                                uint32_t a_wc_in, int c_lo, int c_hi, int lane)
{
#if RVL_PIN_WC
    // the address of the warp's constants is needed once per planet and epoch group; left to
    // itself ptxas re-derives it from %tid, the cluster rank and kernel parameters every time (19
    // instructions) rather than hold one register.  The result of a shuffle cannot be re-derived.
    const uint32_t a_wc = __shfl_sync(kFull, a_wc_in, 0);
#else
    const uint32_t a_wc = a_wc_in;
#endif
    const double tol = hc->tol;
    const int K = hc->K, itmax = hc->itmax, drift_hi = hc->drift_hi, nlin = hc->nlin, N = hc->N;
    const bool has_drift = hc->has_drift != 0;
    const uint32_t a_ic = a_wc + (uint32_t)(K * kPlanetStride) * 8u;
    const uint32_t a_dc = a_ic + (uint32_t)(2 * hc->n_inst) * 8u;
    const uint32_t a_t = hc->a_t0 + (uint32_t)lane * 8u;
    const uint32_t colb = hc->colb;
    const uint32_t a_inst = hc->a_inst0 + (uint32_t)lane;
    const uint32_t lin0 = hc->lin0;
    const int e_base = hc->e_base0 + lane;
    // the lean Newton loop: the point's flag (point_setup) and the launch-wide conditions
    const bool lean = lds_u32(a_dc + 32u + (uint32_t)nlin * 8u + 4u) != 0u &&
                      __double2hiint(tol) < rvl::kHiFinal && itmax >= 2;
    const bool extras = has_drift || nlin > 0;
    double chi = 0.0, prod = 1.0;
    int esum = 0, iters = 0, caps = 0;
    uint32_t worst = 0;  // unsigned maximum of (sign + biased exponent of a variance) - 1
    int nlive = 0;       // variances whose biased exponent went into esum
    for (int ch = c_lo; ch < c_hi; ch += U) {
        // U chunks of 32 epochs; a missing last chunk repeats the previous one, masked
        uint32_t off[U];
        bool live[U];
        double t[U], rvsum[U];
        int it_l[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const bool have = U == 4 || (ch + u) < c_hi;  // (U = 4: whole trips, see rv_lnl_kernel)
            const int cu = have ? ch + u : ch;
            off[u] = (uint32_t)cu * 256u;
            live[u] = have && (e_base + cu * 32) < N;
            t[u] = lds_f64(a_t + off[u]);
            rvsum[u] = 0.0;
            it_l[u] = 0;  // steps after the first; the first of each solve is added with nlive below
        }
        int cap_l = 0;
        for (int p = 0; p < K; ++p) {
            // each solve ADDS its planet's velocity to rvsum (kep_rv :383: the planets' sum, first
            // to last; 0 + v is v)
            solve_planet<VARIANT, U>(kt, tab, t, a_wc + (uint32_t)(p * kPlanetStride) * 8u, tol,
                                     itmax, rvsum, it_l, cap_l, lean);
        }
        caps += cap_l;  // (padded / repeated lanes included: a cap hit is a cap hit)
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint32_t ae = a_t + off[u];
            const int ii = lds_u8(a_inst + off[u] / 8u);
            const uint32_t ai = a_ic + (uint32_t)ii * 16u;
            const double rvm0 = rvl::add(lds_f64(ai), rvsum[u]);  // (rvsum is an exact 0 without planets)
            double rvm = rvm0;
            if (extras) {  // (one uniform test for the plain model: offsets + Keplerians only)
            if (has_drift) {
                // lin*tt + quad*tt^2 + cub*tt^3 + quar*tt^4, left to right (:271); a
                // coefficient that is absent from the model is an exact +0 term: skipped
                const double tt = lds_f64(ae + 3u * colb);
                double dr = rvl::mul(lds_f64(a_dc), tt);
                if (drift_hi > 0) {
                    const double t2 = rvl::mul(tt, tt);
                    dr = rvl::add(dr, rvl::mul(lds_f64(a_dc + 8), t2));
                    if (drift_hi > 1) {
                        dr = rvl::add(dr, rvl::mul(lds_f64(a_dc + 16), rvl::mul(t2, tt)));
                        if (drift_hi > 2)
                            dr = rvl::add(dr, rvl::mul(lds_f64(a_dc + 24), rvl::mul(t2, t2)));
                    }
                }
                rvm = rvl::add(rvm, dr);
            }
            for (int l = 0; l < nlin; ++l)
                rvm = rvl::add(rvm, rvl::mul(lds_f64(a_dc + 32u + (uint32_t)l * 8u),
                                             lds_f64(ae + lin0 + (uint32_t)l * colb)));
            }
            const double res = rvl::sub(lds_f64(ae + colb), rvm);
            const double var = rvl::add(lds_f64(ae + 2u * colb), lds_f64(ai + 8));
            const double term = rvl::mul(rvl::mul(res, res), rvl::rcp(rvl::add(var, var)));
            double mant;
            uint32_t be;
            rvl::split_raw(var, mant, be);
            if (live[u]) {
                chi = rvl::add(chi, term);
                prod = rvl::mul(prod, mant);
                esum += (int)be;  // biased: 1023 per term comes off at the end
                worst = max(worst, be - 1u);
                iters += it_l[u];
                ++nlive;  // (also: K first Newton steps, one per planet)
            }
        }
        if (((ch - c_lo) & 255) >= 254) {  // keep the mantissa product in range
            double mm;
            int ee;
            rvl::split_pos(prod, mm, ee);
            prod = mm;
            esum += ee;
        }
    }
    return ItemSums{chi, prod, esum - 1023 * nlive, iters + K * nlive, caps, worst < 0x7feu ? 1 : 0};
}

// Constants of a split point, published by a setup item: into the warp's block in shared memory.
// (pf_flag, pf0, pf1) is what the previous item requested ahead of time; if the point was not
// ready then, wait for its flag (the setup item is in flight on some warp) and load again.
// Out of line on purpose (see item_epochs).
__device__ __noinline__ unsigned take_point_consts(const double *src, const unsigned *flagp,
                                                   unsigned seq, double *wc, int wstride, int lane,
                                                   unsigned pf_flag, double pf0, double pf1)
{
    if ((pf_flag >> 1) != seq) {
        do {
            pf_flag = ld_acquire_u32(flagp);
        } while ((pf_flag >> 1) != seq);
        pf0 = lane < wstride ? __ldcg(src + lane) : 0.0;
        pf1 = lane + 32 < wstride ? __ldcg(src + lane + 32) : 0.0;
    }
    if (lane < wstride) wc[lane] = pf0;
    if (lane + 32 < wstride) wc[lane + 32] = pf1;
    for (int i = lane + 64; i < wstride; i += 32) wc[i] = __ldcg(src + i);
    __syncwarp();
    return pf_flag;
}

// ---- the likelihood kernel ------------------------------------------------------------------
// U = epochs per lane in flight (1: 1024 threads/SM at <=64 registers; 2: 512 threads/SM at
// <=128 registers, two chunks of 32 epochs per warp trip).
template <int VARIANT, int U, int THREADS>
__global__ void __launch_bounds__(THREADS, 1) rv_lnl_kernel(const KArgs a)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // [0,8) mbarrier, [16,128) HotCtx | [128, 128+sizeof(model)) model | sin/cos table |
    // epoch columns | inst ids | warp consts
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_raw);
    HotCtx *hc = reinterpret_cast<HotCtx *>(smem_raw + 16);
    static_assert(sizeof(HotCtx) <= 112, "HotCtx must fit in front of the model description");
    rvl_model_desc *sm = reinterpret_cast<rvl_model_desc *>(smem_raw + 128);
    const int sl = blockIdx.x % a.Sm;
    const int Ctot = (a.N + 31) / 32;
    const int c0 = sl * a.cpm;
    // chunks resident in this block (>= 1 by construction); U = 4: in whole warp trips -- the
    // columns in HBM are padded to whole groups of 4 chunks (the last epoch repeated), so a trip
    // never meets a missing chunk, only masked epochs (the narrower builds keep the test: at 72
    // registers the code without it spills more than it saves)
    const int nch0 = min(a.cpm, Ctot - c0);
    const int nch = U == 4 ? (nch0 + 3) / 4 * 4 : nch0;
    const int ne = nch * 32;
    unsigned char *stab = smem_raw + 128 + kModelBytes;
    double *scol = reinterpret_cast<double *>(stab + kSinTabBytes);
    uint8_t *sinst = reinterpret_cast<uint8_t *>(scol + (size_t)a.ncol * ne);
    double *wconst = reinterpret_cast<double *>(
        stab + kSinTabBytes + (((size_t)a.ncol * ne * 8 + ne + 127) / 128) * 128);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned n_items = 0;
    if (a.trace && lane == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        a.trace[((size_t)blockIdx.x * (blockDim.x >> 5) + warp) * 4] = t;
    }

    if (tid == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        const unsigned col_bytes = (unsigned)ne * 8u;
        mbar_expect_tx(bar, col_bytes * (unsigned)a.ncol + (unsigned)ne + kSinTabBytes);
        tma_load_1d(stab, g_sintab_hi, kSinTabHiBytes, bar);
        tma_load_1d(stab + kSinTabHiBytes, g_sintab_lo, kSinTabBytes - kSinTabHiBytes, bar);
        for (int cidx = 0; cidx < a.ncol; ++cidx)
            tma_load_1d(scol + (size_t)cidx * ne, a.cols + (size_t)cidx * a.Npad + (size_t)c0 * 32,
                        col_bytes, bar);
        tma_load_1d(sinst, a.inst + (size_t)c0 * 32, (unsigned)ne, bar);
    }
    // model description: plain cooperative copy (1.6 KB) while the TMA is in flight
    {
        const int nw = (int)(sizeof(rvl_model_desc) / 4);
        const uint32_t *src = reinterpret_cast<const uint32_t *>(a.model);
        uint32_t *dst = reinterpret_cast<uint32_t *>(sm);
        for (int i = tid; i < nw; i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    mbar_wait(bar, 0);

    const rvl_model_desc &m = *sm;
    const int K = m.n_planets;
    const double tol = m.tol;
    const int itmax = m.itmax;
    const bool has_drift = m.drift_in_model != 0;
    int drift_hi = 0;  // highest drift coefficient that is a parameter or a non-zero constant
    for (int i = 1; i < 4; ++i)
        if (m.drift[i].slot >= 0 || m.drift[i].value != 0.0) drift_hi = i;
    const int nlin = m.n_linpar;
    double *wc = wconst + (size_t)warp * a.wblock;
    double *srow = wc + a.wstride;  // the point's theta row, staged by one coalesced read
    // (theta may live in pinned host memory -- zero-copy calls -- where the scattered 8-byte
    // reads of point_setup would each be a PCIe transaction)
    auto stage_row = [&](const double *g) {
        __syncwarp();
        for (int i = lane; i < m.ndim; i += 32) srow[i] = g[i];
        __syncwarp();
    };
    // 32-bit shared-window addresses of everything the hot loop reads
    const uint32_t a_wc = smem_u32(wc);
    const uint32_t a_ic = a_wc + (uint32_t)(K * kPlanetStride) * 8u;
    const uint32_t a_t = smem_u32(scol) + (uint32_t)lane * 8u;
    const uint32_t colb = (uint32_t)ne * 8u;  // bytes per column
    const uint32_t a_inst = smem_u32(sinst) + (uint32_t)lane;
    const uint32_t lin0 = (uint32_t)(3 + (has_drift ? 1 : 0)) * colb;
    if (tid == 0) {
        hc->tol = tol; hc->a_t0 = smem_u32(scol); hc->colb = colb; hc->a_inst0 = smem_u32(sinst);
        hc->lin0 = lin0; hc->K = K; hc->itmax = itmax; hc->has_drift = has_drift ? 1 : 0;
        hc->drift_hi = drift_hi; hc->nlin = nlin; hc->n_inst = m.n_inst;
        hc->e_base0 = c0 * 32;  // global epoch index of lane 0 in chunk 0
        hc->N = a.N;
    }
    __syncthreads();

    // the constants of the sin/cos kernels, loaded once and kept (see rvl_math.h: KTab)
#ifndef RVL_PIN_KTAB
#define RVL_PIN_KTAB 1
#endif
    const rvl::KTab kt = RVL_PIN_KTAB ? rvl::load_ktab_pinned() : rvl::load_ktab();
    const SmemSinTab tab{smem_u32(stab)};
    unsigned long long tot_iters = 0, tot_caps = 0, tot_invalid = 0;
    if (a.trace && lane == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        a.trace[((size_t)blockIdx.x * (blockDim.x >> 5) + warp) * 4 + 1] = t;
    }

    // work queue of this epoch range: the index of the NEXT item is requested while the current
    // one is computed, so the atomic's round trip (~1 us) is off the critical path
    unsigned idx = 0;
    if (lane == 0) idx = atomicAdd(&a.work[sl], 1u);
    idx = __shfl_sync(kFull, idx, 0);

    // ---- setup items (they come first in the queue): the per-point constants of the points that
    // are cut into several work items are derived ONCE, by whichever warp draws the item, and
    // published through `ready`.  Consumers can only ever wait for a warp that is already running.
    while (idx < a.n_setup) {
        unsigned next = 0;
        if (lane == 0) next = atomicAdd(&a.work[sl], 1u);
        const long long pt = a.ptS0 + (long long)idx;
        stage_row(a.theta + pt * m.ndim);
        const bool valid = point_setup(m, srow, a.gconsts + (size_t)idx * a.wstride, lane, a.tlo, a.thi);
        __threadfence();
        __syncwarp();
        if (lane == 0) st_release_u32(a.ready + idx, a.seq * 2u + (valid ? 0u : 1u));
        idx = __shfl_sync(kFull, next, 0);
    }
    idx -= a.n_setup;

    // item -> (point, sub-slice of the resident chunks); all warp-uniform.  The item is carried as
    // (phase | sub-slice << 3, index of the point within the phase): few registers across the
    // hot loop; everything else is re-derived from the phase table in the constant bank.
    unsigned it_ks = 0, it_jp = 0;
    auto decode = [&](unsigned i) {
        int k = 0;
        while (k + 1 < a.nph && i >= a.ph[k + 1].idx0) ++k;
        const unsigned Sk = (unsigned)a.ph[k].S;
        const unsigned j = i - a.ph[k].idx0;
        const int sh = a.ph[k].shift;
        it_jp = sh >= 0 ? (j >> sh) : (j / Sk);
        it_ks = (unsigned)k | ((j - it_jp * Sk) << 3);
    };
    if (idx < a.nitems) decode(idx);
    // constants of the NEXT item, requested before the current item's reduction
    unsigned pf_flag = 0;
    double pf0 = 0.0, pf1 = 0.0;
    bool pf_have = false;
    while (idx < a.nitems) {
        const long long pt = a.ph[it_ks & 7u].pt0 + (long long)it_jp;
        const double *row = a.theta + pt * m.ndim;
        unsigned next = 0;
        if (lane == 0) next = atomicAdd(&a.work[sl], 1u);

        __syncwarp();
        bool valid;
        if (a.consts) {  // constants were prepared once per point (S > 1 / fused transform)
            const double *src = a.consts + (size_t)pt * a.wstride;
            for (int i = lane; i < a.wstride; i += 32) wc[i] = __ldg(src + i);
            valid = __ldg(a.flags + pt) == 0;
            __syncwarp();
        } else if (a.n_setup && pt >= a.ptS0) {  // published by a setup item
            const unsigned si = (unsigned)(pt - a.ptS0);
            const double *src = a.gconsts + (size_t)si * a.wstride;
            pf_flag = take_point_consts(src, a.ready + si, a.seq, wc, a.wstride, lane,
                                        pf_have ? pf_flag : 0u, pf0, pf1);
            // (a vote makes the flag provably warp-uniform for the compiler: the hot loop below
            // must stay under uniform control flow)
            valid = __all_sync(kFull, (pf_flag & 1u) == 0u);
        } else {
            stage_row(row);
            valid = point_setup(m, srow, wc, lane, a.tlo, a.thi);
        }
        // what the rest of this iteration needs of the current item (the item variables are
        // re-used for the next one before the reduction)
        const unsigned c_ks = it_ks, c_jp = it_jp;
        const int c_lo = (int)(c_ks >> 3) * a.ph[c_ks & 7u].cps;
        const int c_hi = min(nch, c_lo + a.ph[c_ks & 7u].cps);  // may be empty in a short last range

        // ---- the item's epochs: Kepler solves + Gaussian terms (out of line, see item_epochs) ----
        ItemSums sums{0.0, 1.0, 0, 0, 0, 1};
        if (valid) sums = item_epochs<VARIANT, U>(kt, tab, hc, a_wc, c_lo, c_hi, lane);
        double chi = sums.chi, prod = sums.prod;
        int esum = sums.esum;
        const int iters = sums.iters, caps = sums.caps;
        const bool ok = sums.ok != 0;

        // ---- next item: decode it and request its constants now, so that they arrive while this
        // item's sums are being reduced
        idx = __shfl_sync(kFull, next, 0) - a.n_setup;
        pf_have = false;
        if (idx < a.nitems) {
            decode(idx);
            const long long npt = a.ph[it_ks & 7u].pt0 + (long long)it_jp;
            if (a.n_setup && npt >= a.ptS0) {
                const unsigned si = (unsigned)(npt - a.ptS0);
                const double *src = a.gconsts + (size_t)si * a.wstride;
                pf_flag = ld_acquire_u32(a.ready + si);
                pf0 = lane < a.wstride ? __ldcg(src + lane) : 0.0;
                pf1 = lane + 32 < a.wstride ? __ldcg(src + lane + 32) : 0.0;
                pf_have = true;
            }
        }

        // ---- slice reduction: chi^2 sum, mantissa product, exponent sum ----
        double S1, S2;
        if (valid) {
            const bool all_ok = __all_sync(kFull, ok);
            if (all_ok) {
                {  // every lane's mantissa product back to [1,2): 32 of them multiply to < 2^32
                    double mm;
                    int ee;
                    rvl::split_pos(prod, mm, ee);
                    prod = mm;
                    esum += ee;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    chi = rvl::add(chi, __shfl_xor_sync(kFull, chi, o));
                    prod = rvl::mul(prod, __shfl_xor_sync(kFull, prod, o));
                }
                esum = __reduce_add_sync(kFull, esum);
                // sum ln sqrt(var) = 0.5 (ln prod + esum ln 2); prod < 2^32 is split once more so
                // that the one logarithm of the item is that of a mantissa (no special cases)
                double pm;
                int pe, ph;
                rvl::split_pos(prod, pm, pe);
                const double lm = rvl::log_mantissa(pm, ph);
                const double es = (double)(esum + pe + ph);
                const double ld = rvl::fma_(es, rvl::kLn2Hi, rvl::fma_(es, rvl::kLn2Lo, lm));
                S1 = rvl::mul(0.5, ld);
            } else {
                // a variance that is zero / subnormal / negative / non-finite: plain logs
                double acc = 0.0;
                for (int ch = c_lo; ch < c_hi; ++ch) {
                    const uint32_t o8 = (uint32_t)ch * 256u;
                    if ((c0 * 32 + lane + ch * 32) < a.N) {
                        const int ii = lds_u8(a_inst + o8 / 8u);
                        const double var = rvl::add(lds_f64(a_t + o8 + 2u * colb),
                                                    lds_f64(a_ic + (uint32_t)ii * 16u + 8u));
                        acc = rvl::add(acc, log(sqrt(var)));
                    }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    acc = rvl::add(acc, __shfl_xor_sync(kFull, acc, o));
                    chi = rvl::add(chi, __shfl_xor_sync(kFull, chi, o));
                }
                S1 = acc;
            }
            S2 = chi;
            tot_iters += (unsigned long long)__reduce_add_sync(kFull, iters);
            tot_caps += (unsigned long long)__reduce_add_sync(kFull, caps);
        } else {
            S1 = 0.0;
            S2 = 0.0;
            if (sl == 0 && (c_ks >> 3) == 0u) ++tot_invalid;
        }
        const int c_k = (int)(c_ks & 7u), c_Sk = a.ph[c_ks & 7u].S, c_ss = (int)(c_ks >> 3);
        const long long c_pt = a.ph[c_k].pt0 + (long long)c_jp;
        const int Stot = a.Sm * c_Sk;  // items of this point
        bool finish = Stot == 1;
        if (!finish) {
            // this item's partial sums; the item that arrives LAST adds all of them in epoch order
            // (deterministic) -- no second kernel
            const int slot = sl * c_Sk + c_ss;
            double *pp = a.partial + a.ph[c_k].part0 + (size_t)c_jp * (size_t)Stot * 2;
            int *arr = a.arrive + (c_pt - a.ptS0);
            int old = 0;
            if (lane == 0) {
                pp[2 * slot] = S1;
                pp[2 * slot + 1] = S2;
                old = atom_add_acq_rel(arr, 1);  // release: the two stores above are visible first
            }
            old = __shfl_sync(kFull, old, 0);
            if (old == Stot - 1) {
                finish = true;
                if (lane == 0) *arr = 0;  // ready for the next launch
                __threadfence();
                S1 = 0.0;
                S2 = 0.0;
                for (int base = 0; base < Stot; base += 32) {
                    double v1 = 0.0, v2 = 0.0;
                    if (base + lane < Stot) {
                        v1 = __ldcg(pp + 2 * (base + lane));
                        v2 = __ldcg(pp + 2 * (base + lane) + 1);
                    }
                    const int n = min(32, Stot - base);
                    for (int i = 0; i < n; ++i) {
                        S1 = rvl::add(S1, __shfl_sync(kFull, v1, i));
                        S2 = rvl::add(S2, __shfl_sync(kFull, v2, i));
                    }
                }
            }
        }
        if (finish && lane == 0) {
            // (cte - sum ln sqrt var) - sum r^2/(2 var)   (:80); invalid -> -1e30 (:203)
            const double v = valid ? rvl::sub(rvl::sub(a.cte, S1), S2) : -1e30;
            a.lnl[c_pt] = v;
            // fused all-gather: the value goes straight into every rank's gathered vector (NVLink)
            for (int r = 0; r < a.peers.n; ++r) a.peers.ptr[r][a.peers.offset + c_pt] = v;
        }
        ++n_items;
    }
    if (a.trace && lane == 0) {
        unsigned long long t_done;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_done));
        unsigned long long *o = a.trace + ((size_t)blockIdx.x * (blockDim.x >> 5) + warp) * 4;
        o[2] = t_done; o[3] = n_items;
    }
    if (lane == 0) {
        if (tot_iters) atomicAdd(&a.counters[0], tot_iters);
        if (tot_caps) atomicAdd(&a.counters[1], tot_caps);
        if (tot_invalid) atomicAdd(&a.counters[2], tot_invalid);
    }
    // the last block to leave re-arms the work counters for the next launch on this handle
    __syncthreads();
    if (tid == 0) {
        // release: this block's stores (to peers: at system scope) are ordered before its arrival
        if (a.peers.n) asm volatile("fence.acq_rel.sys;" ::: "memory"); else __threadfence();
        if (atomicAdd(&a.work[a.Sm], 1u) == gridDim.x - 1) {
            for (int i = 0; i <= a.Sm; ++i) a.work[i] = 0u;
            if (a.peers.seq) {
                // acquire side of the other blocks' arrivals, then ONE fence orders everything
                // before the completion slots; the slot stores themselves are relaxed and posted
                // (a release per store would serialise one NVLink round trip per peer: measured
                // +2.2 us per peer inside the kernel)
                asm volatile("fence.acq_rel.sys;" ::: "memory");
                for (int r = 0; r < a.peers.n; ++r) {
                    unsigned long long *f = reinterpret_cast<unsigned long long *>(a.peers.ptr[r]) +
                                            a.peers.flag_off + a.peers.rank;
                    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(f), "l"(a.peers.seq)
                                 : "memory");
                }
            }
        }
    }
}

// consumer side of the fused all-gather: returns once every rank's completion slot holds >= seq.
// The wait is bounded: after timeout_ns of the device's global timer a lane gives up, records
// (seq, bit mask of the missing ranks) in `status` (mapped host memory of the handle) and returns, so a
// peer that died cannot hang this rank's stream forever; the host side reports RVL_EPEER.
__global__ void wait_flags_kernel(const unsigned long long *flags, int n, unsigned long long seq,
                                  unsigned long long timeout_ns, unsigned long long *status)
{
    if ((int)threadIdx.x < n) {
        unsigned long long v, t0, t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        unsigned spins = 0;
        for (;;) {
            asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flags + threadIdx.x)
                         : "memory");
            if (v >= seq) break;
            __nanosleep(64);
            if ((++spins & 1023u) == 0u) {
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
                if (t - t0 > timeout_ns) {
                    if (status) {
                        atomicMax(status, seq);                                // which exchange
                        atomicOr(status + 1, 1ull << threadIdx.x);             // who is missing
                    }
                    break;
                }
            }
        }
    }
}

// ---- once-per-point pass: (optional) unit cube -> theta, then the per-point constants ----------
// One warp per point.  With U != NULL this is the fused prior transform: lane i < ndim evaluates
// ppf_i(u_i), theta is written out (the sampler stores it) and the constants are derived from
// exactly those values.  Used for rvl_transform_loglike (and on request, option "prepare"): the
// likelihood kernel otherwise derives the constants itself, per work item.
__device__ double ppf_eval(const rvl_prior_desc &pr, const double *tables, double q);

__global__ void __launch_bounds__(256) point_prepare_kernel(const rvl_model_desc *model,
                                                            const rvl_prior_desc *priors,
                                                            const double *tables, const double *U,
                                                            double *theta, double *consts,
                                                            int *flags, long long B,
                                                            int wstride, double tlo, double thi)
{
    const int lane = threadIdx.x & 31;
    // the model description is read many times per point: one cooperative copy to shared memory
    __shared__ __align__(16) unsigned char s_model[sizeof(rvl_model_desc)];
    {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(model);
        uint32_t *dst = reinterpret_cast<uint32_t *>(s_model);
        for (int i = threadIdx.x; i < (int)(sizeof(rvl_model_desc) / 4); i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    const long long pt = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (pt >= B) return;  // whole warps
    const rvl_model_desc &m = *reinterpret_cast<const rvl_model_desc *>(s_model);
    // the row is staged in shared memory with ONE coalesced read per warp: theta / U may live in
    // pinned host memory (zero-copy host-buffer calls), where scattered 8-byte reads are costly
    __shared__ double srow_all[8][RVL_MAX_DIM];
    double *srow = srow_all[threadIdx.x >> 5];
    double *row = theta + pt * m.ndim;
    if (U) {
        for (int i = lane; i < m.ndim; i += 32) {
            const double v = ppf_eval(priors[i], tables, U[pt * m.ndim + i]);
            srow[i] = v;
            row[i] = v;  // theta is an output of the fused call
        }
    } else {
        for (int i = lane; i < m.ndim; i += 32) srow[i] = row[i];
    }
    __syncwarp();
    const bool valid = point_setup(m, srow, consts + (size_t)pt * wstride, lane, tlo, thi);
    if (lane == 0) flags[pt] = valid ? 0 : 1;
}

// ---- prior transform: unit cube -> theta (evidence/ultranest/__init__.py:125-137) -----------
__device__ double ppf_eval(const rvl_prior_desc &pr, const double *tables, double q)
{
    const double p0 = pr.p[0], p1 = pr.p[1];
    switch (pr.kind) {
    case RVL_PRIOR_UNIFORM:  // priors.py:41-42
        return rvl::add(p0, rvl::mul(rvl::sub(p1, p0), q));
    case RVL_PRIOR_JEFFREYS:  // :62-63
        return rvl::mul(p0, pow(__ddiv_rn(p1, p0), q));
    case RVL_PRIOR_MODJEFFREYS:  // :82-83
        return rvl::sub(rvl::mul(p0, pow(rvl::add(1.0, __ddiv_rn(p1, p0)), q)), p0);
    case RVL_PRIOR_UNIFORMFREQ:  // :100-101   xmin / (1 - q*(xmax-xmin)/xmax)
        return __ddiv_rn(p0, rvl::sub(1.0, __ddiv_rn(rvl::mul(q, rvl::sub(p1, p0)), p1)));
    case RVL_PRIOR_TRUNCRAYLEIGH: {  // :249-252
        const double s2 = rvl::mul(p0, p0);
        const double A = rvl::sub(1.0, exp(-__ddiv_rn(rvl::mul(p1, p1), rvl::mul(2.0, s2))));
        return sqrt(rvl::mul(rvl::mul(-2.0, s2), log(rvl::sub(1.0, rvl::mul(q, A)))));
    }
    case RVL_PRIOR_NORMAL:  // scipy.stats.norm(loc, scale).ppf
        return rvl::add(rvl::mul(normcdfinv(q), p1), p0);
    case RVL_PRIOR_LOGNORMAL:  // scipy.stats.lognorm(s, loc, scale).ppf
        return rvl::add(rvl::mul(exp(rvl::mul(p0, normcdfinv(q))), pr.p[2]), p1);
    case RVL_PRIOR_TABLE: {
        // interp1d(cdf, x)(q): hi = clip(searchsorted(cdf, q, 'left'), 1, len-1)
        const double *cdf = tables + pr.table_offset;
        const double *x = cdf + pr.table_len;
        int lo = 0, hi = pr.table_len;
        while (lo < hi) {
            const int mid = lo + ((hi - lo) >> 1);
            if (__ldg(cdf + mid) < q) lo = mid + 1; else hi = mid;
        }
        int k = max(1, min(pr.table_len - 1, lo));
        const double x0 = __ldg(x + k - 1), x1 = __ldg(x + k);
        const double c0 = __ldg(cdf + k - 1), c1 = __ldg(cdf + k);
        if (p1 != 0.0) {  // p1 = 1: slopes dx/dq follow the knots -> cubic Hermite segment
            const double *mk = x + pr.table_len;
            const double m0 = __ldg(mk + k - 1), m1 = __ldg(mk + k);
            if (m0 > 0.0 && m1 > 0.0) {
                const double h = c1 - c0, t = (q - c0) / h, t2 = t * t, t3 = t2 * t;
                const double h00 = 2.0 * t3 - 3.0 * t2 + 1.0, h10 = t3 - 2.0 * t2 + t;
                const double h01 = -2.0 * t3 + 3.0 * t2, h11 = t3 - t2;
                return h00 * x0 + h10 * h * m0 + h01 * x1 + h11 * h * m1;
            }
        }
        const double slope = __ddiv_rn(rvl::sub(x1, x0), rvl::sub(c1, c0));
        const double y = rvl::add(rvl::mul(slope, rvl::sub(q, c0)), x0);
        return p0 != 0.0 ? exp10(y) : y;  // p0 = 1: Log10Normal, 10**interp (priors.py:144)
    }
    default:
        return nan("");
    }
}

__global__ void prior_transform_kernel(const rvl_prior_desc *priors, const double *tables,
                                       const double *U, double *Theta, long long total, int ndim)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int col = (int)(i % ndim);
    Theta[i] = ppf_eval(priors[col], tables, U[i]);
}

// ---- the reference's native FFI on the device (trueanomaly.h:4) --------------------------------
// One warp per 32 elements; a per-warp constant block in shared memory feeds solve_planet with
// nmot = 0, epoch = 0, M0 = M[i]: mean_anomaly gives 0*(t-0) + M[i] = M[i] exactly, and
// A = 1, Bs = 0, Ce = 0 / A = 0, Bs = 1 turn the RV term into cos(nu) / -sin(nu)... simpler and
// exact: replay the same loop on (sin E, cos E) and finish with atan2.
__global__ void trueanomaly_kernel(const double *M, int n, double ecc, double *nu, int itmax,
                                   double tol, int *caphit)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int ii = min(i, n - 1);  // whole warps stay converged; extra lanes duplicate the last
    const rvl::KTab kt = rvl::load_ktab();
    const double ec = ecc > 0.99 ? 0.99 : ecc;
    const double m = __ldg(M + ii);
    double E = m, s, c, d = 1e300;
    const bool slow = __any_sync(kFull, !(abs_hi(m) < kHiTrigMax) || !(ec >= -0.99));
    if (slow) { const double2 r = sincos_slow(E); s = r.x; c = r.y; }
    else rvl::sincos_fast(kt, E, s, c);
    int trip = 0;
    for (;;) {
        const bool pa = (fabs(d) > tol) && trip < itmax;
        if (!__any_sync(kFull, pa)) break;
        ++trip;
        double En;
        rvl::newton_step(E, s, c, m, ec, En);
        En = pa ? En : E;
        d = rvl::sub(En, E);
        E = En;
        const int h = abs_hi(d);
        if (__all_sync(kFull, h < kHiTiny)) rvl::advance_tiny(kt, d, s, c);
        else if (__all_sync(kFull, h < kHiSmall)) rvl::advance_small(kt, d, s, c);
        else if (slow || (trip > 2 && __any_sync(kFull, !(abs_hi(E) < kHiTrigMax)))) {
            const double2 r = sincos_slow(E); s = r.x; c = r.y;
        } else rvl::sincos_fast(kt, E, s, c);
    }
    const int cap = (fabs(d) > tol) ? 1 : 0;
    if (i < n) {
        // nu = 2 atan(sqrt((1+e)/(1-e)) tan(E/2))  ==  atan2(sqrt(1-e^2) sin E, cos E - e)
        const double root = sqrt(rvl::mul(rvl::sub(1.0, ec), rvl::add(1.0, ec)));
        nu[i] = atan2(rvl::mul(root, s), rvl::sub(c, ec));
        if (cap) atomicExch(caphit, 1);
    }
}

// ---- model velocity curves at caller times: kep_rv / modelk (:343-463) --------------------------
// One warp per work item = (point b, group g of 32*U consecutive times); lane l, slot u holds time
// g*32*U + u*32 + l, the lane <-> epoch map of the likelihood kernel, so every lane shares the
// eccentricity and the Newton trips stay warp-uniform.  The per-point constants come from
// point_prepare_kernel (d_consts, [B][wstride]); the item copies the planet blocks into the warp's
// shared block and runs the likelihood kernel's solve_planet on them, planet after planet in
// planet order, each solve adding its velocity to the lane's sum exactly as item_epochs does.  Each
// output element is computed by one lane with no reduction across items: a row's curve does not
// depend on the batch it came in.
//   Padding of a point's last group: a slot past T repeats the lane's slot 0 (the last time when
// that is past T too), so a lane whose second slot is padding ran two identical solves per planet
// and its cap hits are exactly twice the live ones.
struct CurveArgs {
    const rvl_model_desc *model;    // device copy
    const double *theta;            // [B][ndim]
    const double *consts;           // [B][wstride]
    const double *times;            // [T]
    double *out;                    // [B][T]
    uint32_t *invalid;              // [B] or NULL
    unsigned long long *cap_hits;   // or NULL
    long long nitems;               // B * G
    int T, G, K, ndim, wstride, itmax;
    uint32_t mask;
    double tol;
};

// RVL_CURVE_MINB: resident 256-thread blocks per SM asked of ptxas (1: no register cap, 116
// registers, no spills; 3: 80 registers with a few spilled bytes)
#ifndef RVL_CURVE_MINB
#define RVL_CURVE_MINB 1
#endif
template <int U>
__global__ void __launch_bounds__(256, RVL_CURVE_MINB) kepler_rv_kernel(const CurveArgs a)
{
    static_assert(U == 2, "cap-hit accounting of the padding assumes two slots per lane");
    __shared__ __align__(16) double s_pc[8][RVL_MAX_PLANETS * kPlanetStride];
    __shared__ __align__(16) unsigned char s_tab[kSinTabBytes];  // the likelihood kernel's table
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double *wc = s_pc[warp];
    const uint32_t a_wc = smem_u32(wc);
    {
        const uint4 *hi = reinterpret_cast<const uint4 *>(g_sintab_hi);
        const uint4 *lo = reinterpret_cast<const uint4 *>(g_sintab_lo);
        uint4 *dst = reinterpret_cast<uint4 *>(s_tab);
        constexpr int nhi = kSinTabHiBytes / 16, n = kSinTabBytes / 16;
        for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = i < nhi ? hi[i] : lo[i - nhi];
        __syncthreads();
    }
    const SmemSinTab tab{smem_u32(s_tab)};
    const rvl::KTab kt = rvl::load_ktab_pinned();
    const int K = a.K, T = a.T, G = a.G;
    // the launch-wide conditions of the lean Newton loop (item_epochs)
    const bool lean_ok = __double2hiint(a.tol) < rvl::kHiFinal && a.itmax >= 2;
    int caps = 0;
    const long long nw = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long it = (long long)blockIdx.x * (blockDim.x >> 5) + warp; it < a.nitems; it += nw) {
        const long long b = it / G;
        const int g = (int)(it - b * G);
        const double *row = a.theta + b * a.ndim;
        // validity of planet `lane`, the arithmetic of point_setup (:425-439)
        bool bad = false;
        if (lane < K) {
            const rvl_planet_desc &pl = a.model->planet[lane];
            if (pl.ecc_mode != RVL_ECC_DIRECT) {
                const double c = par_of(pl.e1, row), s = par_of(pl.e2, row);
                double e = rvl::add(rvl::mul(c, c), rvl::mul(s, s));
                if (pl.ecc_mode == RVL_ECC_ECOS_ESIN) e = sqrt(e);
                bad = e > 1.0;
            }
        }
        const uint32_t badm = __ballot_sync(kFull, bad);
        if (g == 0 && lane == 0 && a.invalid) a.invalid[b] = badm;
        const bool valid = (badm & a.mask) == 0u;

        __syncwarp();
        const double *src = a.consts + b * a.wstride;
        for (int i = lane; i < K * kPlanetStride; i += 32) wc[i] = __ldg(src + i);
        __syncwarp();

        const int j0 = g * 32 * U + lane;
        double t[U], rv[U];
        int it_l[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int j = j0 + u * 32;
            t[u] = T > 0 ? __ldg(a.times + (j < T ? j : (j0 < T ? j0 : T - 1))) : 0.0;
            rv[u] = valid ? 0.0 : __longlong_as_double(0x7ff8000000000000LL);  // NaN row
            it_l[u] = 0;
        }
        int cap_l = 0;
        if (valid) {
            for (int p = 0; p < K; ++p) {
                if (!((a.mask >> p) & 1u)) continue;
                const uint32_t pc = a_wc + (uint32_t)(p * kPlanetStride) * 8u;
                // the lean loop needs every |M| of the item inside the fast sin/cos range (the
                // prepare pass decided that for the data's epochs, not for these times)
                const double nmot = lds_f64(pc), M0 = lds_f64(pc + 8), ec = lds_f64(pc + 16),
                             epoch = lds_f64(pc + 48);
                bool in_range = ec >= -0.99;
#pragma unroll
                for (int u = 0; u < U; ++u)
                    in_range = in_range &&
                               fabs(rvl::mean_anomaly(nmot, t[u], epoch, M0)) < 0.99 * rvl::kTrigFastMax;
                const bool lean = lean_ok && __all_sync(kFull, in_range);
                solve_planet<0, U>(kt, tab, t, pc, a.tol, a.itmax, rv, it_l, cap_l, lean);
            }
        }
        double *o = a.out + b * (long long)T;
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (j0 + u * 32 < T) o[j0 + u * 32] = rv[u];
        caps += j0 + 32 < T ? cap_l : (j0 < T ? cap_l / 2 : 0);
    }
    if (a.cap_hits) {
        const unsigned n = __reduce_add_sync(kFull, (unsigned)caps);
        if (lane == 0 && n) atomicAdd(a.cap_hits, (unsigned long long)n);
    }
}

// ---- register-resident DFMA loop: the FP64 roofline denominator -------------------------------
template <int R>
__global__ void __launch_bounds__(1024) dfma_peak_kernel(double *out, int iters, double, double b)
{
    // R independent chains per thread, 32 warps per SM (grid of tools/ubench.cu)
    double x[R];
#pragma unroll
    for (int r = 0; r < R; ++r) x[r] = threadIdx.x + r;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
#pragma unroll
            // multiplier from the constant bank (uniform-register operand), addend in a
            // register: the operand form that reached the highest rate in tools/ubench.cu
            for (int r = 0; r < R; ++r) x[r] = __fma_rn(x[r], rvl::d_ktab[16], b);
        }
    }
    double s = 0.0;
#pragma unroll
    for (int r = 0; r < R; ++r) s += x[r];
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

thread_local std::string g_create_error;

}  // namespace

// =================================================================================================
// handle + C-ABI
// =================================================================================================
struct rvl_handle {
    int device = 0;
    int sm_count = 0, smem_optin = 0, clock_khz = 0;
    std::string err;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;  // kernel start / end, end of the gather wait

    // host copies of the staged inputs
    int N = 0, Npad = 0, n_inst = 0;
    std::vector<double> h_t, h_rv, h_err;
    double tlo = 0.0, thi = 0.0;  // min / max of h_t
    std::vector<int32_t> h_inst;
    std::vector<double> h_linpar[RVL_MAX_LINPAR];
    bool have_data = false, have_model = false, have_priors = false, cols_dirty = true;
    rvl_model_desc model{};

    // device
    double *d_cols = nullptr;
    uint8_t *d_inst = nullptr;
    int ncol = 0;
    rvl_model_desc *d_model = nullptr;
    rvl_prior_desc *d_priors = nullptr;
    double *d_tables = nullptr;
    int prior_ndim = 0;

    // per-call scratch (grown on demand)
    long long cap_B = 0, cap_flags = 0, cap_arrive = 0;
    size_t cap_partial = 0;
    int *d_arrive = nullptr;
    double *d_gconsts = nullptr;   // constants of the split points (written by the setup items)
    unsigned *d_ready = nullptr;   // their launch-stamped ready flags
    size_t cap_gconsts = 0;
    long long cap_ready = 0;
    unsigned seq = 0;
    unsigned smem_opted = 0;  // kernel builds whose shared-memory opt-in has been set on this device
    // pinned bounce buffers for PAGEABLE caller memory (numpy arrays): a pageable cudaMemcpy is a
    // synchronous, driver-staged copy (~185 us for 491 KB measured); one CPU memcpy into pinned
    // memory that the kernels then read / write in place costs ~30 us
    void *pin_in = nullptr, *pin_out = nullptr, *pin_out2 = nullptr;
    size_t cap_pin_in = 0, cap_pin_out = 0, cap_pin_out2 = 0;
    unsigned long long *d_trace = nullptr;  // option "trace": per-warp time stamps of the last launch
    int trace_rows = 0;
    double *d_theta = nullptr, *d_u = nullptr, *d_lnl = nullptr, *d_partial = nullptr;
    double *d_consts = nullptr;
    size_t cap_consts = 0;
    int *d_flags = nullptr;
    unsigned long long *d_counters = nullptr;  // 3
    unsigned int *d_work = nullptr;            // sm_count + 1 (queues, finished-block counter)
    // rvl_kepler_rv (host buffers): times, curves [B][T], invalid bits, cap-hit counter
    double *d_curve_t = nullptr, *d_curve = nullptr;
    size_t cap_curve_t = 0, cap_curve = 0;
    uint32_t *d_curve_inv = nullptr;
    long long cap_curve_inv = 0;
    unsigned long long *d_curve_caps = nullptr;
    int curve_blocks_per_sm = 0;  // resident blocks of kepler_rv_kernel (0: not asked yet)

    // options
    int opt_variant = 0, opt_slices = 0, opt_warps = 0, opt_timing = 0, opt_zero_copy = 1, opt_ilp = 0, opt_min_chunks = 8, opt_items_per_warp = 4;
    int opt_sched = 1;          // 1: graded phases (coarse -> fine items), 0: one uniform slice count
    int opt_phase_items = 200;  // items per split phase, in percent of the warps serving a queue
    int opt_max_split = 8;      // finest cut: sub-slices per point and resident range
                                // (B200, config 2 at ndraw = 4096: 127 us against 130 us for a
                                // uniform cut in 4 and 159 us with whole-point items first;
                                // every item costs ~430 warp-instructions on top of its epochs)
    int opt_trace = 0;
    int opt_setup_items = 1;    // 1: constants of split points from setup items inside the kernel
    int opt_prepare = 0;        // 1: per-point constants from the prepare pass even without a transform

    // bookkeeping
    uint64_t n_points = 0, n_solves = 0, launches = 0;
    double last_ms = 0.0, last_wait_ms = 0.0;
    bool timing_pending = false, wait_pending = false;

    // fused all-gather: bounded wait.  status[0] = seq of the exchange that timed out (0 = none),
    // status[1] = bit mask of the ranks that never signalled; mapped host memory, written by
    // wait_flags_kernel, read by the host after the stream has been synchronised
    unsigned long long *h_status = nullptr, *d_status = nullptr;
    long long opt_gather_timeout_ms = 10000;

    // rvl_create_multi: this handle only fans out to one child handle per device (rows of every
    // host-buffer call are split into contiguous blocks, one per child)
    std::vector<rvl_handle *> kids;
};

namespace {

int fail(rvl_t *h, int code, const std::string &msg)
{
    if (h) h->err = msg; else g_create_error = msg;
    return code;
}
#define CU(h, call)                                                                              \
    do {                                                                                         \
        cudaError_t e_ = (call);                                                                 \
        if (e_ != cudaSuccess)                                                                   \
            return fail(h, RVL_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e_));       \
    } while (0)

struct DevGuard {
    int prev = -1;
    explicit DevGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// build the epoch columns in HBM: t, vrad, svrad^2, [(t-tref)/365.25], [linpar...], inst ids
int upload_columns(rvl_t *h)
{
    const int N = h->N, Npad = h->Npad;
    const bool drift = h->have_model && h->model.drift_in_model;
    const int nlin = h->have_model ? h->model.n_linpar : 0;
    const int ncol = 3 + (drift ? 1 : 0) + nlin;
    for (int l = 0; l < nlin; ++l)
        if ((int)h->h_linpar[l].size() != N)
            return fail(h, RVL_ESTATE, "linear-parameter column " + std::to_string(l) + " not set");
    std::vector<double> cols((size_t)ncol * Npad);
    std::vector<uint8_t> ids((size_t)Npad);
    for (int j = 0; j < Npad; ++j) {
        const int k = j < N ? j : N - 1;  // padding duplicates the last epoch (masked in-kernel)
        cols[j] = h->h_t[k];
        cols[(size_t)Npad + j] = h->h_rv[k];
        cols[(size_t)2 * Npad + j] = h->h_err[k] * h->h_err[k];  // svrad**2 (:190-192)
        int c = 3;
        if (drift) cols[(size_t)(c++) * Npad + j] = (h->h_t[k] - h->model.tref) / 365.25;  // :270
        for (int l = 0; l < nlin; ++l) cols[(size_t)(c++) * Npad + j] = h->h_linpar[l][k];
        ids[j] = (uint8_t)h->h_inst[k];
    }
    if (h->d_cols) cudaFree(h->d_cols);
    if (h->d_inst) cudaFree(h->d_inst);
    h->d_cols = nullptr; h->d_inst = nullptr;
    CU(h, cudaMalloc(&h->d_cols, cols.size() * sizeof(double)));
    CU(h, cudaMalloc(&h->d_inst, ids.size()));
    CU(h, cudaMemcpy(h->d_cols, cols.data(), cols.size() * sizeof(double), cudaMemcpyHostToDevice));
    CU(h, cudaMemcpy(h->d_inst, ids.data(), ids.size(), cudaMemcpyHostToDevice));
    h->ncol = ncol;
    h->cols_dirty = false;
    return RVL_OK;
}

// device staging for the host-buffer entry points
int ensure_io(rvl_t *h, long long B)
{
    if (B <= h->cap_B) return RVL_OK;
    const long long cap = std::max<long long>(B, 1024);
    cudaFree(h->d_theta); cudaFree(h->d_u); cudaFree(h->d_lnl);
    h->d_theta = h->d_u = h->d_lnl = nullptr;
    h->cap_B = 0;
    const size_t row = (size_t)std::max(1, std::max(h->model.ndim, h->prior_ndim));
    CU(h, cudaMalloc(&h->d_theta, (size_t)cap * row * sizeof(double)));
    CU(h, cudaMalloc(&h->d_u, (size_t)cap * row * sizeof(double)));
    CU(h, cudaMalloc(&h->d_lnl, (size_t)cap * sizeof(double)));
    h->cap_B = cap;
    return RVL_OK;
}

// partial sums and arrival counters of the split points, invalid-point flags and prepared
// per-point constants
int ensure_partial(rvl_t *h, long long B, size_t partial_doubles, long long n_split, bool prepare,
                   int wstride)
{
    if (prepare && B > h->cap_flags) {
        cudaFree(h->d_flags);
        h->d_flags = nullptr; h->cap_flags = 0;
        CU(h, cudaMalloc(&h->d_flags, (size_t)B * sizeof(int)));
        h->cap_flags = B;
    }
    if (partial_doubles > h->cap_partial) {
        cudaFree(h->d_partial);
        h->d_partial = nullptr; h->cap_partial = 0;
        CU(h, cudaMalloc(&h->d_partial, partial_doubles * sizeof(double)));
        h->cap_partial = partial_doubles;
    }
    if (n_split > h->cap_arrive) {
        cudaFree(h->d_arrive);
        h->d_arrive = nullptr; h->cap_arrive = 0;
        CU(h, cudaMalloc(&h->d_arrive, (size_t)n_split * sizeof(int)));
        // zero once: the kernel leaves every counter at zero again (last arriver resets it)
        CU(h, cudaMemset(h->d_arrive, 0, (size_t)n_split * sizeof(int)));
        h->cap_arrive = n_split;
    }
    const size_t needc = (size_t)B * wstride;
    if (prepare && needc > h->cap_consts) {
        cudaFree(h->d_consts);
        h->d_consts = nullptr; h->cap_consts = 0;
        CU(h, cudaMalloc(&h->d_consts, needc * sizeof(double)));
        h->cap_consts = needc;
    }
    return RVL_OK;
}

struct Plan {
    int Sm, cpm, W, U, grid, wstride, wblock;
    size_t smem;
    int nph;
    Phase ph[kMaxPhases];
    unsigned nitems;
    long long ptS0, n_split;
    size_t partial_doubles;
};

size_t smem_need(int ncol, int ne, int W, int wstride)
{
    return 128 + kModelBytes + kSinTabBytes + (((size_t)ncol * ne * 8 + ne + 127) / 128) * 128 +
           (size_t)W * wstride * 8;
}

// Work decomposition.  The epoch axis is cut into Sm resident ranges (the fewest that fit in
// shared memory; block b holds range b % Sm and serves that range's queue).  Within a range a
// point is one item, or -- for the points at the END of the batch -- 2, 4, ... sub-slices, each
// phase holding about one item per warp: the work handed out last is the finest, so all warps of
// the chip run dry together (a batch of ndraw = 4096 points is ONE point per warp otherwise).
struct PlanIn {
    int Ctot, ncol, wstride, wblock, U, W, sm_count, smem_optin;
    int sched, slices, items_per_warp, min_chunks, phase_items, max_split;
};

const char *plan_core(const PlanIn &in, long long B, Plan &pl)
{
    const PlanIn *h = &in;
    const int Ctot = in.Ctot, wstride = in.wstride, U = in.U, W = in.W;
    int Sm = 1, cpm = 0;
    auto cpm_of = [&](int s) { return ((Ctot + s - 1) / s + U - 1) / U * U; };  // whole U-chunk trips
    auto fits = [&](int s) {
        return smem_need(h->ncol, cpm_of(s) * 32, W, in.wblock) <= (size_t)h->smem_optin;
    };
    while (Sm < Ctot && Sm < h->sm_count && !fits(Sm)) ++Sm;
    if (!fits(Sm)) return "epoch range does not fit in shared memory";
    cpm = cpm_of(Sm);
    Sm = (Ctot + cpm - 1) / cpm;  // drop empty trailing ranges
    pl.Sm = Sm; pl.cpm = cpm; pl.W = W; pl.U = U; pl.wstride = wstride;
    pl.grid = std::max(1, h->sm_count / Sm) * Sm;
    pl.smem = smem_need(h->ncol, cpm * 32, W, in.wblock);
    pl.wblock = in.wblock;

    // sub-slice counts available within one resident range: S -> cps = ceil(cpm / S) in whole trips
    auto cps_of = [&](int S) { return ((cpm + S - 1) / S + U - 1) / U * U; };
    auto norm = [&](int S) { const int c = cps_of(S); return (cpm + c - 1) / c; };
    const long long warps_q = (long long)(pl.grid / Sm) * W;  // warps serving one queue
    pl.nph = 0;
    pl.ptS0 = B; pl.n_split = 0; pl.partial_doubles = 0;
    struct Seg { int S; long long n; };
    Seg seg[kMaxPhases];
    int nseg = 0;
    long long left = B;
    if (h->slices > 0 || !h->sched) {
        // one uniform slice count for every point
        long long want;
        if (h->slices > 0) want = (h->slices + Sm - 1) / Sm;
        else {
            want = ((long long)h->items_per_warp * warps_q + B - 1) / std::max<long long>(B, 1);
            want = std::min<long long>(want, std::max(1, cpm / h->min_chunks));
        }
        const int S = norm((int)std::max<long long>(1, std::min<long long>(want, cpm)));
        seg[nseg++] = Seg{S, B};
        left = 0;
    } else {
        // graded: finest phase last; built from the end of the batch backwards
        int Smax = norm(std::max(1, std::min(h->max_split, cpm)));
        const long long per_phase = std::max<long long>(1, warps_q * h->phase_items / 100);
        Seg rev[kMaxPhases];
        int nrev = 0;
        for (int S = Smax; S > 1 && left > 0 && nrev < kMaxPhases - 1; S = norm(S / 2)) {
            const long long n = std::min(left, std::max<long long>(1, per_phase / S));
            if (nrev > 0 && rev[nrev - 1].S == S) rev[nrev - 1].n += n;
            else rev[nrev++] = Seg{S, n};
            left -= n;
            if (norm(S / 2) >= S) break;
        }
        if (left > 0) rev[nrev++] = Seg{1, left};
        left = 0;
        for (int i = nrev - 1; i >= 0; --i) seg[nseg++] = rev[i];
    }
    unsigned long long idx = 0;
    long long pt = 0;
    size_t part = 0;
    for (int i = 0; i < nseg; ++i) {
        Phase &p = pl.ph[pl.nph++];
        p.idx0 = (unsigned)idx; p.S = seg[i].S; p.cps = cps_of(seg[i].S);
        p.shift = -1;
        for (int b = 0; b < 31; ++b)
            if ((1 << b) == seg[i].S) p.shift = b;
        p.pt0 = pt; p.part0 = (long long)part;
        const int Stot = Sm * seg[i].S;
        if (Stot > 1) {
            if (pl.n_split == 0) pl.ptS0 = pt;
            pl.n_split += seg[i].n;
            part += (size_t)seg[i].n * Stot * 2;
        } else if (pl.n_split > 0) {
            return "internal: whole-point phase after a split phase";
        }
        idx += (unsigned long long)seg[i].n * seg[i].S;
        pt += seg[i].n;
    }
    if (idx > 0xfffffff0ULL) return "batch too large for one call";
    pl.nitems = (unsigned)idx;
    pl.partial_doubles = part;
    return nullptr;
}

// doubles of per-point constants (point_setup's layout; +1: the lean flag)
int consts_stride(const rvl_model_desc &m)
{
    return (m.n_planets * kPlanetStride + 2 * m.n_inst + 4 + m.n_linpar + 1 + 1) & ~1;
}

int make_plan(rvl_t *h, long long B, Plan &pl)
{
    const rvl_model_desc &m = h->model;
    PlanIn in{};
    in.Ctot = (h->N + 31) / 32;  // (the columns themselves are padded further: see rvl_set_data)
    in.ncol = h->ncol;
    in.wstride = consts_stride(m);
    in.wblock = in.wstride + ((m.ndim + 1) & ~1);
    // epochs per lane in flight: 4 (512 threads, 128 registers) when every warp has a long queue of
    // whole points AND a point is long enough to amortise its setup over the 16 warps per SM left --
    // the per-pass control instructions are then shared by four solves; 2 (896 threads, 72 registers)
    // for sampler-sized batches and for short or planet-poor points, where the drain and the
    // per-point work matter more.  Measured, B200, final build, U = 2 against U = 4: config 3
    // (N 5000, K 4) at 524288 theta U = 4 wins; the same at N 2500 / 1250: a tie; config 2 (K 2,
    // drift) at 1048576 theta 19.8 vs 23.8 ms, at N 4000 18.9 vs 19.7; config 5 (N 10000, K 3) at 131072
    // theta 33.5 vs 33.9 ms; config 1 (N 200, K 1) 2.9 vs 3.8 ms; config 2 at 4096 theta 0.110 vs 0.125.
    int ilp = h->opt_ilp;
    if (ilp == 0)
        ilp = (B >= (long long)h->sm_count * 16 * 16 && m.n_planets >= 4 &&
               (long long)h->N * m.n_planets >= 16384) ? 4 : 2;
    in.U = h->opt_variant == 0 ? ilp : 1;
    const int w_default = in.U == 1 ? 32 : in.U == 2 ? 28 : in.U == 3 ? 20 : 16;
    const int w_max = in.U <= 2 ? 32 : in.U == 3 ? 20 : 16;
    in.W = std::max(1, std::min(w_max, h->opt_warps > 0 ? h->opt_warps : w_default));
    in.sm_count = h->sm_count; in.smem_optin = h->smem_optin;
    in.sched = h->opt_sched; in.slices = h->opt_slices; in.items_per_warp = h->opt_items_per_warp;
    in.min_chunks = h->opt_min_chunks; in.phase_items = h->opt_phase_items;
    in.max_split = h->opt_max_split;
    const char *e = plan_core(in, B, pl);
    return e ? fail(h, RVL_EINVAL, e) : RVL_OK;
}

template <int V, int U, int T>
int launch_lnl_v(rvl_t *h, const KArgs &a, const Plan &pl, cudaStream_t st)
{
    // opt in to the large dynamic shared memory once per kernel build and handle (device), not on
    // every launch: the attribute call is a driver round trip on the host-latency path
    const unsigned bit = V ? (1u << 31) : (1u << ((U - 1) * 8 + T / 128 - 1));
    if (!(h->smem_opted & bit)) {
        CU(h, cudaFuncSetAttribute(rv_lnl_kernel<V, U, T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   h->smem_optin));
        h->smem_opted |= bit;
    }
    rv_lnl_kernel<V, U, T><<<pl.grid, std::min(pl.W * 32, T), pl.smem, st>>>(a);
    CU(h, cudaGetLastError());
    return RVL_OK;
}

// enqueue: [prepare pass], zero work counters, likelihood kernel, [combine].  All pointers are
// device pointers.  dU != NULL: fused prior transform -- theta is WRITTEN to dTheta by the prepare
// pass and the likelihood is evaluated on exactly those values.
int enqueue_loglike(rvl_t *h, const double *dU, double *dTheta, long long B, double *dlnL,
                    cudaStream_t st, bool timed, const PeerOut *peers = nullptr,
                    bool force_prepare = false)
{
    if (!h->have_data || !h->have_model) return fail(h, RVL_ESTATE, "set data and model first");
    if (dU && !h->have_priors) return fail(h, RVL_ESTATE, "set priors first");
    if (dU && h->prior_ndim != h->model.ndim) return fail(h, RVL_ESTATE, "priors and model disagree on ndim");
    if (h->cols_dirty) { int rc = upload_columns(h); if (rc) return rc; }
    if (B <= 0) return RVL_OK;
    if (B > 0xfffffff0LL) return fail(h, RVL_EINVAL, "batch too large for one call (max ~4.29e9)");
    Plan pl;
    int rc = make_plan(h, B, pl);
    if (rc) return rc;
    const bool prepare = dU != nullptr || h->opt_prepare || force_prepare;
    rc = ensure_partial(h, B, pl.partial_doubles, pl.n_split, prepare, pl.wstride);
    if (rc) return rc;
    if (prepare) {
        const int wpb = 8;  // warps (= points) per block
        point_prepare_kernel<<<(unsigned)((B + wpb - 1) / wpb), wpb * 32, 0, st>>>(
            h->d_model, h->d_priors, h->d_tables, dU, dTheta, h->d_consts, h->d_flags, B,
            pl.wstride, h->tlo, h->thi);
        CU(h, cudaGetLastError());
        ++h->launches;
    }
    const bool setup_items = !prepare && h->opt_setup_items && pl.Sm == 1 && pl.n_split > 0 &&
                             (unsigned long long)pl.nitems + (unsigned long long)pl.n_split < 0xfffffff0ULL;
    if (setup_items) {
        const size_t need = (size_t)pl.n_split * pl.wstride;
        if (need > h->cap_gconsts) {
            cudaFree(h->d_gconsts);
            h->d_gconsts = nullptr; h->cap_gconsts = 0;
            CU(h, cudaMalloc(&h->d_gconsts, need * sizeof(double)));
            h->cap_gconsts = need;
        }
        if (pl.n_split > h->cap_ready || h->seq >= 0x7ffffff0u) {
            cudaFree(h->d_ready);
            h->d_ready = nullptr; h->cap_ready = 0;
            const long long cap = std::max(pl.n_split, h->cap_ready);
            CU(h, cudaMalloc(&h->d_ready, (size_t)cap * sizeof(unsigned)));
            CU(h, cudaMemset(h->d_ready, 0, (size_t)cap * sizeof(unsigned)));  // stamp 0 = never
            h->cap_ready = cap;
            h->seq = 0;
        }
        ++h->seq;
    }
    KArgs a{};
    a.n_setup = setup_items ? (unsigned)pl.n_split : 0u;
    a.seq = h->seq; a.gconsts = h->d_gconsts; a.ready = h->d_ready;
    a.model = h->d_model; a.cols = h->d_cols; a.inst = h->d_inst; a.theta = dTheta; a.lnl = dlnL;
    a.partial = h->d_partial; a.arrive = h->d_arrive; a.flags = h->d_flags;
    a.counters = h->d_counters; a.work = h->d_work;
    a.consts = prepare ? h->d_consts : nullptr;
    a.tlo = h->tlo; a.thi = h->thi;
    a.B = B; a.ptS0 = pl.ptS0; a.cte = -0.5 * h->N * log(2 * M_PI); a.N = h->N; a.Npad = h->Npad;
    a.ncol = h->ncol; a.Sm = pl.Sm; a.cpm = pl.cpm; a.nitems = pl.nitems; a.nph = pl.nph;
    a.wstride = pl.wstride; a.wblock = pl.wblock;
    for (int i = 0; i < pl.nph; ++i) a.ph[i] = pl.ph[i];
    if (peers) a.peers = *peers;
    if (h->opt_trace) {
        if (!h->d_trace) CU(h, cudaMalloc(&h->d_trace, (size_t)h->sm_count * 32 * 4 * sizeof(unsigned long long)));
        a.trace = h->d_trace;
        h->trace_rows = pl.grid * pl.W;
    }
    if (timed) CU(h, cudaEventRecord(h->ev0, st));
    if (h->opt_variant == 1) rc = launch_lnl_v<1, 1, 1024>(h, a, pl, st);
    else if (pl.U == 2 && pl.W <= 16) rc = launch_lnl_v<0, 2, 512>(h, a, pl, st);
    else if (pl.U == 2 && pl.W <= 20) rc = launch_lnl_v<0, 2, 640>(h, a, pl, st);
    else if (pl.U == 2 && pl.W <= 24) rc = launch_lnl_v<0, 2, 768>(h, a, pl, st);
    else if (pl.U == 2 && pl.W <= 28) rc = launch_lnl_v<0, 2, 896>(h, a, pl, st);
    else if (pl.U == 2) rc = launch_lnl_v<0, 2, 1024>(h, a, pl, st);
    else if (pl.U == 3) rc = launch_lnl_v<0, 3, 640>(h, a, pl, st);
    else if (pl.U == 4) rc = launch_lnl_v<0, 4, 512>(h, a, pl, st);
    else rc = launch_lnl_v<0, 1, 1024>(h, a, pl, st);
    if (rc) return rc;
    if (timed) { CU(h, cudaEventRecord(h->ev1, st)); h->timing_pending = true; }
    ++h->launches;
    h->n_points += (uint64_t)B;
    h->n_solves += (uint64_t)B * (uint64_t)h->N * (uint64_t)h->model.n_planets;
    return RVL_OK;
}

int enqueue_transform(rvl_t *h, const double *dU, long long B, double *dTheta, cudaStream_t st)
{
    if (!h->have_priors) return fail(h, RVL_ESTATE, "set priors first");
    if (B <= 0) return RVL_OK;
    const long long total = B * h->prior_ndim;
    const int tb = 256;
    prior_transform_kernel<<<(unsigned)((total + tb - 1) / tb), tb, 0, st>>>(
        h->d_priors, h->d_tables, dU, dTheta, total, h->prior_ndim);
    CU(h, cudaGetLastError());
    ++h->launches;
    return RVL_OK;
}

// Model velocity curves, device pointers: the prepare pass derives every point's constants into
// d_consts, then kepler_rv_kernel evaluates them at the caller's times.  rvl_counters untouched.
int enqueue_kepler_rv(rvl_t *h, const double *dTheta, long long B, const double *dTimes, int T,
                      uint32_t mask, double *dOut, uint32_t *dInvalid, unsigned long long *dCaps,
                      cudaStream_t st)
{
    if (!h->have_model) return fail(h, RVL_ESTATE, "set the model first");
    const rvl_model_desc &m = h->model;
    if (m.n_planets < 32 && (mask >> m.n_planets) != 0u)
        return fail(h, RVL_EINVAL, "planet_mask names a planet the model does not have");
    if (B <= 0) return RVL_OK;
    const int wstride = consts_stride(m);
    int rc = ensure_partial(h, B, 0, 0, /*prepare=*/true, wstride);
    if (rc) return rc;
    const int wpb = 8;  // warps (= points) per block
    point_prepare_kernel<<<(unsigned)((B + wpb - 1) / wpb), wpb * 32, 0, st>>>(
        h->d_model, nullptr, nullptr, nullptr, const_cast<double *>(dTheta), h->d_consts, h->d_flags,
        B, wstride, h->tlo, h->thi);
    CU(h, cudaGetLastError());
    ++h->launches;
    constexpr int U = 2, kThreads = 256;
    if (!h->curve_blocks_per_sm) {
        int n = 0;
        CU(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kepler_rv_kernel<U>, kThreads, 0));
        h->curve_blocks_per_sm = std::max(1, n);
    }
    CurveArgs a{};
    a.model = h->d_model; a.theta = dTheta; a.consts = h->d_consts; a.times = dTimes; a.out = dOut;
    a.invalid = dInvalid; a.cap_hits = dCaps;
    // T == 0: one item per point that only writes the invalid bits
    a.T = T; a.G = T > 0 ? (T + 32 * U - 1) / (32 * U) : 1; a.mask = T > 0 ? mask : 0u;
    a.K = m.n_planets; a.ndim = m.ndim; a.wstride = wstride; a.itmax = m.itmax; a.tol = m.tol;
    a.nitems = B * (long long)a.G;
    const long long wpb2 = kThreads / 32;
    const long long blocks = std::min<long long>((a.nitems + wpb2 - 1) / wpb2,
                                                 (long long)h->sm_count * h->curve_blocks_per_sm);
    kepler_rv_kernel<U><<<(unsigned)blocks, kThreads, 0, st>>>(a);
    CU(h, cudaGetLastError());
    ++h->launches;
    return RVL_OK;
}

// Device alias of a pinned (page-locked, mapped) host buffer, or NULL for pageable memory.
// The kernels then read theta / write lnL in place over PCIe: no staging copy, no extra launch.
void *pinned_alias(rvl_t *h, const void *p)
{
    if (!h->opt_zero_copy || !p) return nullptr;
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) == cudaSuccess && at.type == cudaMemoryTypeHost)
        return at.devicePointer;
    cudaGetLastError();  // pageable memory: clear the error some driver versions record
    return nullptr;
}

// Pageable buffers up to this size go through the pinned bounce buffers; larger ones through the
// driver's own chunked staging (cudaMemcpyAsync), which overlaps its chunks.
constexpr size_t kBounceMax = (size_t)32 << 20;

bool is_pinned(const void *p)
{
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) == cudaSuccess && at.type == cudaMemoryTypeHost) return true;
    cudaGetLastError();
    return false;
}

int ensure_pin(rvl_t *h, void **buf, size_t *cap, size_t need)
{
    if (need <= *cap) return RVL_OK;
    if (*buf) cudaFreeHost(*buf);
    *buf = nullptr; *cap = 0;
    const size_t sz = std::max(need, (size_t)1 << 20);
    CU(h, cudaHostAlloc(buf, sz, cudaHostAllocDefault));
    *cap = sz;
    return RVL_OK;
}

// Input side: returns in *src a PINNED host pointer holding the caller's data (the caller's own
// buffer if it is pinned, else the bounce buffer after one memcpy), or the caller's pointer
// unchanged with *pinned = false (too large / bouncing disabled).
int bounce_in(rvl_t *h, const void *user, size_t nb, const void **src, bool *pinned)
{
    *src = user;
    *pinned = is_pinned(user);
    if (*pinned || !h->opt_zero_copy || nb == 0 || nb > kBounceMax) return RVL_OK;
    int rc = ensure_pin(h, &h->pin_in, &h->cap_pin_in, nb);
    if (rc) return rc;
    memcpy(h->pin_in, user, nb);
    *src = h->pin_in;
    *pinned = true;
    return RVL_OK;
}

// Output side: a pinned host pointer the kernels can write in place (the caller's buffer, or a
// bounce buffer that is copied out after the stream has been synchronised), or NULL.
int bounce_out(rvl_t *h, void *user, size_t nb, void **buf, size_t *cap, void **dst, bool *copy_back)
{
    *copy_back = false;
    *dst = nullptr;
    if (!h->opt_zero_copy || !user || nb == 0) return RVL_OK;
    if (is_pinned(user)) { *dst = user; return RVL_OK; }
    if (nb > kBounceMax) return RVL_OK;
    int rc = ensure_pin(h, buf, cap, nb);
    if (rc) return rc;
    *dst = *buf;
    *copy_back = true;
    return RVL_OK;
}

int finish_timing(rvl_t *h)
{
    if (h->timing_pending) {
        float ms = 0.f;
        CU(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
        h->last_ms = ms;
        h->timing_pending = false;
        if (h->wait_pending) {  // time between the end of the kernel and the last peer's signal
            CU(h, cudaEventElapsedTime(&ms, h->ev1, h->ev2));
            h->last_wait_ms = ms;
            h->wait_pending = false;
        }
    }
    return RVL_OK;
}

// ---- host-buffer calls in two halves: enqueue everything on the handle's stream, then wait and
// copy the bounce buffers back.  A multi-device handle runs the first half on every child before
// the second half of any, so the devices work concurrently under ONE host thread.
struct HostCall {
    double *lnL = nullptr, *Theta = nullptr;  // caller buffers that still need a copy-back
    void *lnl_host = nullptr, *th_host = nullptr;
    size_t lnl_bytes = 0, th_bytes = 0;
};

int hostcall_end(rvl_t *h, HostCall &hc)
{
    CU(h, cudaStreamSynchronize(h->stream));
    if (hc.Theta) memcpy(hc.Theta, hc.th_host, hc.th_bytes);
    if (hc.lnL) memcpy(hc.lnL, hc.lnl_host, hc.lnl_bytes);
    return finish_timing(h);
}

// theta (host) -> lnL (host), everything enqueued on h->stream; no synchronisation.
// A pinned theta is read in place (zero-copy): the likelihood kernel reads every row ONCE, with
// one coalesced warp read (the setup item of a split point, or the point's only item), so the
// PCIe transfer overlaps the arithmetic instead of preceding it.  When the epoch axis needs
// several resident ranges every range would read the row: theta is then staged by a DMA copy.
// Pageable buffers (numpy arrays) pass through pinned bounce buffers.  lnL is written in place.
int loglike_begin(rvl_t *h, const double *Theta, long long B, double *lnL, HostCall &hc,
                  const PeerOut *peers = nullptr, double *dev_out = nullptr)
{
    int rc = ensure_io(h, B);
    if (rc) return rc;
    const size_t nb = (size_t)B * h->model.ndim * sizeof(double);
    Plan pl;
    if (h->cols_dirty) { rc = upload_columns(h); if (rc) return rc; }
    rc = make_plan(h, B, pl);
    if (rc) return rc;
    const bool once = pl.Sm == 1 && (h->opt_setup_items || pl.n_split == 0) && !h->opt_prepare;
    const void *src;
    bool src_pinned;
    rc = bounce_in(h, Theta, nb, &src, &src_pinned);
    if (rc) return rc;
    double *th_dev = (src_pinned && (h->opt_zero_copy > 1 || (h->opt_zero_copy == 1 && once)))
                         ? (double *)pinned_alias(h, src) : nullptr;
    const bool via_prepare = th_dev != nullptr && !once;
    if (!th_dev) {
        th_dev = h->d_theta;
        if (nb) CU(h, cudaMemcpyAsync(h->d_theta, src, nb, cudaMemcpyHostToDevice, h->stream));
    }
    if (dev_out)  // the caller collects the result from device memory itself (gather variant)
        return enqueue_loglike(h, nullptr, th_dev, B, dev_out, h->stream, h->opt_timing != 0, peers,
                               via_prepare);
    void *out_host;
    bool out_copy;
    rc = bounce_out(h, lnL, (size_t)B * sizeof(double), &h->pin_out, &h->cap_pin_out, &out_host, &out_copy);
    if (rc) return rc;
    double *out_dev = out_host ? (double *)pinned_alias(h, out_host) : nullptr;
    rc = enqueue_loglike(h, nullptr, th_dev, B, out_dev ? out_dev : h->d_lnl, h->stream,
                         h->opt_timing != 0, peers, via_prepare);
    if (rc) return rc;
    if (!out_dev)
        CU(h, cudaMemcpyAsync(lnL, h->d_lnl, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (out_dev && out_copy) { hc.lnL = lnL; hc.lnl_host = out_host; hc.lnl_bytes = (size_t)B * sizeof(double); }
    return RVL_OK;
}

int transform_begin(rvl_t *h, const double *U, long long B, double *Theta, HostCall &hc)
{
    int rc = ensure_io(h, B);
    if (rc) return rc;
    const size_t nb = (size_t)B * h->prior_ndim * sizeof(double);
    // elementwise and HBM-bound on the device, PCIe-bound here: U is read and theta written in
    // place through pinned memory (the caller's, or the bounce buffers for pageable arrays)
    const void *src;
    bool src_pinned;
    rc = bounce_in(h, U, nb, &src, &src_pinned);
    if (rc) return rc;
    const double *u_dev = src_pinned ? (const double *)pinned_alias(h, src) : nullptr;
    if (!u_dev) {
        CU(h, cudaMemcpyAsync(h->d_u, src, nb, cudaMemcpyHostToDevice, h->stream));
        u_dev = h->d_u;
    }
    void *out_host;
    bool out_copy;
    rc = bounce_out(h, Theta, nb, &h->pin_out, &h->cap_pin_out, &out_host, &out_copy);
    if (rc) return rc;
    double *th_dev = out_host ? (double *)pinned_alias(h, out_host) : nullptr;
    rc = enqueue_transform(h, u_dev, B, th_dev ? th_dev : h->d_theta, h->stream);
    if (rc) return rc;
    if (!th_dev)
        CU(h, cudaMemcpyAsync(Theta, h->d_theta, nb, cudaMemcpyDeviceToHost, h->stream));
    if (th_dev && out_copy) { hc.Theta = Theta; hc.th_host = out_host; hc.th_bytes = nb; }
    return RVL_OK;
}

int transform_loglike_begin(rvl_t *h, const double *U, long long B, double *Theta, double *lnL,
                            HostCall &hc)
{
    int rc = ensure_io(h, B);
    if (rc) return rc;
    const size_t nb = (size_t)B * h->prior_ndim * sizeof(double);
    // pinned buffers (the caller's, or the bounce buffers for pageable arrays) are read / written
    // in place by the prepare pass and the kernels
    const void *src;
    bool src_pinned;
    rc = bounce_in(h, U, nb, &src, &src_pinned);
    if (rc) return rc;
    const double *u_dev = src_pinned ? (const double *)pinned_alias(h, src) : nullptr;
    if (!u_dev) {
        CU(h, cudaMemcpyAsync(h->d_u, src, nb, cudaMemcpyHostToDevice, h->stream));
        u_dev = h->d_u;
    }
    void *th_host = nullptr, *out_host = nullptr;
    bool th_copy = false, out_copy = false;
    if (Theta) {
        rc = bounce_out(h, Theta, nb, &h->pin_out2, &h->cap_pin_out2, &th_host, &th_copy);
        if (rc) return rc;
    }
    rc = bounce_out(h, lnL, (size_t)B * sizeof(double), &h->pin_out, &h->cap_pin_out, &out_host, &out_copy);
    if (rc) return rc;
    double *th_dev = th_host ? (double *)pinned_alias(h, th_host) : nullptr;
    double *out_dev = out_host ? (double *)pinned_alias(h, out_host) : nullptr;
    rc = enqueue_loglike(h, u_dev, th_dev ? th_dev : h->d_theta, B, out_dev ? out_dev : h->d_lnl,
                         h->stream, h->opt_timing != 0);
    if (rc) return rc;
    if (Theta && !th_dev)
        CU(h, cudaMemcpyAsync(Theta, h->d_theta, nb, cudaMemcpyDeviceToHost, h->stream));
    if (!out_dev)
        CU(h, cudaMemcpyAsync(lnL, h->d_lnl, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (th_dev && th_copy) { hc.Theta = Theta; hc.th_host = th_host; hc.th_bytes = nb; }
    if (out_dev && out_copy) { hc.lnL = lnL; hc.lnl_host = out_host; hc.lnl_bytes = (size_t)B * sizeof(double); }
    return RVL_OK;
}

// ---- multi-device handle (rvl_create_multi): contiguous row blocks, one per child ----------------
// mode 0: Theta -> lnL; 1: U -> Theta; 2: U -> (Theta), lnL.  Child i owns rows
// [i*ceil(B/n), min(B, (i+1)*ceil(B/n))): the partition of SURVEY.md 8(e).  Every child reads its
// block of the caller's (pinned) buffer in place and writes its block of the result in place, so
// the "gather" of the single-process path is the kernels' own stores.
int multi_fail(rvl_t *h, rvl_t *kid, int rc)
{
    h->err = "device " + std::to_string(kid->device) + ": " + kid->err;
    return rc;
}

int multi_rows(rvl_t *h, const double *in, const double *U, double *Theta, double *lnL, long long B,
               int mode)
{
    if (B == 0) return RVL_OK;
    const int n = (int)h->kids.size();
    const long long per = (B + n - 1) / n;
    std::vector<HostCall> hc((size_t)n);
    std::vector<char> live((size_t)n, 0);
    int rc = RVL_OK;
    for (int i = 0; i < n && rc == RVL_OK; ++i) {
        const long long lo = std::min(B, (long long)i * per), hi = std::min(B, lo + per);
        if (hi <= lo) continue;
        rvl_t *k = h->kids[i];
        if (mode != 1 && (!k->have_data || !k->have_model)) return fail(h, RVL_ESTATE, "set data and model first");
        if (mode != 0 && !k->have_priors) return fail(h, RVL_ESTATE, "set priors first");
        if (mode == 2 && k->prior_ndim != k->model.ndim) return fail(h, RVL_ESTATE, "priors and model disagree on ndim");
        const size_t nd = (size_t)(mode == 0 ? k->model.ndim : k->prior_ndim);
        DevGuard g(k->device);
        if (mode == 0) rc = loglike_begin(k, in + (size_t)lo * nd, hi - lo, lnL + lo, hc[i]);
        else if (mode == 1) rc = transform_begin(k, U + (size_t)lo * nd, hi - lo, Theta + (size_t)lo * nd, hc[i]);
        else rc = transform_loglike_begin(k, U + (size_t)lo * nd, hi - lo,
                                          Theta ? Theta + (size_t)lo * nd : nullptr, lnL + lo, hc[i]);
        if (rc) rc = multi_fail(h, k, rc); else live[i] = 1;
    }
    for (int i = 0; i < n; ++i) {  // always drain what was enqueued, even after a failure
        if (!live[i]) continue;
        rvl_t *k = h->kids[i];
        DevGuard g(k->device);
        const int r2 = hostcall_end(k, hc[i]);
        if (r2 && rc == RVL_OK) rc = multi_fail(h, k, r2);
    }
    return rc;
}

// status of the bounded wait of the fused all-gather (after the stream has been synchronised)
int check_gather_status(rvl_t *h)
{
    if (h->h_status && h->h_status[0] != 0) {
        char buf[160];
        snprintf(buf, sizeof buf,
                 "fused all-gather timed out after %lld ms: exchange %llu, ranks missing (bit mask) 0x%llx",
                 h->opt_gather_timeout_ms, h->h_status[0], h->h_status[1]);
        h->h_status[0] = 0; h->h_status[1] = 0;
        return fail(h, RVL_EPEER, buf);
    }
    return RVL_OK;
}

}  // namespace

extern "C" {

int rvl_abi_version(void) { return RVL_ABI_VERSION; }

int rvl_create(rvl_t **out, int device)
{
    if (!out) return fail(nullptr, RVL_EINVAL, "out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, RVL_ENODEV,
                    std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count=0") +
                        " (librvlnl has no CPU fallback)");
    if (device < 0) cudaGetDevice(&device);
    if (device >= ndev) return fail(nullptr, RVL_ENODEV, "device index out of range");
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess)
        return fail(nullptr, RVL_ECUDA, "cudaGetDeviceProperties failed");
    if (prop.major != 10)
        return fail(nullptr, RVL_ENODEV,
                    "device is sm_" + std::to_string(prop.major * 10 + prop.minor) +
                        "; librvlnl is built for sm_100a only");
    rvl_t *h = new (std::nothrow) rvl_handle();
    if (!h) return fail(nullptr, RVL_ENOMEM, "out of host memory");
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    h->smem_optin = (int)prop.sharedMemPerBlockOptin;
    h->clock_khz = prop.clockRate;
    DevGuard g(device);
    auto bail = [&](const char *what, cudaError_t ce) {
        std::string msg = std::string(what) + ": " + cudaGetErrorString(ce);
        rvl_destroy(h);
        return fail(nullptr, RVL_ECUDA, msg);
    };
    cudaError_t ce;
    if ((ce = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("stream", ce);
    if ((ce = cudaEventCreate(&h->ev0)) != cudaSuccess) return bail("event", ce);
    if ((ce = cudaEventCreate(&h->ev1)) != cudaSuccess) return bail("event", ce);
    if ((ce = cudaEventCreate(&h->ev2)) != cudaSuccess) return bail("event", ce);
    if ((ce = cudaMalloc(&h->d_counters, 3 * sizeof(unsigned long long))) != cudaSuccess) return bail("malloc", ce);
    if ((ce = cudaMemset(h->d_counters, 0, 3 * sizeof(unsigned long long))) != cudaSuccess) return bail("memset", ce);
    // work counters + finished-block counter: zero now, the kernel re-arms them when it ends
    if ((ce = cudaMalloc(&h->d_work, sizeof(unsigned) * (size_t)(h->sm_count + 1))) != cudaSuccess) return bail("malloc", ce);
    if ((ce = cudaMemset(h->d_work, 0, sizeof(unsigned) * (size_t)(h->sm_count + 1))) != cudaSuccess) return bail("memset", ce);
    if ((ce = cudaMalloc(&h->d_model, sizeof(rvl_model_desc))) != cudaSuccess) return bail("malloc", ce);
    if ((ce = cudaHostAlloc((void **)&h->h_status, 2 * sizeof(unsigned long long), cudaHostAllocMapped)) != cudaSuccess) return bail("status word", ce);
    h->h_status[0] = 0; h->h_status[1] = 0;
    if ((ce = cudaHostGetDevicePointer((void **)&h->d_status, h->h_status, 0)) != cudaSuccess) return bail("status word", ce);
    *out = h;
    return RVL_OK;
}

int rvl_create_multi(rvl_t **out, const int32_t *devices, int32_t n_devices)
{
    if (!out) return fail(nullptr, RVL_EINVAL, "out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, RVL_ENODEV,
                    std::string("no CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "count=0") +
                        " (librvlnl has no CPU fallback)");
    if (n_devices < 0 || n_devices > RVL_MAX_PEERS || (n_devices > 0 && !devices))
        return fail(nullptr, RVL_EINVAL, "bad device list");
    std::vector<int> devs;
    if (n_devices == 0) for (int d = 0; d < std::min(ndev, RVL_MAX_PEERS); ++d) devs.push_back(d);  // every device of the box
    else devs.assign(devices, devices + n_devices);
    for (size_t i = 0; i < devs.size(); ++i)
        for (size_t j = 0; j < i; ++j)
            if (devs[i] == devs[j]) return fail(nullptr, RVL_EINVAL, "device listed twice");
    rvl_t *h = new (std::nothrow) rvl_handle();
    if (!h) return fail(nullptr, RVL_ENOMEM, "out of host memory");
    h->device = devs[0];
    for (int d : devs) {
        rvl_t *k = nullptr;
        const int rc = rvl_create(&k, d);
        if (rc) {  // g_create_error holds the reason
            const std::string msg = "device " + std::to_string(d) + ": " + g_create_error;
            rvl_destroy(h);
            return fail(nullptr, rc, msg);
        }
        h->kids.push_back(k);
    }
    h->sm_count = h->kids[0]->sm_count; h->smem_optin = h->kids[0]->smem_optin; h->clock_khz = h->kids[0]->clock_khz;
    *out = h;
    return RVL_OK;
}

int rvl_device_count(rvl_t *h, int32_t *n)
{
    if (!h || !n) return RVL_EINVAL;
    *n = h->kids.empty() ? 1 : (int32_t)h->kids.size();
    return RVL_OK;
}

void rvl_destroy(rvl_t *h)
{
    if (!h) return;
    if (!h->kids.empty()) {
        for (rvl_t *k : h->kids) rvl_destroy(k);
        h->kids.clear();
        delete h;
        return;
    }
    DevGuard g(h->device);
    // launches of the *_dev entry points may still be running on caller streams
    cudaDeviceSynchronize();
    cudaFree(h->d_cols); cudaFree(h->d_inst); cudaFree(h->d_model); cudaFree(h->d_priors);
    cudaFree(h->d_tables); cudaFree(h->d_theta); cudaFree(h->d_u); cudaFree(h->d_lnl);
    cudaFree(h->d_partial); cudaFree(h->d_flags); cudaFree(h->d_counters); cudaFree(h->d_work);
    cudaFree(h->d_consts); cudaFree(h->d_arrive); cudaFree(h->d_trace);
    cudaFree(h->d_gconsts); cudaFree(h->d_ready);
    cudaFree(h->d_curve_t); cudaFree(h->d_curve); cudaFree(h->d_curve_inv); cudaFree(h->d_curve_caps);
    if (h->pin_in) cudaFreeHost(h->pin_in);
    if (h->pin_out) cudaFreeHost(h->pin_out);
    if (h->pin_out2) cudaFreeHost(h->pin_out2);
    if (h->h_status) cudaFreeHost(h->h_status);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->ev2) cudaEventDestroy(h->ev2);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

const char *rvl_last_error(const rvl_t *h) { return h ? h->err.c_str() : g_create_error.c_str(); }

// a multi-device handle replicates the staging calls on every child (the epoch data and the model
// table are small and read-only: SURVEY.md 8(e))
#define RVL_FANOUT(h, call)                                                                      \
    do {                                                                                         \
        if (!(h)->kids.empty()) {                                                                \
            for (rvl_t *k : (h)->kids) {                                                         \
                const int rc_ = (call);                                                          \
                if (rc_) return multi_fail(h, k, rc_);                                           \
            }                                                                                    \
            return RVL_OK;                                                                       \
        }                                                                                        \
    } while (0)

int rvl_set_data(rvl_t *h, const double *t, const double *rv, const double *err,
                 const int32_t *inst, int32_t n, int32_t n_inst)
{
    if (!h) return RVL_EINVAL;
    RVL_FANOUT(h, rvl_set_data(k, t, rv, err, inst, n, n_inst));
    if (!t || !rv || !err || !inst) return fail(h, RVL_EINVAL, "NULL data pointer");
    if (n <= 0) return fail(h, RVL_EINVAL, "n must be positive");
    if (n_inst <= 0 || n_inst > RVL_MAX_INST)
        return fail(h, RVL_EINVAL, "n_inst must be in [1, " + std::to_string(RVL_MAX_INST) + "]");
    for (int j = 0; j < n; ++j)
        if (inst[j] < 0 || inst[j] >= n_inst) return fail(h, RVL_EINVAL, "instrument id out of range");
    // padded (the last epoch repeated, masked in the kernel) to whole groups of 4 chunks of 32: a
    // warp trip of U = 4 chunks then never meets a missing chunk
    h->N = n; h->Npad = (n + 127) / 128 * 128; h->n_inst = n_inst;
    h->h_t.assign(t, t + n); h->h_rv.assign(rv, rv + n); h->h_err.assign(err, err + n);
    h->h_inst.assign(inst, inst + n);
    h->tlo = *std::min_element(t, t + n);
    h->thi = *std::max_element(t, t + n);
    for (auto &c : h->h_linpar) c.clear();
    h->have_data = true; h->cols_dirty = true;
    return RVL_OK;
}

int rvl_set_linpar(rvl_t *h, int32_t idx, const double *col, int32_t n)
{
    if (!h) return RVL_EINVAL;
    RVL_FANOUT(h, rvl_set_linpar(k, idx, col, n));
    if (!h->have_data) return fail(h, RVL_ESTATE, "set data first");
    if (idx < 0 || idx >= RVL_MAX_LINPAR || !col || n != h->N)
        return fail(h, RVL_EINVAL, "bad linear-parameter column");
    h->h_linpar[idx].assign(col, col + n);
    h->cols_dirty = true;
    return RVL_OK;
}

static bool param_ok(const rvl_param &p, int ndim) { return p.slot >= -1 && p.slot < ndim; }

int rvl_set_model(rvl_t *h, const rvl_model_desc *d)
{
    if (!h) return RVL_EINVAL;
    RVL_FANOUT(h, rvl_set_model(k, d));
    if (!d) return fail(h, RVL_EINVAL, "desc is NULL");
    if (d->abi_version != RVL_ABI_VERSION) return fail(h, RVL_EINVAL, "abi_version mismatch");
    if (d->ndim < 0 || d->ndim > RVL_MAX_DIM) return fail(h, RVL_EINVAL, "ndim out of range");
    if (d->n_planets < 0 || d->n_planets > RVL_MAX_PLANETS) return fail(h, RVL_EINVAL, "n_planets out of range");
    if (d->n_inst <= 0 || d->n_inst > RVL_MAX_INST) return fail(h, RVL_EINVAL, "n_inst out of range");
    if (d->n_linpar < 0 || d->n_linpar > RVL_MAX_LINPAR) return fail(h, RVL_EINVAL, "n_linpar out of range");
    if (h->have_data && d->n_inst != h->n_inst) return fail(h, RVL_EINVAL, "n_inst differs from the staged data");
    if (d->itmax < 1) return fail(h, RVL_EINVAL, "itmax must be >= 1");
    if (!(d->tol > 0)) return fail(h, RVL_EINVAL, "tol must be positive");
    for (int p = 0; p < d->n_planets; ++p) {
        const rvl_planet_desc &pl = d->planet[p];
        if (!param_ok(pl.amp, d->ndim) || !param_ok(pl.period, d->ndim) || !param_ok(pl.e1, d->ndim) ||
            !param_ok(pl.e2, d->ndim) || !param_ok(pl.phase, d->ndim) || !param_ok(pl.epoch, d->ndim))
            return fail(h, RVL_EINVAL, "planet parameter slot out of range");
        if (pl.ecc_mode < 0 || pl.ecc_mode > 2 || pl.phase_mode < 0 || pl.phase_mode > 1)
            return fail(h, RVL_EINVAL, "bad parametrisation enum");
    }
    for (int i = 0; i < d->n_inst; ++i)
        if (!param_ok(d->offset[i], d->ndim) || !param_ok(d->jitter[i], d->ndim))
            return fail(h, RVL_EINVAL, "instrument parameter slot out of range");
    for (int i = 0; i < 4; ++i)
        if (!param_ok(d->drift[i], d->ndim)) return fail(h, RVL_EINVAL, "drift slot out of range");
    for (int i = 0; i < d->n_linpar; ++i)
        if (!param_ok(d->linpar[i], d->ndim)) return fail(h, RVL_EINVAL, "linpar slot out of range");
    DevGuard g(h->device);
    h->model = *d;
    CU(h, cudaMemcpy(h->d_model, d, sizeof(*d), cudaMemcpyHostToDevice));
    h->have_model = true; h->cols_dirty = true;
    // scratch rows depend on ndim
    h->cap_B = 0;
    return RVL_OK;
}

int rvl_set_priors(rvl_t *h, const rvl_prior_desc *priors, int32_t ndim, const double *tables,
                   int64_t n_table_doubles)
{
    if (!h) return RVL_EINVAL;
    RVL_FANOUT(h, rvl_set_priors(k, priors, ndim, tables, n_table_doubles));
    if (!priors || ndim <= 0 || ndim > RVL_MAX_DIM) return fail(h, RVL_EINVAL, "bad priors / ndim");
    for (int i = 0; i < ndim; ++i) {
        const rvl_prior_desc &p = priors[i];
        if (p.kind < 0 || p.kind > RVL_PRIOR_TABLE) return fail(h, RVL_EINVAL, "unknown prior kind");
        if (p.kind == RVL_PRIOR_TABLE &&
            (p.table_len < 2 || p.table_offset < 0 || !tables ||
             p.table_offset + (p.p[1] != 0.0 ? 3LL : 2LL) * p.table_len > n_table_doubles))
            return fail(h, RVL_EINVAL, "prior table out of bounds");
    }
    DevGuard g(h->device);
    cudaFree(h->d_priors); cudaFree(h->d_tables);
    h->d_priors = nullptr; h->d_tables = nullptr;
    CU(h, cudaMalloc(&h->d_priors, sizeof(rvl_prior_desc) * (size_t)ndim));
    CU(h, cudaMemcpy(h->d_priors, priors, sizeof(rvl_prior_desc) * (size_t)ndim, cudaMemcpyHostToDevice));
    if (n_table_doubles > 0 && tables) {
        CU(h, cudaMalloc(&h->d_tables, sizeof(double) * (size_t)n_table_doubles));
        CU(h, cudaMemcpy(h->d_tables, tables, sizeof(double) * (size_t)n_table_doubles, cudaMemcpyHostToDevice));
    }
    h->prior_ndim = ndim; h->have_priors = true;
    h->cap_B = 0;
    return RVL_OK;
}

int rvl_set_option(rvl_t *h, const char *name, int64_t value)
{
    if (!h || !name) return RVL_EINVAL;
    RVL_FANOUT(h, rvl_set_option(k, name, value));
    const std::string n(name);
    if (n == "variant") { if (value < 0 || value > 1) return fail(h, RVL_EINVAL, "variant in {0,1}"); h->opt_variant = (int)value; }
    else if (n == "slices") h->opt_slices = (int)std::max<int64_t>(0, value);
    else if (n == "warps") h->opt_warps = (int)std::max<int64_t>(0, std::min<int64_t>(32, value));
    else if (n == "timing") h->opt_timing = value != 0;
    else if (n == "zero_copy") h->opt_zero_copy = (int)std::max<int64_t>(0, std::min<int64_t>(2, value));
    else if (n == "min_chunks") h->opt_min_chunks = (int)std::max<int64_t>(1, value);
    else if (n == "items_per_warp") h->opt_items_per_warp = (int)std::max<int64_t>(1, value);
    else if (n == "sched") h->opt_sched = value != 0;
    else if (n == "phase_items") h->opt_phase_items = (int)std::max<int64_t>(1, std::min<int64_t>(100000, value));
    else if (n == "max_split") h->opt_max_split = (int)std::max<int64_t>(1, std::min<int64_t>(4096, value));
    else if (n == "prepare") h->opt_prepare = value != 0;
    else if (n == "trace") h->opt_trace = value != 0;
    else if (n == "setup_items") h->opt_setup_items = value != 0;
    else if (n == "gather_timeout_ms") h->opt_gather_timeout_ms = std::max<int64_t>(1, value);
    else if (n == "ilp") { if (value < 0 || value > 4) return fail(h, RVL_EINVAL, "ilp in {0 (automatic),1,2,3,4}"); h->opt_ilp = (int)value; }
    else return fail(h, RVL_EINVAL, "unknown option " + n);
    return RVL_OK;
}

int rvl_loglike_dev(rvl_t *h, const double *dTheta, int64_t B, double *dlnL, void *stream)
{
    if (!h) return RVL_EINVAL;
    if (!h->kids.empty()) return fail(h, RVL_EINVAL, "device-pointer entry points need a single-device handle");
    if (B < 0 || (B > 0 && (!dTheta || !dlnL))) return fail(h, RVL_EINVAL, "bad arguments");
    DevGuard g(h->device);
    return enqueue_loglike(h, nullptr, const_cast<double *>(dTheta), B, dlnL, (cudaStream_t)stream,
                           h->opt_timing != 0);
}

int rvl_loglike_dev_scatter(rvl_t *h, const double *dTheta, int64_t B, double *dlnL,
                            const uint64_t *peer_ptrs, int32_t n_peers, int64_t offset,
                            void *stream)
{
    if (!h) return RVL_EINVAL;
    if (!h->kids.empty()) return fail(h, RVL_EINVAL, "device-pointer entry points need a single-device handle");
    if (B < 0 || (B > 0 && (!dTheta || !dlnL))) return fail(h, RVL_EINVAL, "bad arguments");
    if (n_peers < 0 || n_peers > RVL_MAX_PEERS || (n_peers > 0 && !peer_ptrs) || offset < 0)
        return fail(h, RVL_EINVAL, "bad peer list");
    PeerOut po{};
    po.n = n_peers;
    po.offset = offset;
    for (int r = 0; r < n_peers; ++r) po.ptr[r] = reinterpret_cast<double *>(peer_ptrs[r]);
    DevGuard g(h->device);
    return enqueue_loglike(h, nullptr, const_cast<double *>(dTheta), B, dlnL, (cudaStream_t)stream,
                           h->opt_timing != 0, &po);
}

int rvl_loglike_dev_gather(rvl_t *h, const double *dTheta, int64_t B, double *dlnL,
                           const uint64_t *peer_ptrs, int32_t n_peers, int32_t rank, int64_t offset,
                           int64_t flag_offset, uint64_t seq, void *stream)
{
    if (!h) return RVL_EINVAL;
    if (!h->kids.empty()) return fail(h, RVL_EINVAL, "device-pointer entry points need a single-device handle");
    if (B <= 0 || !dTheta || !dlnL) return fail(h, RVL_EINVAL, "bad arguments");
    if (n_peers < 1 || n_peers > RVL_MAX_PEERS || !peer_ptrs || offset < 0 || rank < 0 ||
        rank >= n_peers || flag_offset < 0 || seq == 0)
        return fail(h, RVL_EINVAL, "bad peer list");
    PeerOut po{};
    po.n = n_peers;
    po.offset = offset;
    po.flag_off = flag_offset;
    po.seq = seq;
    po.rank = rank;
    for (int r = 0; r < n_peers; ++r) po.ptr[r] = reinterpret_cast<double *>(peer_ptrs[r]);
    DevGuard g(h->device);
    int rc = enqueue_loglike(h, nullptr, const_cast<double *>(dTheta), B, dlnL, (cudaStream_t)stream,
                             h->opt_timing != 0, &po);
    if (rc) return rc;
    wait_flags_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const unsigned long long *>(po.ptr[rank]) + flag_offset, n_peers, seq,
        (unsigned long long)h->opt_gather_timeout_ms * 1000000ull, h->d_status);
    CU(h, cudaGetLastError());
    ++h->launches;
    if (h->timing_pending) { CU(h, cudaEventRecord(h->ev2, (cudaStream_t)stream)); h->wait_pending = true; }
    return RVL_OK;
}

int rvl_transform_dev(rvl_t *h, const double *dU, int64_t B, double *dTheta, void *stream)
{
    if (!h) return RVL_EINVAL;
    if (!h->kids.empty()) return fail(h, RVL_EINVAL, "device-pointer entry points need a single-device handle");
    if (B < 0 || (B > 0 && (!dU || !dTheta))) return fail(h, RVL_EINVAL, "bad arguments");
    DevGuard g(h->device);
    return enqueue_transform(h, dU, B, dTheta, (cudaStream_t)stream);
}

int rvl_transform_loglike_dev(rvl_t *h, const double *dU, int64_t B, double *dTheta, double *dlnL,
                              void *stream)
{
    if (!h) return RVL_EINVAL;
    if (!h->kids.empty()) return fail(h, RVL_EINVAL, "device-pointer entry points need a single-device handle");
    if (B < 0 || (B > 0 && (!dU || !dTheta || !dlnL))) return fail(h, RVL_EINVAL, "bad arguments");
    if (h->have_model && h->have_priors && h->prior_ndim != h->model.ndim)
        return fail(h, RVL_ESTATE, "priors and model disagree on ndim");
    DevGuard g(h->device);
    return enqueue_loglike(h, dU, dTheta, B, dlnL, (cudaStream_t)stream, h->opt_timing != 0);
}

int rvl_loglike(rvl_t *h, const double *Theta, int64_t B, double *lnL)
{
    if (!h) return RVL_EINVAL;
    if (B < 0 || (B > 0 && (!Theta || !lnL))) return fail(h, RVL_EINVAL, "bad arguments");
    if (!h->kids.empty()) return multi_rows(h, Theta, nullptr, nullptr, lnL, B, /*mode=*/0);
    if (!h->have_data || !h->have_model) return fail(h, RVL_ESTATE, "set data and model first");
    if (B == 0) return RVL_OK;
    DevGuard g(h->device);
    HostCall hc;
    int rc = loglike_begin(h, Theta, B, lnL, hc);
    if (rc) return rc;
    return hostcall_end(h, hc);
}

int rvl_transform(rvl_t *h, const double *U, int64_t B, double *Theta)
{
    if (!h) return RVL_EINVAL;
    if (B < 0 || (B > 0 && (!U || !Theta))) return fail(h, RVL_EINVAL, "bad arguments");
    if (!h->kids.empty()) return multi_rows(h, nullptr, U, Theta, nullptr, B, /*mode=*/1);
    if (!h->have_priors) return fail(h, RVL_ESTATE, "set priors first");
    if (B == 0) return RVL_OK;
    DevGuard g(h->device);
    HostCall hc;
    int rc = transform_begin(h, U, B, Theta, hc);
    if (rc) return rc;
    return hostcall_end(h, hc);
}

int rvl_transform_loglike(rvl_t *h, const double *U, int64_t B, double *Theta, double *lnL)
{
    if (!h) return RVL_EINVAL;
    if (B < 0 || (B > 0 && (!U || !lnL))) return fail(h, RVL_EINVAL, "bad arguments");
    if (!h->kids.empty()) return multi_rows(h, nullptr, U, Theta, lnL, B, /*mode=*/2);
    if (!h->have_data || !h->have_model || !h->have_priors)
        return fail(h, RVL_ESTATE, "set data, model and priors first");
    if (h->prior_ndim != h->model.ndim) return fail(h, RVL_ESTATE, "priors and model disagree on ndim");
    if (B == 0) return RVL_OK;
    DevGuard g(h->device);
    HostCall hc;
    int rc = transform_loglike_begin(h, U, B, Theta, lnL, hc);
    if (rc) return rc;
    return hostcall_end(h, hc);
}

/* per-rank host-buffer form of the fused all-gather (one process per GPU): this rank's rows of
 * theta in host memory in, the gathered lnL of ALL ranks in host memory out */
int rvl_loglike_gather(rvl_t *h, const double *Theta, int64_t B, double *lnL_all,
                       const uint64_t *peer_ptrs, int32_t n_peers, int32_t rank,
                       int64_t flag_offset, uint64_t seq)
{
    if (!h) return RVL_EINVAL;
    if (!h->kids.empty()) return fail(h, RVL_EINVAL, "not available on a multi-device handle");
    if (B <= 0 || !Theta || !lnL_all) return fail(h, RVL_EINVAL, "bad arguments");
    if (n_peers < 1 || n_peers > RVL_MAX_PEERS || !peer_ptrs || rank < 0 || rank >= n_peers ||
        flag_offset < (int64_t)n_peers * B || seq == 0)
        return fail(h, RVL_EINVAL, "bad peer list");
    if (!h->have_data || !h->have_model) return fail(h, RVL_ESTATE, "set data and model first");
    PeerOut po{};
    po.n = n_peers;
    po.offset = (long long)rank * B;
    po.flag_off = flag_offset;
    po.seq = seq;
    po.rank = rank;
    for (int r = 0; r < n_peers; ++r) po.ptr[r] = reinterpret_cast<double *>(peer_ptrs[r]);
    DevGuard g(h->device);
    HostCall hc;
    int rc = ensure_io(h, B);
    if (rc) return rc;
    rc = loglike_begin(h, Theta, B, nullptr, hc, &po, h->d_lnl);
    if (rc) return rc;
    wait_flags_kernel<<<1, 32, 0, h->stream>>>(
        reinterpret_cast<const unsigned long long *>(po.ptr[rank]) + flag_offset, n_peers, seq,
        (unsigned long long)h->opt_gather_timeout_ms * 1000000ull, h->d_status);
    CU(h, cudaGetLastError());
    ++h->launches;
    if (h->timing_pending) { CU(h, cudaEventRecord(h->ev2, h->stream)); h->wait_pending = true; }
    CU(h, cudaMemcpyAsync(lnL_all, po.ptr[rank], (size_t)n_peers * (size_t)B * sizeof(double),
                          cudaMemcpyDeviceToHost, h->stream));
    rc = hostcall_end(h, hc);
    if (rc) return rc;
    return check_gather_status(h);
}

int rvl_trueanomaly(rvl_t *h, const double *M, int32_t n, double ecc, double *nu,
                    int32_t niterationmax, double tol)
{
    if (!h) return RVL_EINVAL;
    if (n < 0 || (n > 0 && (!M || !nu)) || niterationmax < 1) return fail(h, RVL_EINVAL, "bad arguments");
    if (n == 0) return 0;
    if (!h->kids.empty()) return rvl_trueanomaly(h->kids[0], M, n, ecc, nu, niterationmax, tol);
    DevGuard g(h->device);
    double *dM = nullptr, *dnu = nullptr;
    int *dcap = nullptr;
    int cap = 0;
    // one exit: the three scratch buffers are released whatever fails
    cudaError_t e = cudaMalloc(&dM, sizeof(double) * (size_t)n);
    if (e == cudaSuccess) e = cudaMalloc(&dnu, sizeof(double) * (size_t)n);
    if (e == cudaSuccess) e = cudaMalloc(&dcap, sizeof(int));
    if (e == cudaSuccess) e = cudaMemsetAsync(dcap, 0, sizeof(int), h->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dM, M, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess) {
        const int tb = 128;
        trueanomaly_kernel<<<(n + tb - 1) / tb, tb, 0, h->stream>>>(dM, n, ecc, dnu, niterationmax, tol, dcap);
        ++h->launches;
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(nu, dnu, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&cap, dcap, sizeof(int), cudaMemcpyDeviceToHost, h->stream);
    const cudaError_t e2 = cudaStreamSynchronize(h->stream);
    cudaFree(dM); cudaFree(dnu); cudaFree(dcap);
    if (e != cudaSuccess) return fail(h, RVL_ECUDA, std::string("rvl_trueanomaly: ") + cudaGetErrorString(e));
    if (e2 != cudaSuccess) return fail(h, RVL_ECUDA, std::string("rvl_trueanomaly: ") + cudaGetErrorString(e2));
    return cap ? -1 : 0;  // same 0 / -1 convention as trueanomaly.c:32-40
}

int rvl_kepler_rv_dev(rvl_t *h, const double *dTheta, int64_t B, const double *dTimes, int32_t T,
                      uint32_t planet_mask, double *dOut, uint32_t *dInvalid, uint64_t *dCapHits,
                      void *stream)
{
    if (!h) return RVL_EINVAL;
    if (!h->kids.empty()) return fail(h, RVL_EINVAL, "device-pointer entry points need a single-device handle");
    if (B < 0 || T < 0 || (B > 0 && (!dTheta || (T > 0 && (!dTimes || !dOut)))))
        return fail(h, RVL_EINVAL, "bad arguments");
    DevGuard g(h->device);
    return enqueue_kepler_rv(h, dTheta, B, dTimes, T, planet_mask, dOut, dInvalid,
                             reinterpret_cast<unsigned long long *>(dCapHits), (cudaStream_t)stream);
}

int rvl_kepler_rv(rvl_t *h, const double *Theta, int64_t B, const double *times, int32_t T,
                  uint32_t planet_mask, double *out, uint32_t *invalid, uint64_t *cap_hits)
{
    if (!h) return RVL_EINVAL;
    if (B < 0 || T < 0 || (B > 0 && (!Theta || (T > 0 && (!times || !out)))))
        return fail(h, RVL_EINVAL, "bad arguments");
    if (!h->kids.empty()) {
        const int rc = rvl_kepler_rv(h->kids[0], Theta, B, times, T, planet_mask, out, invalid, cap_hits);
        return rc ? multi_fail(h, h->kids[0], rc) : RVL_OK;
    }
    if (!h->have_model) return fail(h, RVL_ESTATE, "set the model first");
    if (B == 0) return RVL_OK;
    DevGuard g(h->device);
    int rc = ensure_io(h, B);
    if (rc) return rc;
    const size_t nT = (size_t)std::max(1, T), nout = (size_t)B * (size_t)T;
    if (nT > h->cap_curve_t) {
        cudaFree(h->d_curve_t);
        h->d_curve_t = nullptr; h->cap_curve_t = 0;
        CU(h, cudaMalloc(&h->d_curve_t, nT * sizeof(double)));
        h->cap_curve_t = nT;
    }
    if (nout > h->cap_curve) {
        cudaFree(h->d_curve);
        h->d_curve = nullptr; h->cap_curve = 0;
        CU(h, cudaMalloc(&h->d_curve, nout * sizeof(double)));
        h->cap_curve = nout;
    }
    if (B > h->cap_curve_inv) {
        cudaFree(h->d_curve_inv);
        h->d_curve_inv = nullptr; h->cap_curve_inv = 0;
        CU(h, cudaMalloc(&h->d_curve_inv, (size_t)B * sizeof(uint32_t)));
        h->cap_curve_inv = B;
    }
    if (!h->d_curve_caps) CU(h, cudaMalloc(&h->d_curve_caps, sizeof(unsigned long long)));
    cudaStream_t st = h->stream;
    const size_t nb = (size_t)B * h->model.ndim * sizeof(double);
    if (nb) CU(h, cudaMemcpyAsync(h->d_theta, Theta, nb, cudaMemcpyHostToDevice, st));
    if (T > 0) CU(h, cudaMemcpyAsync(h->d_curve_t, times, (size_t)T * sizeof(double), cudaMemcpyHostToDevice, st));
    CU(h, cudaMemsetAsync(h->d_curve_caps, 0, sizeof(unsigned long long), st));
    rc = enqueue_kepler_rv(h, h->d_theta, B, h->d_curve_t, T, planet_mask, h->d_curve, h->d_curve_inv,
                           h->d_curve_caps, st);
    if (rc) return rc;
    unsigned long long caps = 0;
    if (nout) CU(h, cudaMemcpyAsync(out, h->d_curve, nout * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (invalid)
        CU(h, cudaMemcpyAsync(invalid, h->d_curve_inv, (size_t)B * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CU(h, cudaMemcpyAsync(&caps, h->d_curve_caps, sizeof caps, cudaMemcpyDeviceToHost, st));
    CU(h, cudaStreamSynchronize(st));
    if (cap_hits) *cap_hits += caps;
    return RVL_OK;
}

int rvl_counters(rvl_t *h, rvl_counters_t *out)
{
    if (!h || !out) return RVL_EINVAL;
    if (!h->kids.empty()) {  // sums over the devices
        rvl_counters_t acc{};
        for (rvl_t *k : h->kids) {
            rvl_counters_t c{};
            const int rc = rvl_counters(k, &c);
            if (rc) return multi_fail(h, k, rc);
            acc.n_points += c.n_points; acc.n_solves += c.n_solves; acc.n_newton_iters += c.n_newton_iters;
            acc.n_cap_hits += c.n_cap_hits; acc.n_invalid += c.n_invalid;
        }
        *out = acc;
        return RVL_OK;
    }
    DevGuard g(h->device);
    unsigned long long c[3] = {0, 0, 0};
    CU(h, cudaStreamSynchronize(h->stream));
    CU(h, cudaMemcpy(c, h->d_counters, sizeof c, cudaMemcpyDeviceToHost));
    out->n_points = h->n_points; out->n_solves = h->n_solves;
    out->n_newton_iters = c[0]; out->n_cap_hits = c[1]; out->n_invalid = c[2];
    return RVL_OK;
}

int rvl_reset_counters(rvl_t *h)
{
    if (!h) return RVL_EINVAL;
    RVL_FANOUT(h, rvl_reset_counters(k));
    DevGuard g(h->device);
    CU(h, cudaStreamSynchronize(h->stream));
    CU(h, cudaMemset(h->d_counters, 0, 3 * sizeof(unsigned long long)));
    h->n_points = 0; h->n_solves = 0;
    return RVL_OK;
}

int rvl_last_kernel_ms(rvl_t *h, double *ms)
{
    if (!h || !ms) return RVL_EINVAL;
    if (!h->kids.empty()) {  // the devices run concurrently: the call's kernel time is the longest
        double worst = 0.0;
        for (rvl_t *k : h->kids) {
            double v = 0.0;
            const int rc = rvl_last_kernel_ms(k, &v);
            if (rc) return multi_fail(h, k, rc);
            worst = std::max(worst, v);
        }
        *ms = worst;
        return RVL_OK;
    }
    if (h->timing_pending) {  // *_dev launches: wait for the kernel's end event
        DevGuard g(h->device);
        CU(h, cudaEventSynchronize(h->wait_pending ? h->ev2 : h->ev1));
        int rc = finish_timing(h);
        if (rc) return rc;
    }
    *ms = h->last_ms;
    return RVL_OK;
}

int rvl_last_gather_wait_ms(rvl_t *h, double *ms)
{
    if (!h || !ms) return RVL_EINVAL;
    double k = 0.0;
    const int rc = rvl_last_kernel_ms(h, &k);  // resolves the pending events
    if (rc) return rc;
    *ms = h->last_wait_ms;
    return RVL_OK;
}

int rvl_launch_count(rvl_t *h, uint64_t *n)
{
    if (!h || !n) return RVL_EINVAL;
    *n = h->launches;
    for (rvl_t *k : h->kids) *n += k->launches;
    return RVL_OK;
}

/* Recovery after a faulted or aborted launch: the work / arrival counters and the ready stamps
 * re-arm themselves only when a launch runs to its end; this puts them back to the state of a
 * fresh handle (the stream is drained first).  Also clears a recorded all-gather timeout. */
int rvl_reset(rvl_t *h)
{
    if (!h) return RVL_EINVAL;
    RVL_FANOUT(h, rvl_reset(k));
    DevGuard g(h->device);
    cudaStreamSynchronize(h->stream);
    cudaGetLastError();  // a sticky launch failure is reported by the next call, not swallowed here
    CU(h, cudaMemset(h->d_work, 0, sizeof(unsigned) * (size_t)(h->sm_count + 1)));
    if (h->d_arrive) CU(h, cudaMemset(h->d_arrive, 0, (size_t)h->cap_arrive * sizeof(int)));
    if (h->d_ready) CU(h, cudaMemset(h->d_ready, 0, (size_t)h->cap_ready * sizeof(unsigned)));
    h->seq = 0;
    h->timing_pending = false;
    if (h->h_status) { h->h_status[0] = 0; h->h_status[1] = 0; }
    return RVL_OK;
}

/* 0 when no bounded wait of the fused all-gather has expired on this handle since the last check;
 * RVL_EPEER (message: the exchange number and the missing ranks) otherwise.  For the asynchronous
 * rvl_loglike_dev_gather: call it after synchronising the stream. */
/* ---- gather through a host segment shared by the ranks' processes -------------------------------
 * One process per GPU, HOST consumers: instead of every rank copying the whole gathered vector back
 * (world x B doubles over each PCIe link), every rank's kernel stores ITS lnL block straight into a
 * host memory segment that all the processes map (POSIX shared memory, registered with CUDA by each
 * of them): B doubles per link, overlapped with the arithmetic, no device-side gather buffer, no
 * D2H copy.  Completion: the launch's last block stores `seq` into this rank's flag slot of the same
 * segment (system-scope release, after every block has fenced its stores); the ranks then wait for
 * all slots on the HOST (rvl_wait_host_flags). */
int rvl_host_register(void *ptr, int64_t bytes, uint64_t *dev_ptr)
{
    if (!ptr || bytes <= 0 || !dev_ptr) return fail(nullptr, RVL_EINVAL, "bad arguments");
    cudaError_t e = cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterMapped | cudaHostRegisterPortable);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(nullptr, RVL_ECUDA, std::string("cudaHostRegister: ") + cudaGetErrorString(e)); }
    void *d = nullptr;
    e = cudaHostGetDevicePointer(&d, ptr, 0);
    if (e != cudaSuccess) { cudaHostUnregister(ptr); cudaGetLastError(); return fail(nullptr, RVL_ECUDA, std::string("cudaHostGetDevicePointer: ") + cudaGetErrorString(e)); }
    *dev_ptr = (uint64_t)(uintptr_t)d;
    return RVL_OK;
}

int rvl_host_unregister(void *ptr)
{
    if (!ptr) return RVL_EINVAL;
    const cudaError_t e = cudaHostUnregister(ptr);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(nullptr, RVL_ECUDA, std::string("cudaHostUnregister: ") + cudaGetErrorString(e)); }
    return RVL_OK;
}

int rvl_loglike_scatter_host(rvl_t *h, const double *Theta, int64_t B, uint64_t shared_dev_ptr,
                             int64_t offset, int64_t flag_offset, int32_t rank, uint64_t seq)
{
    if (!h) return RVL_EINVAL;
    if (!h->kids.empty()) return fail(h, RVL_EINVAL, "not available on a multi-device handle");
    if (B <= 0 || !Theta || !shared_dev_ptr || offset < 0 || flag_offset < 0 || rank < 0 || seq == 0)
        return fail(h, RVL_EINVAL, "bad arguments");
    if (!h->have_data || !h->have_model) return fail(h, RVL_ESTATE, "set data and model first");
    PeerOut po{};
    po.n = 1;
    po.ptr[0] = reinterpret_cast<double *>((uintptr_t)shared_dev_ptr);
    po.offset = offset;
    po.flag_off = flag_offset;
    po.seq = seq;
    po.rank = rank;
    DevGuard g(h->device);
    HostCall hc;
    int rc = ensure_io(h, B);
    if (rc) return rc;
    rc = loglike_begin(h, Theta, B, nullptr, hc, &po, h->d_lnl);
    if (rc) return rc;
    return hostcall_end(h, hc);
}

int rvl_wait_host_flags(const uint64_t *flags, int32_t n, uint64_t seq, int32_t timeout_ms)
{
    if (!flags || n < 1 || n > 4096) return RVL_EINVAL;
    const volatile uint64_t *f = flags;
    const auto t0 = std::chrono::steady_clock::now();
    for (int i = 0; i < n; ++i) {
        unsigned spins = 0;
        while (f[i] < seq) {
#if defined(__x86_64__) || defined(__i386__)
            __builtin_ia32_pause();
#endif
            if ((++spins & 0xfffu) == 0u) {
                const auto ms = std::chrono::duration_cast<std::chrono::milliseconds>(
                                    std::chrono::steady_clock::now() - t0).count();
                if (timeout_ms >= 0 && ms > timeout_ms) {
                    g_create_error = "shared-host gather timed out: rank " + std::to_string(i) + " never signalled exchange " + std::to_string((unsigned long long)seq);
                    return RVL_EPEER;
                }
            }
        }
    }
    __atomic_thread_fence(__ATOMIC_ACQUIRE);
    return RVL_OK;
}

int rvl_gather_status(rvl_t *h)
{
    if (!h) return RVL_EINVAL;
    if (!h->kids.empty()) return RVL_OK;
    return check_gather_status(h);
}

int rvl_fp64_peak(rvl_t *h, double *tflops)
{
    if (!h || !tflops) return RVL_EINVAL;
    if (!h->kids.empty()) {  // sum over the devices
        double tot = 0.0;
        for (rvl_t *k : h->kids) {
            double v = 0.0;
            const int rc = rvl_fp64_peak(k, &v);
            if (rc) return multi_fail(h, k, rc);
            tot += v;
        }
        *tflops = tot;
        return RVL_OK;
    }
    DevGuard g(h->device);
    const int blocks = h->sm_count, tb = 1024, iters = 4000;
    double *out = nullptr;
    CU(h, cudaMalloc(&out, sizeof(double) * (size_t)blocks * tb));
    double best = 0.0;
    for (int rep = 0; rep < 9; ++rep) {  // best over chain counts 2, 4, 8 and repetitions
        const int R = rep % 3 == 0 ? 2 : (rep % 3 == 1 ? 4 : 8);
        CU(h, cudaEventRecord(h->ev0, h->stream));
        if (R == 2) dfma_peak_kernel<2><<<blocks, tb, 0, h->stream>>>(out, iters, 0.999999, 1e-9);
        else if (R == 4) dfma_peak_kernel<4><<<blocks, tb, 0, h->stream>>>(out, iters, 0.999999, 1e-9);
        else dfma_peak_kernel<8><<<blocks, tb, 0, h->stream>>>(out, iters, 0.999999, 1e-9);
        CU(h, cudaEventRecord(h->ev1, h->stream));
        CU(h, cudaStreamSynchronize(h->stream));
        ++h->launches;
        float ms = 0.f;
        CU(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
        const double flops = 2.0 * 8.0 * R * (double)iters * (double)blocks * tb;
        if (rep >= 3) best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    cudaFree(out);
    *tflops = best;
    return RVL_OK;
}

int rvl_read_trace(rvl_t *h, uint64_t *out, int32_t cap_rows, int32_t *rows)
{
    if (!h || !out || !rows) return RVL_EINVAL;
    *rows = 0;
    if (!h->kids.empty()) return rvl_read_trace(h->kids[0], out, cap_rows, rows);
    if (!h->d_trace || h->trace_rows <= 0) return fail(h, RVL_ESTATE, "no trace recorded (option \"trace\")");
    if (cap_rows < h->trace_rows) return fail(h, RVL_EINVAL, "trace buffer too small");
    DevGuard g(h->device);
    CU(h, cudaDeviceSynchronize());
    CU(h, cudaMemcpy(out, h->d_trace, (size_t)h->trace_rows * 4 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    *rows = h->trace_rows;
    return RVL_OK;
}

int rvl_plan_describe(const int32_t *in, int64_t B, int64_t *out, int32_t cap)
{
    if (!in || !out || cap < 8) return RVL_EINVAL;
    PlanIn pi{};
    pi.Ctot = in[0]; pi.ncol = in[1]; pi.wstride = in[2]; pi.wblock = in[2]; pi.U = in[3]; pi.W = in[4];
    pi.sm_count = in[5]; pi.smem_optin = in[6]; pi.sched = in[7]; pi.slices = in[8];
    pi.items_per_warp = in[9]; pi.min_chunks = in[10]; pi.phase_items = in[11]; pi.max_split = in[12];
    if (pi.Ctot < 1 || pi.U < 1 || pi.U > 4 || pi.W < 1 || pi.sm_count < 1 || B < 1) return RVL_EINVAL;
    Plan pl{};
    if (plan_core(pi, B, pl)) return RVL_EINVAL;
    if (cap < 8 + 5 * pl.nph) return RVL_EINVAL;
    out[0] = pl.Sm; out[1] = pl.cpm; out[2] = pl.grid; out[3] = pl.nph; out[4] = pl.nitems;
    out[5] = pl.ptS0; out[6] = pl.n_split; out[7] = (int64_t)pl.partial_doubles;
    for (int i = 0; i < pl.nph; ++i) {
        int64_t *o = out + 8 + 5 * i;
        o[0] = pl.ph[i].idx0; o[1] = pl.ph[i].S; o[2] = pl.ph[i].cps; o[3] = pl.ph[i].pt0;
        o[4] = pl.ph[i].part0;
    }
    return RVL_OK;
}

int rvl_device_info(rvl_t *h, int32_t *sm_count, int32_t *smem_optin, int32_t *clock_khz)
{
    if (!h) return RVL_EINVAL;
    if (sm_count) *sm_count = h->sm_count;
    if (smem_optin) *smem_optin = h->smem_optin;
    if (clock_khz) *clock_khz = h->clock_khz;
    return RVL_OK;
}

}  // extern "C"
