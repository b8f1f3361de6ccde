// emul.cpp — TEST HARNESS ONLY (never shipped, never on the product path).
//
// Replays the arithmetic of rv_lnl_kernel (evidence_b200/csrc/rvlnl.cu) on the CPU, lane by lane
// in warp lock-step, by compiling the very same FP64 core (evidence_b200/csrc/rvl_math.h) for the
// host.  It exists so that the numerics of the kernel's optimisations (reciprocal-multiply Newton
// step, warp-uniform small-step sin/cos advance, mantissa-product log-det) can be checked against
// the reference's golden outputs in a container without a GPU.  Differences from the device:
// the reciprocal seed (float division instead of MUFU.RCP64H) and libm instead of libdevice in
// the once-per-point setup; both are below the last-ulp level of what they feed.
//
// It also counts how many warp-trips took each sin/cos path, which gives the FP64 instruction
// count per Kepler solve that the roofline discussion in DESIGN.md uses.
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../../evidence_b200/csrc/rvl_lean.h"
#include "../../evidence_b200/csrc/rvl_math.h"
#include "../../include/rvlnl.h"

namespace {

constexpr int W = 32;
constexpr int kPlanetStride = 8;

struct Stats {
    long long trips_full, trips_small, trips_tiny, solves_warp, newton_iters, caps, trips_medium;
};

inline double par_of(const rvl_param &p, const double *row) { return p.slot >= 0 ? row[p.slot] : p.value; }


inline int abs_hi(double x) { return rvl::hi32(x) & 0x7fffffff; }
using rvl::kHiTrigMax, rvl::kHiTiny, rvl::kHiSmall, rvl::kHiMid, rvl::kHiMedium;

// one planet for U chunks of 32 epochs (U*32 solves) in lock-step: mirrors solve_planet<0, U>
void solve_planet_warp(int U, const double *const *t, const double *pc, double tol, int itmax,
                       double (*out)[W], int (*iters)[W], int *caps, Stats &st)
{
    const double nmot = pc[0], M0 = pc[1], ec = pc[2], A = pc[3], Bs = pc[4], Ce = pc[5], epoch = pc[6];
    double M[2][W], E[2][W], s[2][W], c[2][W], d[2][W];
    int last[2][W];
    bool big = false;
    for (int u = 0; u < U; ++u)
        for (int l = 0; l < W; ++l) {
            M[u][l] = rvl::mean_anomaly(nmot, t[u][l], epoch, M0);
            E[u][l] = M[u][l];
            big = big || !(abs_hi(M[u][l]) < kHiTrigMax);
            d[u][l] = 1e300;
            s[u][l] = 0.0;
            c[u][l] = 1.0;
            last[u][l] = 0;
        }
    const bool slow = big || !(ec >= -0.99);
    ++st.solves_warp;
    int trip = 0;
    for (;;) {
        bool all_tiny = true, all_small = true, all_mid = true, all_medium = true, any_big = false;
        for (int u = 0; u < U; ++u)
            for (int l = 0; l < W; ++l) {
                const int h = abs_hi(d[u][l]);
                all_tiny = all_tiny && (h < kHiTiny);
                all_small = all_small && (h < kHiSmall);
                all_mid = all_mid && (h < kHiMid);
                all_medium = all_medium && (h < kHiMedium);
                any_big = any_big || !(abs_hi(E[u][l]) < kHiTrigMax);
            }
        bool all_final = true;
        const int tol_hi = rvl::hi32(tol);
        for (int u = 0; u < U; ++u)
            for (int l = 0; l < W; ++l) all_final = all_final && (abs_hi(d[u][l]) < tol_hi);
        if (all_final && tol_hi < rvl::kHiFinal) {  // the last pass: shorter series, then out
            ++st.trips_tiny;
            for (int u = 0; u < U; ++u) for (int l = 0; l < W; ++l) rvl::advance_final(rvl::h_ktab, d[u][l], s[u][l], c[u][l]);
            break;
        }
        if (all_tiny) { ++st.trips_tiny; for (int u = 0; u < U; ++u) for (int l = 0; l < W; ++l) rvl::advance_tiny(rvl::h_ktab, d[u][l], s[u][l], c[u][l]); }
        else if (all_small) { ++st.trips_small; for (int u = 0; u < U; ++u) for (int l = 0; l < W; ++l) rvl::advance_small(rvl::h_ktab, d[u][l], s[u][l], c[u][l]); }
        else if (!slow && all_mid) { ++st.trips_medium; for (int u = 0; u < U; ++u) for (int l = 0; l < W; ++l) rvl::advance_mid(rvl::h_ktab, d[u][l], s[u][l], c[u][l]); }
        else if (!slow && all_medium) { ++st.trips_medium; for (int u = 0; u < U; ++u) for (int l = 0; l < W; ++l) rvl::advance_medium(rvl::h_ktab, d[u][l], s[u][l], c[u][l]); }
        else {
            ++st.trips_full;
            const bool lib = slow || (trip > 2 && any_big);
            for (int u = 0; u < U; ++u)
                for (int l = 0; l < W; ++l) {
                    if (lib) { s[u][l] = sin(E[u][l]); c[u][l] = cos(E[u][l]); }
                    else rvl::sincos_fast(rvl::h_ktab, E[u][l], s[u][l], c[u][l]);
                }
        }
        bool pa[2][W], any_left = false;
        for (int u = 0; u < U; ++u)
            for (int l = 0; l < W; ++l) {
                pa[u][l] = rvl::abs_gt(d[u][l], rvl::hi32(tol), (uint32_t)rvl::lo32(tol));
                any_left = any_left || pa[u][l];
            }
        if (trip >= itmax || !any_left) break;
        ++trip;
        for (int u = 0; u < U; ++u)
            for (int l = 0; l < W; ++l) {
                double En;
                rvl::newton_step(E[u][l], s[u][l], c[u][l], M[u][l], ec, En);
                En = pa[u][l] ? En : E[u][l];
                d[u][l] = En - E[u][l];
                E[u][l] = En;
                last[u][l] = pa[u][l] ? trip : last[u][l];
            }
    }
    for (int u = 0; u < U; ++u)
        for (int l = 0; l < W; ++l) {
            iters[u][l] += last[u][l];
            caps[l] += (fabs(d[u][l]) > tol) ? 1 : 0;
            out[u][l] = rvl::kepler_rv2(s[u][l], c[u][l], ec, A, Bs, Ce, pc[7]);
        }
}

bool point_setup(const rvl_model_desc &m, const double *row, double *wc)
{
    const int K = m.n_planets;
    bool bad = false;
    for (int p = 0; p < K; ++p) {
        const rvl_planet_desc &pl = m.planet[p];
        double amp = par_of(pl.amp, row);
        if (pl.amp_is_log) amp = rvl::exp_cr(amp);
        double per = par_of(pl.period, row);
        if (pl.period_is_log) per = rvl::exp_cr(per);
        const double a = par_of(pl.e1, row), b = par_of(pl.e2, row);
        double ecc, omega;
        if (pl.ecc_mode == RVL_ECC_SECOS_SESIN) { ecc = a * a + b * b; omega = atan2(b, a); bad = bad || ecc > 1.0; }
        else if (pl.ecc_mode == RVL_ECC_ECOS_ESIN) { ecc = sqrt(a * a + b * b); omega = atan2(b, a); bad = bad || ecc > 1.0; }
        else { ecc = a; omega = b; }
        double M0 = par_of(pl.phase, row);
        if (pl.phase_mode == RVL_PHASE_ML0) M0 = M0 - omega;
        const double ec = ecc > 0.99 ? 0.99 : ecc;
        double sw, cw;
        if (abs_hi(omega) < kHiTrigMax) rvl::sincos_fast(rvl::h_ktab, omega, sw, cw);
        else { sw = sin(omega); cw = cos(omega); }
        const double root = sqrt((1.0 - ec) * (1.0 + ec));
        double *pc = wc + p * kPlanetStride;
        pc[0] = 6.283185307179586 / per;
        pc[1] = M0; pc[2] = ec; pc[3] = amp * cw; pc[4] = -((amp * sw) * root);
        pc[5] = amp * (ecc * cw); pc[6] = par_of(pl.epoch, row); pc[7] = -(pc[3] * ec);
    }
    double *ic = wc + K * kPlanetStride;
    for (int i = 0; i < m.n_inst; ++i) {
        ic[2 * i] = par_of(m.offset[i], row);
        double j2 = 0.0;
        if (m.jitter_in_model) { const double j = par_of(m.jitter[i], row); j2 = j * j; }
        ic[2 * i + 1] = j2;
    }
    double *dc = ic + 2 * m.n_inst;
    for (int l = 0; l < 4; ++l) dc[l] = m.drift_in_model ? par_of(m.drift[l], row) : 0.0;
    for (int l = 0; l < m.n_linpar; ++l) dc[4 + l] = par_of(m.linpar[l], row);
    return !bad;
}

}  // namespace

extern "C" int emul_loglike(const rvl_model_desc *mp, const double *t, const double *rv,
                            const double *err, const int32_t *inst, int N,
                            const double *const *linpar, const double *theta, long long B, int S,
                            int U, double *lnl, long long *stats_out)
{
    if (U != 2) U = 1;
    const rvl_model_desc &m = *mp;
    const int Npad = (N + 31) / 32 * 32, Ctot = Npad / 32, K = m.n_planets;
    if (S < 1) S = 1;
    const int cps = (Ctot + S - 1) / S;
    S = (Ctot + cps - 1) / cps;
    // padded columns exactly as upload_columns() builds them
    const int nlin = m.n_linpar;
    double *ct = (double *)malloc(sizeof(double) * Npad * (4 + nlin));
    double *crv = ct + Npad, *cs2 = ct + 2 * Npad, *ctt = ct + 3 * Npad, *clin = ct + 4 * Npad;
    uint8_t *cid = (uint8_t *)malloc(Npad);
    for (int j = 0; j < Npad; ++j) {
        const int k = j < N ? j : N - 1;
        ct[j] = t[k]; crv[j] = rv[k]; cs2[j] = err[k] * err[k];
        ctt[j] = (t[k] - m.tref) / 365.25;
        for (int l = 0; l < nlin; ++l) clin[(size_t)l * Npad + j] = linpar[l][k];
        cid[j] = (uint8_t)inst[k];
    }
    const double cte = -0.5 * N * log(2 * M_PI);
    Stats st;
    memset(&st, 0, sizeof st);
    double wc[RVL_MAX_PLANETS * kPlanetStride + 2 * RVL_MAX_INST + 4 + RVL_MAX_LINPAR];
    for (long long b = 0; b < B; ++b) {
        const double *row = theta + b * m.ndim;
        const bool valid = point_setup(m, row, wc);
        if (!valid) { lnl[b] = -1e30; continue; }
        const double *ic = wc + K * kPlanetStride, *dc = ic + 2 * m.n_inst;
        double s1 = 0.0, s2 = 0.0;
        for (int sl = 0; sl < S; ++sl) {
            const int c0 = sl * cps, nch = (cps < Ctot - c0) ? cps : Ctot - c0;
            double chi[W], prod[W];
            int esum[W], iters[W], caps[W];
            bool ok[W];
            for (int l = 0; l < W; ++l) { chi[l] = 0; prod[l] = 1; esum[l] = 0; iters[l] = 0; caps[l] = 0; ok[l] = true; }
            for (int ch = 0; ch < nch; ch += U) {
                int j0[2];
                bool have[2];
                const double *tp[2];
                double rvsum[2][W], v[2][W];
                int it_l[2][W], cap_l[W];
                for (int u = 0; u < U; ++u) {
                    have[u] = (ch + u) < nch;
                    j0[u] = (c0 + (have[u] ? ch + u : ch)) * 32;
                    tp[u] = ct + j0[u];
                    for (int l = 0; l < W; ++l) { rvsum[u][l] = 0; it_l[u][l] = 0; }
                }
                for (int l = 0; l < W; ++l) cap_l[l] = 0;
                for (int p = 0; p < K; ++p) {
                    solve_planet_warp(U, tp, wc + p * kPlanetStride, m.tol, m.itmax, v, it_l, cap_l, st);
                    for (int u = 0; u < U; ++u)
                        for (int l = 0; l < W; ++l) rvsum[u][l] = (p == 0) ? v[u][l] : rvsum[u][l] + v[u][l];
                }
                for (int l = 0; l < W; ++l) {
                    caps[l] += cap_l[l];
                    for (int u = 0; u < U; ++u) {
                        const int j = j0[u] + l;
                        const bool live = have[u] && j < N;
                        const int ii = cid[j];
                        double rvm = ic[2 * ii];
                        if (K > 0) rvm = rvm + rvsum[u][l];
                        if (m.drift_in_model) {
                            const double tt = ctt[j], t2 = tt * tt;
                            double dr = dc[0] * tt;
                            dr = dr + dc[1] * t2;
                            dr = dr + dc[2] * (t2 * tt);
                            dr = dr + dc[3] * (t2 * t2);
                            rvm = rvm + dr;
                        }
                        for (int q = 0; q < nlin; ++q) rvm = rvm + dc[4 + q] * clin[(size_t)q * Npad + j];
                        const double res = crv[j] - rvm;
                        const double var = cs2[j] + ic[2 * ii + 1];
                        const double term = (res * res) * rvl::rcp(var + var);
                        double mant; int ex;
                        const bool okv = rvl::split_pos(var, mant, ex);
                        if (live) {
                            chi[l] = chi[l] + term; prod[l] = prod[l] * mant; esum[l] += ex; ok[l] = ok[l] && okv;
                            iters[l] += it_l[u][l];
                        }
                    }
                    if ((ch & 255) == 254 || (ch & 255) == 255) { double mm; int ee; rvl::split_pos(prod[l], mm, ee); prod[l] = mm; esum[l] += ee; }
                }
            }
            bool all_ok = true;
            for (int l = 0; l < W; ++l) all_ok = all_ok && ok[l];
            double S1;
            if (all_ok) {
                for (int l = 0; l < W; ++l) { double mm; int ee; rvl::split_pos(prod[l], mm, ee); prod[l] = mm; esum[l] += ee; }
                for (int o = 16; o > 0; o >>= 1) {  // xor butterfly, as __shfl_xor_sync
                    double nchi[W], nprod[W];
                    for (int l = 0; l < W; ++l) { nchi[l] = chi[l] + chi[l ^ o]; nprod[l] = prod[l] * prod[l ^ o]; }
                    memcpy(chi, nchi, sizeof chi); memcpy(prod, nprod, sizeof prod);
                }
                { int tot = 0; for (int l = 0; l < W; ++l) tot += esum[l]; for (int l = 0; l < W; ++l) esum[l] = tot; }
                double pm;
                int32_t pe, ph;
                rvl::split_pos(prod[0], pm, pe);
                const double lm = rvl::log_mantissa(pm, ph);
                const double es = (double)(esum[0] + pe + ph);
                const double ld = fma(es, rvl::kLn2Hi, fma(es, rvl::kLn2Lo, lm));
                S1 = 0.5 * ld;
            } else {
                double acc[W];
                for (int l = 0; l < W; ++l) acc[l] = 0;
                for (int ch = 0; ch < nch; ++ch)
                    for (int l = 0; l < W; ++l) {
                        const int j = (c0 + ch) * 32 + l;
                        if (j < N) acc[l] = acc[l] + log(sqrt(cs2[j] + ic[2 * cid[j] + 1]));
                    }
                for (int o = 16; o > 0; o >>= 1) {
                    double na[W], nchi[W];
                    for (int l = 0; l < W; ++l) { na[l] = acc[l] + acc[l ^ o]; nchi[l] = chi[l] + chi[l ^ o]; }
                    memcpy(acc, na, sizeof acc); memcpy(chi, nchi, sizeof chi);
                }
                S1 = acc[0];
            }
            for (int l = 0; l < W; ++l) { st.newton_iters += iters[l]; st.caps += caps[l]; }
            if (S == 1) { s1 = S1; s2 = chi[0]; }
            else { s1 = s1 + S1; s2 = s2 + chi[0]; }
        }
        lnl[b] = (cte - s1) - s2;
    }
    if (stats_out) {
        stats_out[0] = st.trips_full; stats_out[1] = st.trips_small; stats_out[2] = st.trips_tiny;
        stats_out[3] = st.solves_warp; stats_out[4] = st.newton_iters; stats_out[5] = st.caps;
        stats_out[6] = st.trips_medium;
    }
    free(ct); free(cid);
    return 0;
}

// sin/cos core against libm, for a range of arguments: returns max abs error
extern "C" double emul_sincos_maxerr(const double *x, int n)
{
    double worst = 0;
    for (int i = 0; i < n; ++i) {
        double s, c;
        rvl::sincos_fast(rvl::h_ktab, x[i], s, c);
        const double es = fabs(s - sin(x[i])), ecs = fabs(c - cos(x[i]));
        if (es > worst) worst = es;
        if (ecs > worst) worst = ecs;
    }
    return worst;
}

extern "C" double emul_rcp(double x) { return rvl::rcp(x); }
extern "C" void emul_exp_cr(const double *x, int n, double *y) { for (int i = 0; i < n; ++i) y[i] = rvl::exp_cr(x[i]); }
