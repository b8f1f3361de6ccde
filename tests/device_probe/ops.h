// ops.h — TEST HARNESS ONLY: the FP64 core of the likelihood kernel (evidence_b200/csrc/rvl_math.h,
// rvl_lean.h), one operation per call, for the device probe (probe.cu) and its host build
// (host.cpp).  Each function calls the core exactly as rvlnl.cu does, so the two builds of this file
// run the kernel's arithmetic: tests/test_math_core_host.py checks the host build against mpmath,
// tests/test_gpu_math_core.py the device build against the host build and against mpmath.
//
// Every operation reads kIn doubles of one argument and writes kOut doubles of its result.
#pragma once
#include "../../evidence_b200/csrc/rvl_lean.h"
#include "../../evidence_b200/csrc/rvl_math.h"

namespace probe {

constexpr int kIn = 8, kOut = 4;

// operation ids (tests/_probe.py keeps the same list)
enum Op : int {
    kSincosTab = 0,    // x -> s, c
    kSincosFast,       // x -> s, c
    kAdvanceFinal,     // s, c, d -> s', c'
    kAdvanceTiny,
    kAdvanceSmall,
    kAdvanceMid,
    kAdvanceMedium,
    kChain,            // s, c, d, q, k -> s', c' after k advances by d, d q, d q^2, ...
    kRcpSeed,          // x -> y
    kRcp,              // x -> y
    kNewtonStep,       // E, s, c, M, ec -> E_new, d
    kKeplerRv2,        // s, c, ec, A, Bs, Ce, mAec -> rv
    kLogMantissa,      // m -> ln, half
    kExpCr,            // x -> y
    kSplitPos,         // v -> mant, expo, valid
    kSplitRaw,         // v -> mant, be
    kMeanAnomaly,      // nmot, t, epoch, M0 -> M
    kNumOps
};

RVL_HD int abs_hi(double x) { return rvl::hi32(x) & 0x7fffffff; }

// the series the lean loop (rvlnl.cu, solve_planet) advances by for a step of size |d|: the
// thresholds of rvl_lean.h, and the final series wherever it holds (|d| < 2e-4; the loop takes it
// on its last pass, when every |d| is below the tolerance)
RVL_HD void advance_as_loop(const rvl::KTab &kt, double d, double &s, double &c)
{
    const int h = abs_hi(d);
    if (h < rvl::kHiFinal) rvl::advance_final(kt, d, s, c);
    else if (h < rvl::kHiTiny) rvl::advance_tiny(kt, d, s, c);
    else if (h < rvl::kHiSmall) rvl::advance_small(kt, d, s, c);
    else if (h < rvl::kHiMid) rvl::advance_mid(kt, d, s, c);
    else rvl::advance_medium(kt, d, s, c);
}

template <class Tab>
RVL_HD void run_op(int op, const rvl::KTab &kt, const Tab &tab, const double *in, double *out)
{
    for (int i = 0; i < kOut; ++i) out[i] = 0.0;
    double s = in[0], c = in[1];
    switch (op) {
    case kSincosTab: rvl::sincos_tab(kt, tab, in[0], out[0], out[1]); return;
    case kSincosFast: rvl::sincos_fast(kt, in[0], out[0], out[1]); return;
    case kAdvanceFinal: rvl::advance_final(kt, in[2], s, c); break;
    case kAdvanceTiny: rvl::advance_tiny(kt, in[2], s, c); break;
    case kAdvanceSmall: rvl::advance_small(kt, in[2], s, c); break;
    case kAdvanceMid: rvl::advance_mid(kt, in[2], s, c); break;
    case kAdvanceMedium: rvl::advance_medium(kt, in[2], s, c); break;
    case kChain: {
        double d = in[2];
        const int k = (int)in[4];
        for (int i = 0; i < k; ++i) {
            advance_as_loop(kt, d, s, c);
            d = rvl::mul(d, in[3]);
        }
        break;
    }
    case kRcpSeed: out[0] = rvl::rcp_seed(in[0]); return;
    case kRcp: out[0] = rvl::rcp(in[0]); return;
    case kNewtonStep: out[1] = rvl::newton_step(in[0], in[1], in[2], in[3], in[4], out[0]); return;
    case kKeplerRv2: out[0] = rvl::kepler_rv2(in[0], in[1], in[2], in[3], in[4], in[5], in[6]); return;
    case kLogMantissa: {
        int32_t half;
        out[0] = rvl::log_mantissa(in[0], half);
        out[1] = half;
        return;
    }
    case kExpCr: out[0] = rvl::exp_cr(in[0]); return;
    case kSplitPos: {
        int32_t expo;
        out[2] = rvl::split_pos(in[0], out[0], expo) ? 1.0 : 0.0;
        out[1] = expo;
        return;
    }
    case kSplitRaw: {
        uint32_t be;
        rvl::split_raw(in[0], out[0], be);
        out[1] = be;
        return;
    }
    case kMeanAnomaly: out[0] = rvl::mean_anomaly(in[0], in[1], in[2], in[3]); return;
    default: out[0] = out[1] = out[2] = out[3] = -1.0; return;
    }
    out[0] = s;
    out[1] = c;
}

}  // namespace probe
