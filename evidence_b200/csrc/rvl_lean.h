// rvl_lean.h — what the lean Newton loop of rvlnl.cu shares with the code that replays or probes it:
// the thresholds that pick the sin/cos path of a pass, and (device only) the sin/cos table of
// rvl::sincos_tab and its shared-memory accessor.  One copy, included by the kernel source, the host
// replays (tests/host_emul) and the device probe (tests/device_probe).
#pragma once
#include "rvl_math.h"

namespace rvl {

// high words of |x| as integers order like |x| itself (positive doubles sort as integers)
constexpr int kHiTrigMax = 0x40F86A00;  // 1e5 = 0x40F86A0000000000: |x| < 1e5  <=>  abs_hi < this
constexpr int kHiTiny = 0x3F500000;     // abs_hi(d) <  this  <=>  |d| <  2^-10
constexpr int kHiSmall = 0x3FA00000;    // abs_hi(d) <  this  <=>  |d| <  2^-5
constexpr int kHiMid = 0x3FC00000;      // abs_hi(d) <  this  <=>  |d| <  2^-3
constexpr int kHiMedium = 0x3FE80000;   // abs_hi(d) <  this  <=>  |d| <  0.75

#if defined(__CUDACC__)
// ---- the sin/cos table of rvl::sincos_tab (rvl_sintab.h) ---------------------------------------
// In global memory as two arrays, the (sin, cos) hi parts and then the lo parts; every block that
// runs the lean Newton loop copies both into its shared memory once, and the loop reads them
// through SmemSinTab.  Two arrays rather than one of whole rows: a 16-byte load of rows with a
// 16-byte stride spreads 32 random rows over twice the banks that a 32-byte stride would.
__device__ const double2 g_sintab_hi[kSinTabN] = {RVL_SINTAB(RVL_SINTAB_HI_ROW)};
__device__ const double2 g_sintab_lo[kSinTabN] = {RVL_SINTAB(RVL_SINTAB_LO_ROW)};

struct SmemSinTab {
    uint32_t hi;  // shared-window address of the hi rows; the lo rows follow them
    __device__ __forceinline__ TabRow operator()(int32_t j) const
    {
        // (not volatile: the table does not change once it is in shared memory, so the loads
        // may be scheduled like arithmetic)
        TabRow t;
        // one address for both loads (left to itself the compiler shifts, masks and adds)
        uint32_t a;
        asm("mad.lo.u32 %0, %1, 16, %2;" : "=r"(a) : "r"(j), "r"(hi));
        asm("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(t.sh), "=d"(t.ch) : "r"(a));
        asm("ld.shared.v2.f64 {%0, %1}, [%2+16384];" : "=d"(t.sl), "=d"(t.cl) : "r"(a));
        return t;
    }
};
static_assert(sizeof(g_sintab_hi) == 16384, "SmemSinTab addresses the lo rows at +16384");
#endif

}  // namespace rvl
