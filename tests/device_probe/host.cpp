// host.cpp — TEST HARNESS ONLY: the operations of ops.h compiled for the host (g++ -ffp-contract=off),
// with the host copies of the coefficient and sin/cos tables.  Same interface as probe.cu's probe_run.
#include "ops.h"

extern "C" int host_run(int op, const double *in, double *out, long long n)
{
    if (op < 0 || op >= probe::kNumOps || n < 0) return 1;
    const rvl::HostSinTab tab{};
    for (long long i = 0; i < n; ++i) probe::run_op(op, rvl::h_ktab, tab, in + i * probe::kIn, out + i * probe::kOut);
    return 0;
}
