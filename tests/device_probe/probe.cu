// probe.cu — TEST HARNESS ONLY: runs the operations of ops.h on the device, one thread per argument,
// with the coefficient table loaded by rvl::load_ktab() or rvl::load_ktab_pinned() and the sin/cos
// table read from shared memory through rvl::SmemSinTab, as the likelihood kernel reads them.
#include <cuda_runtime.h>
#include <stdint.h>

#include "ops.h"

namespace {

template <bool kPinned>
__global__ void __launch_bounds__(256) probe_kernel(int op, long long n, const double *in, double *out)
{
    // the likelihood kernel's table: hi rows, then lo rows, copied with plain loads
    __shared__ __align__(16) unsigned char s_tab[2 * sizeof(rvl::g_sintab_hi)];
    {
        const uint4 *hi = reinterpret_cast<const uint4 *>(rvl::g_sintab_hi);
        const uint4 *lo = reinterpret_cast<const uint4 *>(rvl::g_sintab_lo);
        uint4 *dst = reinterpret_cast<uint4 *>(s_tab);
        constexpr int nhi = (int)(sizeof(rvl::g_sintab_hi) / 16), nall = 2 * nhi;
        for (int i = threadIdx.x; i < nall; i += blockDim.x) dst[i] = i < nhi ? hi[i] : lo[i - nhi];
        __syncthreads();
    }
    const rvl::SmemSinTab tab{(uint32_t)__cvta_generic_to_shared(s_tab)};
    const rvl::KTab kt = kPinned ? rvl::load_ktab_pinned() : rvl::load_ktab();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double a[probe::kIn], r[probe::kOut];
#pragma unroll
    for (int k = 0; k < probe::kIn; ++k) a[k] = in[i * probe::kIn + k];
    probe::run_op(op, kt, tab, a, r);
#pragma unroll
    for (int k = 0; k < probe::kOut; ++k) out[i * probe::kOut + k] = r[k];
}

}  // namespace

// in: [n][kIn] doubles, out: [n][kOut] doubles, both in host memory.  Returns 0, or the CUDA error.
extern "C" int probe_run(int op, int pinned, const double *in, double *out, long long n)
{
    if (op < 0 || op >= probe::kNumOps || n < 0) return (int)cudaErrorInvalidValue;
    if (n == 0) return 0;
    const size_t bin = (size_t)n * probe::kIn * sizeof(double), bout = (size_t)n * probe::kOut * sizeof(double);
    double *din = nullptr, *dout = nullptr;
    cudaError_t err = cudaMalloc(&din, bin);
    if (err == cudaSuccess) err = cudaMalloc(&dout, bout);
    if (err == cudaSuccess) err = cudaMemcpy(din, in, bin, cudaMemcpyHostToDevice);
    if (err == cudaSuccess) {
        const int threads = 256;
        const unsigned blocks = (unsigned)((n + threads - 1) / threads);
        if (pinned) probe_kernel<true><<<blocks, threads>>>(op, n, din, dout);
        else probe_kernel<false><<<blocks, threads>>>(op, n, din, dout);
        err = cudaGetLastError();
    }
    if (err == cudaSuccess) err = cudaDeviceSynchronize();
    if (err == cudaSuccess) err = cudaMemcpy(out, dout, bout, cudaMemcpyDeviceToHost);
    cudaFree(dout);  // (cudaFree(nullptr) is a no-op)
    cudaFree(din);
    return (int)err;
}
