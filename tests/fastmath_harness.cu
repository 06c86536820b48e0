// fastmath_harness.cu -- element-wise evaluation of the fast-math primitives of csrc/fastmath.cuh (and of scan_moment.cuh's copy of
// atan2_fast on shared-memory tables) over device arrays, for tests/test_fastmath_gpu.py. The headers are included as they are: this
// file holds no copy of a primitive. One kernel and one extern "C" launcher per primitive; the launchers take device pointers and a
// count, run on the default stream and return the launch's cudaError_t.
#include "fastmath.cuh"
#include "scan_moment.cuh"

namespace
{

constexpr int kThreads = 256;

inline unsigned blocks_for(long n) { return (unsigned) ((n + kThreads - 1) / kThreads); }

__global__ void k_rcp_fast(const double * x, double * out, long n)
{
    for (long i = blockIdx.x * (long) blockDim.x + threadIdx.x; i < n; i += (long) gridDim.x * blockDim.x) out[i] = nuslam::rcp_fast(x[i]);
}

__global__ void k_div_fast(const double * a, const double * b, double * out, long n)
{
    for (long i = blockIdx.x * (long) blockDim.x + threadIdx.x; i < n; i += (long) gridDim.x * blockDim.x) out[i] = nuslam::div_fast(a[i], b[i]);
}

__global__ void k_rsqrt_fast(const double * x, double * out, long n)
{
    for (long i = blockIdx.x * (long) blockDim.x + threadIdx.x; i < n; i += (long) gridDim.x * blockDim.x) out[i] = nuslam::rsqrt_fast(x[i]);
}

__global__ void k_rsqrt_1(const double * x, double * out, long n)
{
    for (long i = blockIdx.x * (long) blockDim.x + threadIdx.x; i < n; i += (long) gridDim.x * blockDim.x) out[i] = nuslam::rsqrt_1(x[i]);
}

__global__ void k_wrap_angle(const double * a, double * out, long n)
{
    for (long i = blockIdx.x * (long) blockDim.x + threadIdx.x; i < n; i += (long) gridDim.x * blockDim.x) out[i] = nuslam::wrap_angle(a[i]);
}

__global__ void k_atan2_fast(const double * y, const double * x, double * out, long n)
{
    for (long i = blockIdx.x * (long) blockDim.x + threadIdx.x; i < n; i += (long) gridDim.x * blockDim.x) out[i] = nuslam::atan2_fast(y[i], x[i]);
}

__global__ void k_atan2_unit(const double * y, const double * x, const double * rs, double * out, long n)
{
    for (long i = blockIdx.x * (long) blockDim.x + threadIdx.x; i < n; i += (long) gridDim.x * blockDim.x)
        out[i] = nuslam::atan2_unit(y[i], x[i], rs[i]);
}

// the tables filled as k_scan_moment fills them
__global__ void k_atan2_tab(const double * y, const double * x, double * out, long n)
{
    __shared__ __align__(16) nuslam::MomentTables tabs;
    for (int k = threadIdx.x; k < 65 + 16; k += blockDim.x)
    {
        if (k < 65) tabs.tab[k] = nuslam::kAtanTab[k];
        else reinterpret_cast<double2 *>(tabs.oct)[k - 65] = reinterpret_cast<const double2 *>(nuslam::kAtanOct)[k - 65];
    }
    __syncthreads();
    for (long i = blockIdx.x * (long) blockDim.x + threadIdx.x; i < n; i += (long) gridDim.x * blockDim.x)
        out[i] = nuslam::atan2_tab(y[i], x[i], tabs);
}

__global__ void k_sincos_fast(const double * a, double * s, double * c, long n)
{
    for (long i = blockIdx.x * (long) blockDim.x + threadIdx.x; i < n; i += (long) gridDim.x * blockDim.x) nuslam::sincos_fast(a[i], s + i, c + i);
}

__global__ void k_sincos_small(const double * a, double * s, double * c, long n)
{
    for (long i = blockIdx.x * (long) blockDim.x + threadIdx.x; i < n; i += (long) gridDim.x * blockDim.x) nuslam::sincos_small(a[i], s + i, c + i);
}

}   // namespace

extern "C" {

int fm_rcp_fast(const double * x, double * out, long n) { k_rcp_fast<<<blocks_for(n), kThreads>>>(x, out, n); return (int) cudaGetLastError(); }
int fm_div_fast(const double * a, const double * b, double * out, long n) { k_div_fast<<<blocks_for(n), kThreads>>>(a, b, out, n); return (int) cudaGetLastError(); }
int fm_rsqrt_fast(const double * x, double * out, long n) { k_rsqrt_fast<<<blocks_for(n), kThreads>>>(x, out, n); return (int) cudaGetLastError(); }
int fm_rsqrt_1(const double * x, double * out, long n) { k_rsqrt_1<<<blocks_for(n), kThreads>>>(x, out, n); return (int) cudaGetLastError(); }
int fm_wrap_angle(const double * a, double * out, long n) { k_wrap_angle<<<blocks_for(n), kThreads>>>(a, out, n); return (int) cudaGetLastError(); }
int fm_atan2_fast(const double * y, const double * x, double * out, long n) { k_atan2_fast<<<blocks_for(n), kThreads>>>(y, x, out, n); return (int) cudaGetLastError(); }
int fm_atan2_unit(const double * y, const double * x, const double * rs, double * out, long n)
{
    k_atan2_unit<<<blocks_for(n), kThreads>>>(y, x, rs, out, n);
    return (int) cudaGetLastError();
}
int fm_atan2_tab(const double * y, const double * x, double * out, long n) { k_atan2_tab<<<blocks_for(n), kThreads>>>(y, x, out, n); return (int) cudaGetLastError(); }
int fm_sincos_fast(const double * a, double * s, double * c, long n) { k_sincos_fast<<<blocks_for(n), kThreads>>>(a, s, c, n); return (int) cudaGetLastError(); }
int fm_sincos_small(const double * a, double * s, double * c, long n) { k_sincos_small<<<blocks_for(n), kThreads>>>(a, s, c, n); return (int) cudaGetLastError(); }

}
