// ekf_fast_api.cuh -- the seam between the library's two translation units.
//
// nuslam_b200.cu (the C ABI, the oracle-order, scan, simulator and large-map kernels) is compiled whole-program; ekf_fast_tu.cu (the FAST
// filter kernels and the list kernel they hand filters to) is compiled as relocatable device code and linked against the device runtime,
// because those kernels launch the list kernel themselves (ekf_strict.cuh strict_tail). Relocatable code costs the other kernels time
// (ABI calls into the math library's slow paths, constant tables behind relocations: closed loop +15 %, scan kernel +7 %, measured),
// so only the kernels that need it are built that way.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include "ekf_strict.cuh"

namespace nuslam
{

constexpr int kFastMMax = 16;   // measurements per step handled by the FAST kernels
inline bool fast_supported(int n) { return n >= 1 && n <= 12; }

// Known correspondence at the BASELINE map size is served by the resident pair kernel (ekf_res2.cuh). NUSLAM_KERNEL=fast hands it to
// the register-fragment kernel (ekf_fast.cuh, which serves everything else) for A/B timing and the agreement test; unset or any other
// value: the resident pair kernel. Read at every call, so that a process can switch between the two.
inline bool force_fast_kernel()
{
    const char * e = getenv("NUSLAM_KERNEL");
    return e && strcmp(e, "fast") == 0;
}

struct FastLaunch
{
    int n_landmarks, sm_count;
    int64_t batch;
    int32_t * worklist;
    int32_t * wl_count;   // [0] entries, [1] finished blocks of the list kernel, [2] finished warps of the FAST kernel, [3] device-launch error
    cudaStream_t stream;
    int strict_warps;     // launch shape of the list kernel
    size_t strict_smem;   // per warp, bytes
};

// One FAST-mode call: the register / resident kernel over the batch, then k_ekf_strict_list over the filters it handed over (launched by
// the kernel itself when the library is built with tail launches, else from here). op: kOpStep or kOpUpdate.
// Returns 0, or -1 when the configuration is not covered (the caller runs the oracle-order kernel over the batch), or 1 with *err / *where
// set when a CUDA call failed.
int fast_path_launch(const FastLaunch & fl, const EkfParams & p, bool do_predict, int op, cudaError_t * err, const char ** where);

// 1 when the FAST kernels launch the list kernel themselves (built with -rdc=true, not switched off by NUSLAM_NO_TAIL_LAUNCH)
int tail_launch_active();

// kernel-experiment builds (-DNUSLAM_TIMING): per-phase clock64 sums of block 0 / warp 0 of the FAST kernel
int fast_timing_read(long long * out16, int reset);

}   // namespace nuslam
