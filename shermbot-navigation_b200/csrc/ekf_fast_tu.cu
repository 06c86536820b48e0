// ekf_fast_tu.cu -- the FAST filter kernels and their launcher, built as relocatable device code (see ekf_fast_api.cuh).
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define NUSLAM_TU_FAST 1
#include "nuslam_b200.h"
#include "ekf_common.cuh"
#include "ekf_strict.cuh"
#include "ekf_fast_api.cuh"
#include "ekf_fast.cuh"
#include "ekf_res2.cuh"

namespace nuslam
{

int tail_launch_active()
{
    static const int on = (NUSLAM_TAIL_LAUNCH && getenv("NUSLAM_NO_TAIL_LAUNCH") == nullptr) ? 1 : 0;   // the switch is for A/B timing
    return on;
}

namespace
{
template <int OP>
int fast_path(const FastLaunch & fl, const EkfParams & p_in, bool do_predict, cudaError_t * err, const char ** where)
{
    // known correspondence at the BASELINE map size: the resident pair kernel (ekf_res2.cuh; NUSLAM_KERNEL=fast selects ekf_fast.cuh for
    // A/B timing); everything else: ekf_fast.cuh
    const bool res2 = !force_fast_kernel() && res2_supported(fl.n_landmarks, p_in);
    const int warps = fl.strict_warps;
    const size_t smem = fl.strict_smem * warps;
    static size_t configured_dev[kMaxDevices][8] = {{0}};
    size_t * configured = configured_dev[device_slot()];
    if (configured[OP] < smem)
    {
        *err = cudaFuncSetAttribute(k_ekf_strict_list<OP, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
        if (*err != cudaSuccess)
        {
            *where = "cudaFuncSetAttribute(k_ekf_strict_list)";
            return 1;
        }
        configured[OP] = smem;
    }
    int64_t blocks = (fl.batch + warps - 1) / warps;
    const int64_t resident = (int64_t) fl.sm_count * 4;
    if (blocks > resident) blocks = resident;
    // the resident pair kernel and the register-fragment kernel launch the list kernel themselves, behind their own grid and only when a
    // filter was handed over (ekf_strict.cuh strict_tail): a step of a built map is one launch
    const bool tail = tail_launch_active() && smem <= 48 * 1024;
    EkfParams p = p_in;
    if (tail)
    {
        p.tail_blocks = (int) blocks;
        p.tail_threads = warps * 32;
        p.tail_smem = (int) smem;
    }
    const int rc = res2 ? launch_res2_n<12>(p, do_predict, fl.sm_count, fl.worklist, fl.wl_count, fl.stream)
                        : launch_fast(fl.n_landmarks, p, do_predict, fl.sm_count, fl.worklist, fl.wl_count, fl.stream);
    // not covered by the FAST kernels (more than 16 measurements per step, ragged counts with known ids, a state pointer that is not
    // 8-byte aligned): the caller runs the oracle-order kernel over the whole batch
    if (rc == -1) return -1;
    if (rc)
    {
        *err = (cudaError_t) rc;
        *where = "fast kernel launch";
        return 1;
    }
    if (tail) return 0;
    k_ekf_strict_list<OP, 1><<<(unsigned) blocks, warps * 32, smem, fl.stream>>>(p, fl.worklist, fl.wl_count, fl.wl_count + 1);
    const cudaError_t le = cudaGetLastError();
    if (le != cudaSuccess)
    {
        // the list kernel resets the counters itself when it runs; it did not: the next call must not replay this call's entries
        cudaMemsetAsync(fl.wl_count, 0, sizeof(int32_t) * 2, fl.stream);
        *err = le;
        *where = "strict list kernel launch";
        return 1;
    }
    return 0;
}
}   // namespace

int fast_path_launch(const FastLaunch & fl, const EkfParams & p, bool do_predict, int op, cudaError_t * err, const char ** where)
{
    return op == kOpStep ? fast_path<kOpStep>(fl, p, do_predict, err, where) : fast_path<kOpUpdate>(fl, p, do_predict, err, where);
}

int fast_timing_read(long long * out16, int reset)
{
#ifdef NUSLAM_TIMING
    if (out16) cudaMemcpyFromSymbol(out16, g_fast_timing, sizeof(long long) * 16);
    if (reset)
    {
        long long z[16] = {0};
        cudaMemcpyToSymbol(g_fast_timing, z, sizeof(z));
    }
    return 0;
#else
    (void) out16;
    (void) reset;
    return -1;
#endif
}

}   // namespace nuslam
