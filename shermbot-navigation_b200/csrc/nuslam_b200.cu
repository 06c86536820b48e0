// nuslam_b200.cu -- C ABI (include/nuslam_b200.h) over the sm_100a kernels.
//
// Host side of the drop-in boundary: owns device memory, streams and staging, validates arguments and
// launches the kernels in ekf_strict.cuh / ekf_fast.cuh / scan_detect.cuh. No CPU arithmetic path exists
// here: without a CUDA device every compute entry point fails with NUSLAM_ERR_CUDA.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <new>
#include <string>

#include "nuslam_b200.h"
#include "ekf_common.cuh"
#include "ekf_strict.cuh"
#include "ekf_misc.cuh"
#include "ekf_fast_api.cuh"   // the known-correspondence FAST kernels live in ekf_fast_tu.cu (relocatable device code: they launch the list kernel themselves)
#include "ekf_fast.cuh"       // on-device association: the register-fragment kernel of this unit (whole-program build, internal linkage)
#include "scan_moment.cuh"
#include "scan_detect.cuh"
#include "ekf_large.cuh"
#include "world_sim.cuh"

namespace
{

thread_local std::string g_last_error;

int fail(int code, const char * what)
{
    g_last_error = what;
    return code;
}

int cuda_fail(cudaError_t e, const char * where)
{
    char buf[512];
    snprintf(buf, sizeof(buf), "%s: %s", where, cudaGetErrorString(e));
    g_last_error = buf;
    return NUSLAM_ERR_CUDA;
}

#define CU(call)                                              \
    do                                                        \
    {                                                         \
        cudaError_t e_ = (call);                              \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call);   \
    } while (0)

// grow-only device scratch buffer
struct DevBuf
{
    void * p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes)
    {
        if (bytes <= cap) return NUSLAM_OK;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(staging)");
        cap = bytes;
        return NUSLAM_OK;
    }
    void release()
    {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

}   // namespace

struct nuslam_ekf
{
    nuslam_ekf_config cfg;
    int64_t batch = 0;
    int len = 0;
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 0;
    // state
    double * x = nullptr;
    double * sigma = nullptr;
    int32_t * seen = nullptr;
    int32_t * status = nullptr;
    bool own_state = true;
    // staging for NUSLAM_HOST calls
    DevBuf s_tw, s_z, s_ids, s_ids_out, s_misc;
    // fused scan step (nuslam_ekf_scan_step): ranges staging, detection outputs, measurements
    DevBuf f_ranges, f_ncl, f_nci, f_circ, f_z, f_mv;
    // FAST mode: filters whose step contains a first touch are handed to the strict kernel through this list
    // pipelined host-buffer steps (nuslam_ekf_step_async): kAsyncSlots slots of staged inputs / state snapshots, copy streams, events
    struct AsyncSlot
    {
        DevBuf tw, z, ids, xsnap;
        cudaEvent_t h2d_done = nullptr, kernel_done = nullptr, d2h_done = nullptr;
        bool busy = false;
    } slots[3];
    cudaStream_t s_in = nullptr, s_out = nullptr;
    uint64_t async_count = 0;
    DevBuf ids_cache;          // nuslam_ekf_set_ids: B x ids_cache_m known-correspondence ids kept on the device
    int32_t ids_cache_m = 0;
    bool async_dry = false;   // nuslam_ekf_async_dry_run: step_async performs its copies and event chaining, no kernel (copy ceiling)
    // LARGE-MAP mode (state too long for the on-chip batched kernels): delayed-update scratch, see ekf_large.cuh
    bool large = false;
    double * lg_x2 = nullptr;
    double * lg_U = nullptr;
    double * lg_V = nullptr;
    double * lg_P = nullptr;
    int32_t * lg_seen_snap = nullptr;
    DevBuf lg_ids_slot, lg_assoc_result;   // unknown correspondence in large-map mode
    DevBuf lg_nn_slots;                    // NUSLAM_OPT_NEAREST_NEIGHBOUR in large-map mode: B x ceil(n / 128) CTA minima
    double * x_snap_next = nullptr;        // pipelined host path: where the next step's kernels also write the state vector
    int32_t * worklist = nullptr;   // batch entries
    int32_t * wl_count = nullptr;   // [0] = entries, [1] = finished blocks of the list kernel, [2] finished warps of the FAST kernel, [3] device-launch error
    size_t strict_smem = 0;   // per-warp shared memory of the strict kernels, bytes
    int strict_warps = 4;
    DevBuf joint_t;           // NUSLAM_OPT_JOINT_COMPATIBILITY: T[0..kJcbbMMax], the joint thresholds
};

namespace
{

int select_device(const nuslam_ekf * h)
{
    CU(cudaSetDevice(h->device));
    return NUSLAM_OK;
}

// copy `bytes` from a user pointer (host or device) into a staging buffer when it lives on the host
template <typename T>
int stage_in(nuslam_ekf * h, DevBuf & buf, const T * user, size_t count, int mem, const T ** dev_out)
{
    if (!user)
    {
        *dev_out = nullptr;
        return NUSLAM_OK;
    }
    if (mem == NUSLAM_DEVICE)
    {
        *dev_out = user;
        return NUSLAM_OK;
    }
    int rc = buf.reserve(count * sizeof(T));
    if (rc) return rc;
    CU(cudaMemcpyAsync(buf.p, user, count * sizeof(T), cudaMemcpyHostToDevice, h->stream));
    *dev_out = static_cast<const T *>(buf.p);
    return NUSLAM_OK;
}

nuslam::EkfParams make_params(nuslam_ekf * h)
{
    nuslam::EkfParams p;
    memset(&p, 0, sizeof(p));
    p.batch = h->batch;
    p.len = h->len;
    p.n = h->cfg.n_landmarks;
    p.m = 0;
    p.x = h->x;
    p.sigma = h->sigma;
    p.seen = h->seen;
    p.status = h->status;
    memcpy(p.Q, h->cfg.Q, sizeof(p.Q));
    memcpy(p.R, h->cfg.R, sizeof(p.R));
    p.amin = h->cfg.assoc_min;
    p.amax = h->cfg.assoc_max;
    p.options = h->cfg.options;
    p.x_snap = h->x_snap_next;
    p.joint_t = static_cast<const double *>(h->joint_t.p);
    return p;
}

// NUSLAM_OPT_JOINT_COMPATIBILITY: T[p] = chi2_{2p}^-1(conf), conf = 1 - exp(-amin / 2), so T[1] = amin. Bisection on the survival function
// of chi2 at even degrees of freedom, exp(-x/2) sum_{i<p} (x/2)^i / i!, which falls strictly in x.
void joint_thresholds(double amin, double * T)
{
    const double q = exp(-0.5 * amin);
    T[0] = 0.0;
    T[1] = amin;
    for (int p = 2; p <= nuslam::kJcbbMMax; ++p)
    {
        auto sf = [p](double x) {
            double t = 1.0, s = 1.0;
            for (int i = 1; i < p; ++i)
            {
                t *= 0.5 * x / i;
                s += t;
            }
            return exp(-0.5 * x) * s;
        };
        double lo = T[p - 1], hi = 2.0 * lo + 8.0;
        while (sf(hi) > q && hi < 1e300) hi *= 2.0;
        for (int it = 0; it < 2000; ++it)
        {
            const double mid = 0.5 * (lo + hi);
            if (!(mid > lo && mid < hi)) break;
            if (sf(mid) > q) lo = mid;
            else hi = mid;
        }
        T[p] = hi;
    }
}

// NUSLAM_OPT_JOINT_COMPATIBILITY searches at most kJcbbMMax measurements per step (checked before any work of a step is enqueued)
int joint_m_check(const nuslam_ekf * h, bool unknown_ids, int m)
{
    if ((h->cfg.options & NUSLAM_OPT_JOINT_COMPATIBILITY) && unknown_ids && m > nuslam::kJcbbMMax)
        return fail(NUSLAM_ERR_UNSUPPORTED, "NUSLAM_OPT_JOINT_COMPATIBILITY associates at most 16 measurements per step");
    return NUSLAM_OK;
}

template <int OP>
int launch_strict(nuslam_ekf * h, const nuslam::EkfParams & p)
{
    const int warps = h->strict_warps;
    const size_t smem = h->strict_smem * warps;
    static size_t configured_dev[nuslam::kMaxDevices][8] = {{0}};
    size_t * configured = configured_dev[nuslam::device_slot()];
    if (configured[OP] < smem)
    {
        CU(cudaFuncSetAttribute(nuslam::k_ekf_strict<OP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
        configured[OP] = smem;
    }
    const int64_t blocks = (h->batch + warps - 1) / warps;
    nuslam::k_ekf_strict<OP><<<(unsigned) blocks, warps * 32, smem, h->stream>>>(p);
    CU(cudaGetLastError());
    return NUSLAM_OK;
}

// FAST mode: the register / resident kernel, then the strict kernel over the filters it handed over (usually none).
// Known correspondence: ekf_fast_tu.cu -- the kernel launches the list kernel itself, one launch per step of a built map.
// On-device association (ids == NULL): this unit's whole-program build of ekf_fast.cuh + a host launch of the list kernel (the
// relocatable build costs the association kernel 1.5 %, and with unknown correspondence hand-overs -- new landmarks -- are frequent:
// closed loop 0.62 against 0.56 ms per step, measured).
template <int OP>
int launch_fast_then_strict(nuslam_ekf * h, const nuslam::EkfParams & p, bool do_predict)
{
    if (p.ids == nullptr)
    {
        const int rc = nuslam::launch_fast(h->cfg.n_landmarks, p, do_predict, h->sm_count, h->worklist, h->wl_count, h->stream);
        if (rc == -1) return launch_strict<OP>(h, p);
        if (rc) return cuda_fail((cudaError_t) rc, "fast kernel launch");
        const int warps = h->strict_warps;
        const size_t smem = h->strict_smem * warps;
        static size_t configured_dev[nuslam::kMaxDevices][8] = {{0}};
        size_t * configured = configured_dev[nuslam::device_slot()];
        if (configured[OP] < smem)
        {
            CU(cudaFuncSetAttribute(nuslam::k_ekf_strict_list<OP, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
            configured[OP] = smem;
        }
        int64_t blocks = (h->batch + warps - 1) / warps;
        const int64_t resident = (int64_t) h->sm_count * 4;
        if (blocks > resident) blocks = resident;
        nuslam::k_ekf_strict_list<OP, 0><<<(unsigned) blocks, warps * 32, smem, h->stream>>>(p, h->worklist, h->wl_count, h->wl_count + 1);
        const cudaError_t le = cudaGetLastError();
        if (le != cudaSuccess)
        {
            // the list kernel resets the counters itself when it runs; it did not: the next call must not replay this call's entries
            cudaMemsetAsync(h->wl_count, 0, sizeof(int32_t) * 2, h->stream);
            return cuda_fail(le, "strict list kernel launch");
        }
        return NUSLAM_OK;
    }
    nuslam::FastLaunch fl;
    fl.n_landmarks = h->cfg.n_landmarks;
    fl.sm_count = h->sm_count;
    fl.batch = h->batch;
    fl.worklist = h->worklist;
    fl.wl_count = h->wl_count;
    fl.stream = h->stream;
    fl.strict_warps = h->strict_warps;
    fl.strict_smem = h->strict_smem;
    cudaError_t err = cudaSuccess;
    const char * where = "";
    const int rc = nuslam::fast_path_launch(fl, p, do_predict, OP, &err, &where);
    if (rc == -1) return launch_strict<OP>(h, p);
    if (rc) return cuda_fail(err, where);
    return NUSLAM_OK;
}

nuslam::LargeParams make_large_params(nuslam_ekf * h)
{
    nuslam::LargeParams p;
    memset(&p, 0, sizeof(p));
    p.batch = h->batch;
    p.len = h->len;
    p.n = h->cfg.n_landmarks;
    p.x = h->x;
    p.x2 = h->lg_x2;
    p.sigma = h->sigma;
    p.U = h->lg_U;
    p.V = h->lg_V;
    p.P = h->lg_P;
    p.status = h->status;
    p.strict_from = h->lg_seen_snap ? h->lg_seen_snap + h->batch : nullptr;
    p.applied = h->lg_seen_snap ? h->lg_seen_snap + 2 * h->batch : nullptr;
    p.options = h->cfg.options;
    memcpy(p.Q, h->cfg.Q, sizeof(p.Q));
    memcpy(p.R, h->cfg.R, sizeof(p.R));
    return p;
}

// LARGE-MAP mode, unknown correspondence: the association scratch (allocated on first use) and thresholds of `a`
int large_assoc_scratch(nuslam_ekf * h, nuslam::LargeAssoc & a)
{
    int rc = h->lg_assoc_result.reserve(sizeof(int32_t) * h->batch);
    if (!rc && (h->cfg.options & NUSLAM_OPT_NEAREST_NEIGHBOUR))
        rc = h->lg_nn_slots.reserve(sizeof(nuslam::LargeNNSlot) * h->batch * ((h->cfg.n_landmarks + 127) / 128));
    if (rc) return rc;
    a.result = static_cast<int32_t *>(h->lg_assoc_result.p);
    a.nn = static_cast<nuslam::LargeNNSlot *>(h->lg_nn_slots.p);
    a.amin = h->cfg.assoc_min;
    a.amax = h->cfg.assoc_max;
    CU(cudaMemsetAsync(a.result, 0x7f, sizeof(int32_t) * h->batch, h->stream));   // any value >= every key; finalize resets to INT_MAX
    return NUSLAM_OK;
}

// LARGE-MAP mode: m measurements in delayed passes of at most kLargeMMax; `step_protocol` adds slam.cpp:295-297
// (initializeLandmark for ids above the scan's seen snapshot, seen = max(seen, id)). m_valid (B or null, unknown correspondence
// only): filter b uses only its first m_valid[b] measurements; the passes stay planned from m, so the step needs no host read.
int large_updates(nuslam_ekf * h, const double * z, const int32_t * ids, int m, bool step_protocol, int32_t * ids_out = nullptr,
                  const int32_t * m_valid = nullptr)
{
    nuslam::LargeParams p = make_large_params(h);
    p.m_valid = m_valid;
    nuslam::LargeAssoc assoc;
    if (!ids)
    {
        // unknown correspondence: associateLandmark per measurement against the pass's current covariance
        int rc = h->lg_ids_slot.reserve(sizeof(int32_t) * h->batch * (m > 0 ? m : 1));
        if (!rc) rc = large_assoc_scratch(h, assoc);
        if (rc) return rc;
        assoc.ids_slot = static_cast<int32_t *>(h->lg_ids_slot.p);
        assoc.ids_out = ids_out;
        // slots no kernel writes read 0: those a filter's oracle-order tail never reaches (past its count, or after its process died)
        if (ids_out && m > 0) CU(cudaMemsetAsync(ids_out, 0, sizeof(int32_t) * h->batch * m, h->stream));
    }
    if (step_protocol) CU(cudaMemcpyAsync(h->lg_seen_snap, h->seen, sizeof(int32_t) * h->batch, cudaMemcpyDeviceToDevice, h->stream));
    for (int i0 = 0; i0 < m; i0 += nuslam::kLargeMMax)
    {
        const int cnt = (m - i0 < nuslam::kLargeMMax) ? m - i0 : nuslam::kLargeMMax;
        cudaError_t e = nuslam::launch_large_updates(p, z, ids, m, i0, cnt, step_protocol ? h->lg_seen_snap : nullptr,
                                                     step_protocol ? h->seen : nullptr, h->stream, ids ? nullptr : &assoc);
        if (e != cudaSuccess) return cuda_fail(e, "large-map update pass");
    }
    // x ping-pongs between the state buffer and the scratch: leave the result in the state buffer
    if (p.x != h->x) CU(cudaMemcpyAsync(h->x, p.x, sizeof(double) * (size_t) h->len * h->batch, cudaMemcpyDeviceToDevice, h->stream));
    return NUSLAM_OK;
}

// LARGE-MAP mode, the single associateLandmark call (kOpAssociate): no update is pending, so the candidates read Sigma as it stands
// (pass slot 0) and no oracle-order tail follows; x and Sigma are not written. z: B x 2, id_out: B, both on the device.
int large_associate(nuslam_ekf * h, const double * z, int32_t * id_out)
{
    nuslam::LargeParams p = make_large_params(h);
    p.strict_from = nullptr;
    nuslam::LargeAssoc assoc;
    int rc = h->lg_ids_slot.reserve(sizeof(int32_t) * h->batch);
    if (!rc) rc = large_assoc_scratch(h, assoc);
    if (rc) return rc;
    nuslam::launch_large_associate(p, z, h->seen, static_cast<int32_t *>(h->lg_ids_slot.p), id_out, assoc, h->stream);
    CU(cudaGetLastError());
    return NUSLAM_OK;
}

int finish(nuslam_ekf * h, int mem)
{
    if (mem == NUSLAM_HOST) CU(cudaStreamSynchronize(h->stream));
    return NUSLAM_OK;
}

}   // namespace

extern "C" {

const char * nuslam_last_error(void) { return g_last_error.c_str(); }
int nuslam_version(void) { return NUSLAM_B200_VERSION; }

void nuslam_ekf_default_config(nuslam_ekf_config * cfg, int32_t n_landmarks)
{
    if (!cfg) return;
    memset(cfg, 0, sizeof(*cfg));
    cfg->n_landmarks = n_landmarks;
    cfg->mode = NUSLAM_MODE_STRICT;
    cfg->Q[0] = cfg->Q[4] = cfg->Q[8] = 0.1;   // nuslam/config/slam_params.yaml:3
    cfg->R[0] = cfg->R[3] = 0.001;             // nuslam/config/slam_params.yaml:2
    cfg->assoc_min = 0.01;                     // slam_library.cpp:193
    cfg->assoc_max = 60;                       // slam_library.cpp:194
    cfg->options = 0;                          // the reference's behaviour
    cfg->landmark_prior = nuslam::kLandmarkPrior;   // INT_MAX, slam_library.cpp:30
}

int nuslam_ekf_create(const nuslam_ekf_config * cfg, int64_t batch, int device, void * cuda_stream, nuslam_ekf ** out)
{
    if (!cfg || !out) return fail(NUSLAM_ERR_INVALID, "null config or output pointer");
    if (cfg->n_landmarks < 1 || batch < 1) return fail(NUSLAM_ERR_INVALID, "n_landmarks and batch must be >= 1");
    if (cfg->mode != NUSLAM_MODE_STRICT && cfg->mode != NUSLAM_MODE_FAST && cfg->mode != NUSLAM_MODE_LARGE) return fail(NUSLAM_ERR_INVALID, "unknown mode");
    if (cfg->options & ~(uint32_t) (NUSLAM_OPT_WRAP_INNOVATION | NUSLAM_OPT_JOSEPH | NUSLAM_OPT_PRE_MOTION_JACOBIAN | NUSLAM_OPT_NEAREST_NEIGHBOUR |
                                    NUSLAM_OPT_JOINT_COMPATIBILITY))
        return fail(NUSLAM_ERR_INVALID, "unknown option bit");
    const bool joint = (cfg->options & NUSLAM_OPT_JOINT_COMPATIBILITY) != 0;
    if (joint && (cfg->options & NUSLAM_OPT_NEAREST_NEIGHBOUR))
        return fail(NUSLAM_ERR_INVALID, "NUSLAM_OPT_JOINT_COMPATIBILITY and NUSLAM_OPT_NEAREST_NEIGHBOUR exclude each other");
    if (joint && !(std::isfinite(cfg->assoc_min) && cfg->assoc_min > 0.0))
        return fail(NUSLAM_ERR_INVALID, "NUSLAM_OPT_JOINT_COMPATIBILITY needs a finite assoc_min > 0 (a chi-square gate at 2 dof)");
    if (!(cfg->landmark_prior > 0.0)) return fail(NUSLAM_ERR_INVALID, "landmark_prior must be positive (default config sets INT_MAX)");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceCount (this engine has no CPU path)");
    if (device < 0 || device >= ndev) return fail(NUSLAM_ERR_CUDA, "no such CUDA device (this engine has no CPU path)");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(NUSLAM_ERR_CUDA, "device is not sm_100 or newer; kernels are built for sm_100a only");

    nuslam_ekf * h = new (std::nothrow) nuslam_ekf();
    if (!h) return fail(NUSLAM_ERR_NOMEM, "host allocation failed");
    h->cfg = *cfg;
    h->batch = batch;
    h->len = 3 + 2 * cfg->n_landmarks;
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    h->strict_smem = sizeof(double) * (size_t) (nuslam::strict_smem_doubles(h->len) + (joint ? nuslam::jcbb_smem_doubles(cfg->n_landmarks) : 0));
    h->strict_warps = 4;
    while (h->strict_warps > 1 && h->strict_smem * h->strict_warps > 200 * 1024) h->strict_warps /= 2;
    if (cfg->mode == NUSLAM_MODE_LARGE || h->strict_smem * h->strict_warps > (size_t) prop.sharedMemPerBlockOptin) h->large = true;
    if (joint && h->large)
    {
        delete h;
        return fail(NUSLAM_ERR_UNSUPPORTED, "NUSLAM_OPT_JOINT_COMPATIBILITY runs in the on-chip kernels only (not in large-map mode)");
    }
    // the register kernel covers n_landmarks <= 12; any larger map (that still fits on chip) runs the oracle-order CUDA kernels
    // (same results to the last bit of the reference's arithmetic, lower throughput) -- a FAST request never fails for its size
    if (!h->large && cfg->mode == NUSLAM_MODE_FAST && !nuslam::fast_supported(cfg->n_landmarks)) h->cfg.mode = NUSLAM_MODE_STRICT;
    if (cuda_stream)
    {
        h->stream = static_cast<cudaStream_t>(cuda_stream);
        h->own_stream = false;
    }
    else
    {
        e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess)
        {
            delete h;
            return cuda_fail(e, "cudaStreamCreate");
        }
        h->own_stream = true;
    }
    const size_t l = (size_t) h->len;
    cudaError_t e1 = cudaMalloc(&h->x, sizeof(double) * l * batch);
    cudaError_t e2 = cudaMalloc(&h->sigma, sizeof(double) * l * l * batch);
    cudaError_t e3 = cudaMalloc(&h->seen, sizeof(int32_t) * batch);
    cudaError_t e4 = cudaMalloc(&h->status, sizeof(int32_t) * batch);
    cudaError_t e5 = cudaMalloc(&h->worklist, sizeof(int32_t) * batch);
    cudaError_t e6 = cudaMalloc(&h->wl_count, sizeof(int32_t) * 4);
    if (e5 != cudaSuccess || e6 != cudaSuccess) e1 = cudaErrorMemoryAllocation;
    else cudaMemsetAsync(h->wl_count, 0, sizeof(int32_t) * 4, h->stream);
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess || e4 != cudaSuccess)
    {
        nuslam_ekf_destroy(h);
        return fail(NUSLAM_ERR_NOMEM, "device allocation of the filter state failed");
    }
    h->own_state = true;
    if (h->large)
    {
        cudaError_t l1 = cudaMalloc(&h->lg_x2, sizeof(double) * l * batch);
        cudaError_t l2 = cudaMalloc(&h->lg_U, sizeof(double) * 2 * nuslam::kLargeMMax * l * batch);
        cudaError_t l3 = cudaMalloc(&h->lg_V, sizeof(double) * 2 * nuslam::kLargeMMax * l * batch);
        cudaError_t l4 = cudaMalloc(&h->lg_P, sizeof(double) * 2 * l * batch);
        // [0, B): seen snapshot of the scan, [B, 2B): strict_from of the pass, [2B, 3B): `applied` of the pass (JOSEPH)
        cudaError_t l5 = cudaMalloc(&h->lg_seen_snap, sizeof(int32_t) * 3 * batch);
        if (l1 != cudaSuccess || l2 != cudaSuccess || l3 != cudaSuccess || l4 != cudaSuccess || l5 != cudaSuccess)
        {
            nuslam_ekf_destroy(h);
            return fail(NUSLAM_ERR_NOMEM, "device allocation of the large-map scratch failed");
        }
    }
    cudaMemsetAsync(h->x, 0, sizeof(double) * l * batch, h->stream);
    cudaMemsetAsync(h->sigma, 0, sizeof(double) * l * l * batch, h->stream);
    cudaMemsetAsync(h->seen, 0, sizeof(int32_t) * batch, h->stream);
    cudaMemsetAsync(h->status, 0, sizeof(int32_t) * batch, h->stream);
    if (joint)
    {
        double T[nuslam::kJcbbMMax + 1];
        joint_thresholds(cfg->assoc_min, T);
        int rc = h->joint_t.reserve(sizeof(T));
        if (!rc && cudaMemcpy(h->joint_t.p, T, sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess) rc = fail(NUSLAM_ERR_CUDA, "copy of the joint thresholds");
        if (rc)
        {
            nuslam_ekf_destroy(h);
            return rc;
        }
    }
    *out = h;
    return NUSLAM_OK;
}

int nuslam_ekf_destroy(nuslam_ekf * h)
{
    if (!h) return NUSLAM_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->own_state)
    {
        if (h->x) cudaFree(h->x);
        if (h->sigma) cudaFree(h->sigma);
        if (h->seen) cudaFree(h->seen);
        if (h->status) cudaFree(h->status);
    }
    for (auto & sl : h->slots)
    {
        sl.tw.release();
        sl.z.release();
        sl.ids.release();
        sl.xsnap.release();
        if (sl.h2d_done) cudaEventDestroy(sl.h2d_done);
        if (sl.kernel_done) cudaEventDestroy(sl.kernel_done);
        if (sl.d2h_done) cudaEventDestroy(sl.d2h_done);
    }
    if (h->s_in) cudaStreamDestroy(h->s_in);
    if (h->s_out) cudaStreamDestroy(h->s_out);
    if (h->lg_x2) cudaFree(h->lg_x2);
    if (h->lg_U) cudaFree(h->lg_U);
    if (h->lg_V) cudaFree(h->lg_V);
    if (h->lg_P) cudaFree(h->lg_P);
    if (h->lg_seen_snap) cudaFree(h->lg_seen_snap);
    h->lg_ids_slot.release();
    h->lg_assoc_result.release();
    h->lg_nn_slots.release();
    h->joint_t.release();
    if (h->worklist) cudaFree(h->worklist);
    if (h->wl_count) cudaFree(h->wl_count);
    h->s_tw.release();
    h->s_z.release();
    h->s_ids.release();
    h->s_ids_out.release();
    h->s_misc.release();
    for (DevBuf * b : {&h->f_ranges, &h->f_ncl, &h->f_nci, &h->f_circ, &h->f_z, &h->f_mv}) b->release();
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return NUSLAM_OK;
}

int nuslam_ekf_bind_state(nuslam_ekf * h, double * x_dev, double * sigma_dev, int32_t * seen_dev, int32_t * status_dev)
{
    if (!h || !x_dev || !sigma_dev || !seen_dev || !status_dev) return fail(NUSLAM_ERR_INVALID, "null pointer");
    if (select_device(h)) return NUSLAM_ERR_CUDA;
    CU(cudaStreamSynchronize(h->stream));
    if (h->own_state)
    {
        cudaFree(h->x);
        cudaFree(h->sigma);
        cudaFree(h->seen);
        cudaFree(h->status);
    }
    h->own_state = false;
    h->x = x_dev;
    h->sigma = sigma_dev;
    h->seen = seen_dev;
    h->status = status_dev;
    return NUSLAM_OK;
}

int nuslam_ekf_device_pointers(nuslam_ekf * h, double ** x_dev, double ** sigma_dev, int32_t ** seen_dev, int32_t ** status_dev)
{
    if (!h) return fail(NUSLAM_ERR_INVALID, "null handle");
    if (x_dev) *x_dev = h->x;
    if (sigma_dev) *sigma_dev = h->sigma;
    if (seen_dev) *seen_dev = h->seen;
    if (status_dev) *status_dev = h->status;
    return NUSLAM_OK;
}

int nuslam_ekf_init(nuslam_ekf * h, const double * robot_state, const double * map_state, int mem)
{
    if (!h || !robot_state) return fail(NUSLAM_ERR_INVALID, "null handle or robot_state");
    if (select_device(h)) return NUSLAM_ERR_CUDA;
    const int n = h->cfg.n_landmarks;
    const double * d_robot = nullptr;
    const double * d_map = nullptr;
    int rc = stage_in(h, h->s_tw, robot_state, (size_t) h->batch * 3, mem, &d_robot);
    if (rc) return rc;
    rc = stage_in(h, h->s_z, map_state, (size_t) h->batch * 2 * n, mem, &d_map);
    if (rc) return rc;
    const int64_t total = h->batch * (int64_t) h->len * h->len;
    const int threads = 256;
    const int64_t blocks = (total + threads - 1) / threads;
    nuslam::k_ekf_init<<<(unsigned) blocks, threads, 0, h->stream>>>(h->batch, h->len, d_robot, d_map, h->x, h->sigma, h->seen, h->status, h->cfg.landmark_prior);
    CU(cudaGetLastError());
    return finish(h, mem);
}

int nuslam_ekf_set_state(nuslam_ekf * h, const double * x, const double * sigma, const int32_t * seen, const int32_t * status, int mem)
{
    if (!h) return fail(NUSLAM_ERR_INVALID, "null handle");
    if (select_device(h)) return NUSLAM_ERR_CUDA;
    const cudaMemcpyKind kind = (mem == NUSLAM_HOST) ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    const size_t l = (size_t) h->len;
    if (x) CU(cudaMemcpyAsync(h->x, x, sizeof(double) * l * h->batch, kind, h->stream));
    if (sigma) CU(cudaMemcpyAsync(h->sigma, sigma, sizeof(double) * l * l * h->batch, kind, h->stream));
    if (seen) CU(cudaMemcpyAsync(h->seen, seen, sizeof(int32_t) * h->batch, kind, h->stream));
    if (status) CU(cudaMemcpyAsync(h->status, status, sizeof(int32_t) * h->batch, kind, h->stream));
    return finish(h, mem);
}

int nuslam_ekf_get_state(nuslam_ekf * h, double * x, double * sigma, int32_t * seen, int32_t * status, int mem)
{
    if (!h) return fail(NUSLAM_ERR_INVALID, "null handle");
    if (select_device(h)) return NUSLAM_ERR_CUDA;
    const cudaMemcpyKind kind = (mem == NUSLAM_HOST) ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    const size_t l = (size_t) h->len;
    if (x) CU(cudaMemcpyAsync(x, h->x, sizeof(double) * l * h->batch, kind, h->stream));
    if (sigma) CU(cudaMemcpyAsync(sigma, h->sigma, sizeof(double) * l * l * h->batch, kind, h->stream));
    if (seen) CU(cudaMemcpyAsync(seen, h->seen, sizeof(int32_t) * h->batch, kind, h->stream));
    if (status) CU(cudaMemcpyAsync(status, h->status, sizeof(int32_t) * h->batch, kind, h->stream));
    return finish(h, mem);
}

int nuslam_ekf_predict(nuslam_ekf * h, const double * twists, int mem)
{
    if (!h || !twists) return fail(NUSLAM_ERR_INVALID, "null handle or twists");
    if (select_device(h)) return NUSLAM_ERR_CUDA;
    nuslam::EkfParams p = make_params(h);
    int rc = stage_in(h, h->s_tw, twists, (size_t) h->batch * 3, mem, &p.twists);
    if (rc) return rc;
    if (h->large)
    {
        cudaError_t e = nuslam::launch_large_predict(make_large_params(h), p.twists, h->stream);
        if (e != cudaSuccess) return cuda_fail(e, "large-map predict");
        return finish(h, mem);
    }
    rc = launch_strict<nuslam::kOpPredict>(h, p);   // predict is O(len) in either mode: the strict order costs nothing extra
    if (rc) return rc;
    return finish(h, mem);
}

int nuslam_ekf_associate(nuslam_ekf * h, const double * z, int32_t * id_out, int mem)
{
    if (!h || !z || !id_out) return fail(NUSLAM_ERR_INVALID, "null argument");
    if (select_device(h)) return NUSLAM_ERR_CUDA;
    nuslam::EkfParams p = make_params(h);
    p.m = 1;
    int rc = stage_in(h, h->s_z, z, (size_t) h->batch * 2, mem, &p.z);
    if (rc) return rc;
    if (mem == NUSLAM_HOST)
    {
        rc = h->s_ids_out.reserve(sizeof(int32_t) * h->batch);
        if (rc) return rc;
        p.ids_out = static_cast<int32_t *>(h->s_ids_out.p);
    }
    else
        p.ids_out = id_out;
    // one measurement: joint compatibility is nearest neighbour (T[1] = assoc_min, the same distances)
    if (p.options & NUSLAM_OPT_JOINT_COMPATIBILITY) p.options = (p.options & ~(unsigned) NUSLAM_OPT_JOINT_COMPATIBILITY) | NUSLAM_OPT_NEAREST_NEIGHBOUR;
    rc = h->large ? large_associate(h, p.z, p.ids_out) : launch_strict<nuslam::kOpAssociate>(h, p);
    if (rc) return rc;
    if (mem == NUSLAM_HOST) CU(cudaMemcpyAsync(id_out, p.ids_out, sizeof(int32_t) * h->batch, cudaMemcpyDeviceToHost, h->stream));
    return finish(h, mem);
}

int nuslam_ekf_initialize_landmark(nuslam_ekf * h, const double * z, const int32_t * id, int mem)
{
    if (!h || !z || !id) return fail(NUSLAM_ERR_INVALID, "null argument");
    if (select_device(h)) return NUSLAM_ERR_CUDA;
    nuslam::EkfParams p = make_params(h);
    p.m = 1;
    int rc = stage_in(h, h->s_z, z, (size_t) h->batch * 2, mem, &p.z);
    if (rc) return rc;
    rc = stage_in(h, h->s_ids, id, (size_t) h->batch, mem, &p.ids);
    if (rc) return rc;
    if (h->large)
    {
        nuslam::k_large_init_landmark<<<(unsigned) ((h->batch + 63) / 64), 64, 0, h->stream>>>(make_large_params(h), p.z, p.ids, 1, 0, nullptr, nullptr);
        CU(cudaGetLastError());
        return finish(h, mem);
    }
    rc = launch_strict<nuslam::kOpInit>(h, p);
    if (rc) return rc;
    return finish(h, mem);
}

int nuslam_ekf_update(nuslam_ekf * h, const double * z, const int32_t * id, int mem)
{
    if (!h || !z || !id) return fail(NUSLAM_ERR_INVALID, "null argument");
    if (select_device(h)) return NUSLAM_ERR_CUDA;
    nuslam::EkfParams p = make_params(h);
    p.m = 1;
    int rc = stage_in(h, h->s_z, z, (size_t) h->batch * 2, mem, &p.z);
    if (rc) return rc;
    rc = stage_in(h, h->s_ids, id, (size_t) h->batch, mem, &p.ids);
    if (rc) return rc;
    if (h->large)
    {
        rc = large_updates(h, p.z, p.ids, 1, /*step_protocol=*/false);
        if (rc) return rc;
        return finish(h, mem);
    }
    if (h->cfg.mode == NUSLAM_MODE_FAST && h->cfg.options == 0)
    {
        p.twists = nullptr;   // update only
        rc = launch_fast_then_strict<nuslam::kOpUpdate>(h, p, /*do_predict=*/false);
        if (rc) return rc;
    }
    else
    {
        rc = launch_strict<nuslam::kOpUpdate>(h, p);
        if (rc) return rc;
    }
    return finish(h, mem);
}

int nuslam_ekf_measurement_model(nuslam_ekf * h, const int32_t * j, double * zhat, double * H, int mem)
{
    if (!h || !j) return fail(NUSLAM_ERR_INVALID, "null argument");
    if (select_device(h)) return NUSLAM_ERR_CUDA;
    const int32_t * d_j = nullptr;
    int rc = stage_in(h, h->s_ids, j, (size_t) h->batch, mem, &d_j);
    if (rc) return rc;
    double * d_zhat = zhat;
    double * d_H = H;
    const size_t hz = (size_t) h->batch * 2, hh = (size_t) h->batch * 2 * h->len;
    if (mem == NUSLAM_HOST)
    {
        rc = h->s_misc.reserve(sizeof(double) * (hz + hh));
        if (rc) return rc;
        d_zhat = zhat ? static_cast<double *>(h->s_misc.p) : nullptr;
        d_H = H ? static_cast<double *>(h->s_misc.p) + hz : nullptr;
    }
    const int threads = 128;
    const int64_t blocks = (h->batch + threads - 1) / threads;
    nuslam::k_measurement_model<<<(unsigned) blocks, threads, 0, h->stream>>>(h->batch, h->len, h->cfg.n_landmarks, h->x, d_j, d_zhat, d_H);
    CU(cudaGetLastError());
    if (mem == NUSLAM_HOST)
    {
        if (zhat) CU(cudaMemcpyAsync(zhat, d_zhat, sizeof(double) * hz, cudaMemcpyDeviceToHost, h->stream));
        if (H) CU(cudaMemcpyAsync(H, d_H, sizeof(double) * hh, cudaMemcpyDeviceToHost, h->stream));
    }
    return finish(h, mem);
}

namespace
{

// one iteration of slam.cpp:262-319 for every filter; all pointers in `p` are device pointers
int step_device(nuslam_ekf * h, const nuslam::EkfParams & p)
{
    const int m = p.m;
    if (h->large)
    {
        cudaError_t e = nuslam::launch_large_predict(make_large_params(h), p.twists, h->stream);
        if (e != cudaSuccess) return cuda_fail(e, "large-map predict");
        if (m > 0)
        {
            int rc = large_updates(h, p.z, p.ids, m, /*step_protocol=*/true, p.ids_out, p.m_valid);
            if (rc) return rc;
        }
        if (p.ids && p.ids_out && m > 0) CU(cudaMemcpyAsync(p.ids_out, p.ids, sizeof(int32_t) * h->batch * m, cudaMemcpyDeviceToDevice, h->stream));
        return NUSLAM_OK;
    }
    if ((h->cfg.options & NUSLAM_OPT_JOINT_COMPATIBILITY) && !p.ids) return launch_strict<nuslam::kOpStepJoint>(h, p);
    if (h->cfg.mode == NUSLAM_MODE_FAST && h->cfg.options == 0 && m <= nuslam::kFastMMax)
        // known correspondence, or on-device association (ids == NULL): the register kernel, then the strict kernel over the
        // filters it handed over (first touches, new landmarks)
        return launch_fast_then_strict<nuslam::kOpStep>(h, p, /*do_predict=*/true);
    // STRICT mode (and steps with more than kFastMMax measurements): the oracle-order kernel, association included
    return launch_strict<nuslam::kOpStep>(h, p);
}

}   // namespace

int nuslam_ekf_step(nuslam_ekf * h, const double * twists, const double * z, const int32_t * ids, int32_t m, int32_t * ids_out, int mem)
{
    if (!h || !twists) return fail(NUSLAM_ERR_INVALID, "null handle or twists");
    if (m < 0 || (m > 0 && !z)) return fail(NUSLAM_ERR_INVALID, "m < 0 or null z");
    if (joint_m_check(h, ids == nullptr, m)) return NUSLAM_ERR_UNSUPPORTED;
    if (select_device(h)) return NUSLAM_ERR_CUDA;
    nuslam::EkfParams p = make_params(h);
    p.m = m;
    int rc = stage_in(h, h->s_tw, twists, (size_t) h->batch * 3, mem, &p.twists);
    if (rc) return rc;
    rc = stage_in(h, h->s_z, z, (size_t) h->batch * m * 2, mem, &p.z);
    if (rc) return rc;
    rc = stage_in(h, h->s_ids, ids, (size_t) h->batch * m, mem, &p.ids);
    if (rc) return rc;
    p.ids_out = ids_out;
    if (ids_out && mem == NUSLAM_HOST)
    {
        rc = h->s_ids_out.reserve(sizeof(int32_t) * h->batch * (m > 0 ? m : 1));
        if (rc) return rc;
        p.ids_out = static_cast<int32_t *>(h->s_ids_out.p);
    }
    rc = step_device(h, p);
    if (rc) return rc;
    if (ids_out && mem == NUSLAM_HOST && m > 0)
        CU(cudaMemcpyAsync(ids_out, p.ids_out, sizeof(int32_t) * h->batch * m, cudaMemcpyDeviceToHost, h->stream));
    return finish(h, mem);
}

int nuslam_ekf_scan_step(nuslam_ekf * h, const double * twists, const float * ranges, double min_range, double max_range, int32_t m,
                         int32_t * n_markers_out, double * z_out, int32_t * ids_out, int mem)
{
    if (!h || !twists || !ranges) return fail(NUSLAM_ERR_INVALID, "null handle, twists or ranges");
    if (m < 1) return fail(NUSLAM_ERR_INVALID, "m < 1");
    if (joint_m_check(h, true, m)) return NUSLAM_ERR_UNSUPPORTED;
    if (select_device(h)) return NUSLAM_ERR_CUDA;
    const size_t B = (size_t) h->batch;
    nuslam::EkfParams p = make_params(h);
    p.m = m;
    int rc = stage_in(h, h->s_tw, twists, B * 3, mem, &p.twists);
    if (rc) return rc;
    const float * d_ranges = nullptr;
    rc = stage_in(h, h->f_ranges, ranges, B * NUSLAM_SCAN_BEAMS, mem, &d_ranges);
    if (!rc) rc = h->f_ncl.reserve(sizeof(int32_t) * B);
    if (!rc) rc = h->f_nci.reserve(sizeof(int32_t) * B);
    if (!rc) rc = h->f_circ.reserve(sizeof(double) * 4 * B * m);
    if (!rc) rc = h->f_z.reserve(sizeof(double) * 2 * B * m);
    if (!rc) rc = h->f_mv.reserve(sizeof(int32_t) * B);
    if (!rc && ids_out && mem == NUSLAM_HOST) rc = h->s_ids_out.reserve(sizeof(int32_t) * B * m);
    if (rc) return rc;
    int32_t * d_nci = static_cast<int32_t *>(h->f_nci.p);
    double * d_circ = static_cast<double *>(h->f_circ.p);
    double * d_z = static_cast<double *>(h->f_z.p);
    int32_t * d_mv = static_cast<int32_t *>(h->f_mv.p);
    // Landmarks::main_loop, landmarks.cpp:84-109: the first m markers of every scan, in detection order
    cudaError_t e = (nuslam::scan_fit_mode() == nuslam::kFitMoment ? nuslam::launch_scan_moment : nuslam::launch_scan_detect)(
        d_ranges, (int64_t) B, min_range, max_range, nullptr, static_cast<int32_t *>(h->f_ncl.p), d_nci, d_circ, m, NUSLAM_SCAN_UB, h->device,
        h->sm_count, h->stream);
    if (e != cudaSuccess) return cuda_fail(e, "scan_detect");
    // slam.cpp:282-286: markers -> (range, bearing)
    const int64_t total = (int64_t) B * m;
    nuslam::k_markers_to_measurements<<<(unsigned) ((total + 255) / 256), 256, 0, h->stream>>>(d_circ, d_nci, h->batch, m, m, d_z, d_mv);
    CU(cudaGetLastError());
    // slam.cpp:262-319 with unknown data association
    p.z = d_z;
    p.ids = nullptr;
    p.m_valid = d_mv;
    p.ids_out = (ids_out && mem == NUSLAM_HOST) ? static_cast<int32_t *>(h->s_ids_out.p) : ids_out;
    rc = step_device(h, p);
    if (rc) return rc;
    const cudaMemcpyKind kind = (mem == NUSLAM_HOST) ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    if (n_markers_out) CU(cudaMemcpyAsync(n_markers_out, d_nci, sizeof(int32_t) * B, kind, h->stream));
    if (z_out) CU(cudaMemcpyAsync(z_out, d_z, sizeof(double) * 2 * B * m, kind, h->stream));
    if (ids_out && mem == NUSLAM_HOST) CU(cudaMemcpyAsync(ids_out, p.ids_out, sizeof(int32_t) * B * m, cudaMemcpyDeviceToHost, h->stream));
    return finish(h, mem);
}

namespace
{
// one pipelined host-buffer step. Inputs either as three host arrays (twists, z, ids_host) or as ONE packed host buffer
// [twists | z | ids] copied by a single cudaMemcpyAsync; ids may also come from the handle's device cache (ids_dev).
int step_async_impl(nuslam_ekf * h, const double * twists, const double * z, const int32_t * ids_host, const int32_t * ids_dev, const void * packed,
                    bool packed_has_ids, int32_t m, double * x_out)
{
    if (joint_m_check(h, !ids_host && !ids_dev && !packed_has_ids, m)) return NUSLAM_ERR_UNSUPPORTED;
    if (select_device(h)) return NUSLAM_ERR_CUDA;
    if (!h->s_in)
    {
        CU(cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking));
        for (auto & sl : h->slots)
        {
            CU(cudaEventCreateWithFlags(&sl.h2d_done, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&sl.kernel_done, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&sl.d2h_done, cudaEventDisableTiming));
        }
    }
    auto & sl = h->slots[h->async_count % 3];
    // the slot's previous step must have left: its kernel has consumed the staged inputs and its snapshot has reached the host
    if (sl.busy) CU(cudaEventSynchronize(sl.d2h_done));
    const size_t B = (size_t) h->batch, l = (size_t) h->len;
    const size_t b_tw = sizeof(double) * 3 * B, b_z = sizeof(double) * 2 * B * (size_t) m, b_ids = sizeof(int32_t) * B * (size_t) m;
    const double * d_tw = nullptr;
    const double * d_z = nullptr;
    const int32_t * d_ids = ids_dev;
    int rc = sl.xsnap.reserve(sizeof(double) * l * B);
    if (rc) return rc;
    // stage 1 (copy-in stream): host -> device
    if (packed)
    {
        // [twists B x 3 f64][z B x m x 2 f64][ids B x m i32]: one copy (every section starts 8-byte aligned)
        const size_t total = b_tw + b_z + (packed_has_ids ? b_ids : 0);
        rc = sl.tw.reserve(total);
        if (rc) return rc;
        CU(cudaMemcpyAsync(sl.tw.p, packed, total, cudaMemcpyHostToDevice, h->s_in));
        d_tw = static_cast<const double *>(sl.tw.p);
        d_z = reinterpret_cast<const double *>(static_cast<const char *>(sl.tw.p) + b_tw);
        if (packed_has_ids) d_ids = reinterpret_cast<const int32_t *>(static_cast<const char *>(sl.tw.p) + b_tw + b_z);
    }
    else
    {
        rc = sl.tw.reserve(b_tw);
        if (!rc) rc = sl.z.reserve(b_z > 0 ? b_z : 8);
        if (!rc && ids_host) rc = sl.ids.reserve(b_ids > 0 ? b_ids : 8);
        if (rc) return rc;
        CU(cudaMemcpyAsync(sl.tw.p, twists, b_tw, cudaMemcpyHostToDevice, h->s_in));
        if (m > 0)
        {
            CU(cudaMemcpyAsync(sl.z.p, z, b_z, cudaMemcpyHostToDevice, h->s_in));
            if (ids_host) CU(cudaMemcpyAsync(sl.ids.p, ids_host, b_ids, cudaMemcpyHostToDevice, h->s_in));
        }
        d_tw = static_cast<const double *>(sl.tw.p);
        d_z = static_cast<const double *>(sl.z.p);
        if (ids_host) d_ids = static_cast<const int32_t *>(sl.ids.p);
    }
    CU(cudaEventRecord(sl.h2d_done, h->s_in));
    // stage 2 (compute stream): the step on device buffers, then a snapshot of x so that the next step may start at once
    CU(cudaStreamWaitEvent(h->stream, sl.h2d_done, 0));
    // the step kernels write the snapshot themselves (216 B per filter next to the state store) where they can; the large-map
    // kernels do not: a device-to-device copy stands in
    const bool in_kernel_snapshot = !h->large;
    h->x_snap_next = in_kernel_snapshot ? static_cast<double *>(sl.xsnap.p) : nullptr;
    rc = h->async_dry ? NUSLAM_OK : nuslam_ekf_step(h, d_tw, d_z, d_ids, m, nullptr, NUSLAM_DEVICE);
    h->x_snap_next = nullptr;
    if (rc) return rc;
    if (!in_kernel_snapshot && !h->async_dry) CU(cudaMemcpyAsync(sl.xsnap.p, h->x, sizeof(double) * l * B, cudaMemcpyDeviceToDevice, h->stream));
    CU(cudaEventRecord(sl.kernel_done, h->stream));
    // stage 3 (copy-out stream): device -> host
    CU(cudaStreamWaitEvent(h->s_out, sl.kernel_done, 0));
    CU(cudaMemcpyAsync(x_out, sl.xsnap.p, sizeof(double) * l * B, cudaMemcpyDeviceToHost, h->s_out));
    CU(cudaEventRecord(sl.d2h_done, h->s_out));
    sl.busy = true;
    h->async_count++;
    return NUSLAM_OK;
}
}   // namespace

int nuslam_ekf_step_async(nuslam_ekf * h, const double * twists, const double * z, const int32_t * ids, int32_t m, double * x_out)
{
    if (!h || !twists || !x_out) return fail(NUSLAM_ERR_INVALID, "null argument");
    if (m < 0 || (m > 0 && !z)) return fail(NUSLAM_ERR_INVALID, "m < 0 or null z");
    return step_async_impl(h, twists, z, ids, nullptr, nullptr, false, m, x_out);
}

int nuslam_ekf_set_ids(nuslam_ekf * h, const int32_t * ids, int32_t m, int mem)
{
    if (!h || !ids || m < 1) return fail(NUSLAM_ERR_INVALID, "null argument or m < 1");
    if (select_device(h)) return NUSLAM_ERR_CUDA;
    const size_t bytes = sizeof(int32_t) * (size_t) h->batch * (size_t) m;
    int rc = h->ids_cache.reserve(bytes);
    if (rc) return rc;
    CU(cudaMemcpyAsync(h->ids_cache.p, ids, bytes, mem == NUSLAM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->stream));
    if (mem == NUSLAM_HOST) CU(cudaStreamSynchronize(h->stream));   // the caller's buffer is free on return
    h->ids_cache_m = m;
    return NUSLAM_OK;
}

int nuslam_ekf_step_async_packed(nuslam_ekf * h, const void * packed, int32_t m, int ids_mode, double * x_out)
{
    if (!h || !packed || !x_out) return fail(NUSLAM_ERR_INVALID, "null argument");
    if (m < 0) return fail(NUSLAM_ERR_INVALID, "m < 0");
    const int32_t * cached = nullptr;
    if (ids_mode == NUSLAM_IDS_CACHED)
    {
        if (h->ids_cache_m != m || !h->ids_cache.p) return fail(NUSLAM_ERR_INVALID, "NUSLAM_IDS_CACHED: call nuslam_ekf_set_ids with the same m first");
        cached = static_cast<const int32_t *>(h->ids_cache.p);
    }
    else if (ids_mode != NUSLAM_IDS_PACKED && ids_mode != NUSLAM_IDS_NONE)
        return fail(NUSLAM_ERR_INVALID, "ids_mode is NUSLAM_IDS_NONE, NUSLAM_IDS_PACKED or NUSLAM_IDS_CACHED");
    return step_async_impl(h, nullptr, nullptr, nullptr, cached, packed, ids_mode == NUSLAM_IDS_PACKED, m, x_out);
}

int nuslam_ekf_async_dry_run(nuslam_ekf * h, int on)
{
    if (!h) return fail(NUSLAM_ERR_INVALID, "null handle");
    h->async_dry = on != 0;
    return NUSLAM_OK;
}

int nuslam_ekf_wait_async(nuslam_ekf * h)
{
    if (!h) return fail(NUSLAM_ERR_INVALID, "null handle");
    if (select_device(h)) return NUSLAM_ERR_CUDA;
    for (auto & sl : h->slots)
        if (sl.busy)
        {
            CU(cudaEventSynchronize(sl.d2h_done));
            sl.busy = false;
        }
    return NUSLAM_OK;
}

// kernel-experiment builds only (-DNUSLAM_TIMING): per-phase clock64 sums of block 0 / warp 0 of the FAST kernel
int nuslam_debug_fast_timing(long long * out16, int reset) { return nuslam::fast_timing_read(out16, reset); }

int nuslam_ekf_error_stats(nuslam_ekf * h, const double * truth_pose, const double * truth_map, const int32_t * ids_got, const int32_t * ids_want,
                           int32_t m, double * stats_out)
{
    if (!h || !stats_out) return fail(NUSLAM_ERR_INVALID, "null handle or output");
    if ((ids_got == nullptr) != (ids_want == nullptr) || m < 0) return fail(NUSLAM_ERR_INVALID, "ids_got and ids_want go together");
    if (select_device(h)) return NUSLAM_ERR_CUDA;
    CU(cudaMemsetAsync(stats_out, 0, sizeof(double) * nuslam::kStatsCount, h->stream));
    const int64_t blocks = (h->batch + 255) / 256;
    nuslam::k_error_stats<<<(unsigned) blocks, 256, 0, h->stream>>>(h->x, h->sigma, h->seen, h->status, h->batch, h->len, h->cfg.n_landmarks, truth_pose,
                                                                 truth_map, ids_got, ids_want, m, stats_out);
    CU(cudaGetLastError());
    return NUSLAM_OK;
}

int nuslam_ekf_get_stream(nuslam_ekf * h, void ** cuda_stream_out)
{
    if (!h || !cuda_stream_out) return fail(NUSLAM_ERR_INVALID, "null handle or output");
    *cuda_stream_out = static_cast<void *>(h->stream);
    return NUSLAM_OK;
}

int nuslam_ekf_synchronize(nuslam_ekf * h)
{
    if (!h) return fail(NUSLAM_ERR_INVALID, "null handle");
    if (select_device(h)) return NUSLAM_ERR_CUDA;
    CU(cudaStreamSynchronize(h->stream));
    if (nuslam::tail_launch_active() && h->wl_count)
    {
        // a device-side launch of the list kernel that failed (strict_tail) left its error code here
        int32_t dev_err = 0;
        CU(cudaMemcpy(&dev_err, h->wl_count + 3, sizeof(dev_err), cudaMemcpyDeviceToHost));
        if (dev_err)
        {
            cudaMemset(h->wl_count + 3, 0, sizeof(int32_t));
            return cuda_fail((cudaError_t) dev_err, "device-side launch of the strict list kernel");
        }
    }
    return NUSLAM_OK;
}

int nuslam_tail_launch(void) { return nuslam::tail_launch_active() ? 1 : 0; }

namespace
{
int elementwise_io(const double * in, double * out, int64_t count, int in_width, int out_width, int mem, int device, void * cuda_stream, int which)
{
    if (!in || !out || count < 0) return fail(NUSLAM_ERR_INVALID, "null argument");
    if (count == 0) return NUSLAM_OK;
    CU(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    const double * d_in = in;
    double * d_out = out;
    double * tmp = nullptr;
    if (mem == NUSLAM_HOST)
    {
        CU(cudaMalloc(&tmp, sizeof(double) * count * (in_width + out_width)));
        CU(cudaMemcpyAsync(tmp, in, sizeof(double) * count * in_width, cudaMemcpyHostToDevice, st));
        d_in = tmp;
        d_out = tmp + count * in_width;
    }
    const int threads = 256;
    const int64_t blocks = (count + threads - 1) / threads;
    if (which == 0) nuslam::k_cartesian2polar<<<(unsigned) blocks, threads, 0, st>>>(d_in, d_out, count);
    else if (which == 1) nuslam::k_normalize_angle<<<(unsigned) blocks, threads, 0, st>>>(d_in, d_out, count);
    else nuslam::k_integrate_twist<<<(unsigned) blocks, threads, 0, st>>>(d_in, d_out, count);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && mem == NUSLAM_HOST)
    {
        e = cudaMemcpyAsync(out, d_out, sizeof(double) * count * out_width, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    if (tmp) cudaFree(tmp);
    if (e != cudaSuccess) return cuda_fail(e, "elementwise kernel");
    return NUSLAM_OK;
}
}   // namespace

int nuslam_cartesian2polar(const double * xy, double * rb, int64_t count, int mem, int device, void * cuda_stream)
{
    return elementwise_io(xy, rb, count, 2, 2, mem, device, cuda_stream, 0);
}

int nuslam_normalize_angle(const double * rad_in, double * rad_out, int64_t count, int mem, int device, void * cuda_stream)
{
    return elementwise_io(rad_in, rad_out, count, 1, 1, mem, device, cuda_stream, 1);
}

int nuslam_integrate_twist(const double * twists, double * transforms_out, int64_t count, int mem, int device, void * cuda_stream)
{
    return elementwise_io(twists, transforms_out, count, 3, 4, mem, device, cuda_stream, 2);
}

int nuslam_diffdrive_step(double * state7, const double * thL_new, const double * thR_new, double * twists_out, int64_t count, int mem,
                          int device, void * cuda_stream)
{
    if (!state7 || !thL_new || !thR_new || !twists_out || count < 0) return fail(NUSLAM_ERR_INVALID, "null argument");
    if (count == 0) return NUSLAM_OK;
    CU(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    double * d_state = state7;
    const double * d_l = thL_new;
    const double * d_r = thR_new;
    double * d_tw = twists_out;
    double * tmp = nullptr;
    if (mem == NUSLAM_HOST)
    {
        CU(cudaMalloc(&tmp, sizeof(double) * count * 12));
        CU(cudaMemcpyAsync(tmp, state7, sizeof(double) * count * 7, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(tmp + 7 * count, thL_new, sizeof(double) * count, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(tmp + 8 * count, thR_new, sizeof(double) * count, cudaMemcpyHostToDevice, st));
        d_state = tmp;
        d_l = tmp + 7 * count;
        d_r = tmp + 8 * count;
        d_tw = tmp + 9 * count;
    }
    const int threads = 128;
    nuslam::k_diffdrive_step<<<(unsigned) ((count + threads - 1) / threads), threads, 0, st>>>(d_state, d_l, d_r, d_tw, count);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && mem == NUSLAM_HOST)
    {
        e = cudaMemcpyAsync(state7, d_state, sizeof(double) * count * 7, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(twists_out, d_tw, sizeof(double) * count * 3, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    if (tmp) cudaFree(tmp);
    if (e != cudaSuccess) return cuda_fail(e, "diffdrive_step");
    return NUSLAM_OK;
}

int nuslam_ekf_map_to_odom(nuslam_ekf * h, const double * odom_state7, double * out, int mem)
{
    if (!h || !odom_state7 || !out) return fail(NUSLAM_ERR_INVALID, "null argument");
    if (select_device(h)) return NUSLAM_ERR_CUDA;
    const size_t B = (size_t) h->batch;
    const double * d_odom = nullptr;
    int rc = stage_in(h, h->s_misc, odom_state7, B * 7, mem, &d_odom);
    if (rc) return rc;
    double * d_out = out;
    if (mem == NUSLAM_HOST)
    {
        rc = h->s_z.reserve(sizeof(double) * 3 * B);
        if (rc) return rc;
        d_out = static_cast<double *>(h->s_z.p);
    }
    nuslam::k_map_to_odom<<<(unsigned) ((B + 127) / 128), 128, 0, h->stream>>>(d_odom, h->x, h->len, d_out, h->batch);
    CU(cudaGetLastError());
    if (mem == NUSLAM_HOST) CU(cudaMemcpyAsync(out, d_out, sizeof(double) * 3 * B, cudaMemcpyDeviceToHost, h->stream));
    return finish(h, mem);
}

int nuslam_world_step(double * world, const double * cmd, const double * noise, double dt, const double * tubes, int32_t n_tubes,
                      double tube_rad, double robot_rad, double max_range, float * ranges_out, double * joints_out, int64_t count, int mem,
                      int device, void * cuda_stream)
{
    if (!world || !cmd || !ranges_out || count < 0 || n_tubes < 0 || (n_tubes > 0 && !tubes)) return fail(NUSLAM_ERR_INVALID, "null argument");
    if (n_tubes > nuslam::kWorldMaxTubes) return fail(NUSLAM_ERR_UNSUPPORTED, "at most 64 tubes");
    if (count == 0) return NUSLAM_OK;
    CU(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    nuslam::WorldParams p;
    memset(&p, 0, sizeof(p));
    p.count = count;
    p.n_tubes = n_tubes;
    p.dt = dt;
    p.tube_rad = tube_rad;
    p.robot_rad = robot_rad;
    p.max_range = max_range;
    p.world = world;
    p.cmd = cmd;
    p.noise = noise;
    p.tubes = tubes;
    p.ranges = ranges_out;
    p.joints = joints_out;
    char * tmp = nullptr;
    const size_t b_w = sizeof(double) * 9 * count, b_c = sizeof(double) * 3 * count, b_n = sizeof(double) * 4 * count;
    const size_t b_t = sizeof(double) * 2 * (n_tubes > 0 ? n_tubes : 1), b_r = sizeof(float) * 360 * count, b_j = sizeof(double) * 2 * count;
    if (mem == NUSLAM_HOST)
    {
        auto al = [](size_t v) { return (v + 255) & ~(size_t) 255; };
        CU(cudaMalloc(&tmp, al(b_w) + al(b_c) + al(b_n) + al(b_t) + al(b_r) + al(b_j)));
        char * q = tmp;
        p.world = reinterpret_cast<double *>(q);
        q += al(b_w);
        double * d_cmd = reinterpret_cast<double *>(q);
        q += al(b_c);
        double * d_noise = reinterpret_cast<double *>(q);
        q += al(b_n);
        double * d_tubes = reinterpret_cast<double *>(q);
        q += al(b_t);
        p.ranges = reinterpret_cast<float *>(q);
        q += al(b_r);
        p.joints = reinterpret_cast<double *>(q);
        CU(cudaMemcpyAsync(p.world, world, b_w, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(d_cmd, cmd, b_c, cudaMemcpyHostToDevice, st));
        if (noise) CU(cudaMemcpyAsync(d_noise, noise, b_n, cudaMemcpyHostToDevice, st));
        if (n_tubes > 0) CU(cudaMemcpyAsync(d_tubes, tubes, sizeof(double) * 2 * n_tubes, cudaMemcpyHostToDevice, st));
        p.cmd = d_cmd;
        p.noise = noise ? d_noise : nullptr;
        p.tubes = d_tubes;
    }
    cudaError_t e = nuslam::launch_world_step(p, device, st);
    if (e == cudaSuccess && mem == NUSLAM_HOST)
    {
        e = cudaMemcpyAsync(world, p.world, b_w, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(ranges_out, p.ranges, b_r, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess && joints_out) e = cudaMemcpyAsync(joints_out, p.joints, b_j, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    if (tmp) cudaFree(tmp);
    if (e != cudaSuccess) return cuda_fail(e, "world_step");
    return NUSLAM_OK;
}

int nuslam_diffdrive_convert_twist(double wheel_base, double wheel_rad, const double * twists, double * wheel_vel_out, int64_t count, int mem,
                                   int device, void * cuda_stream)
{
    if (!twists || !wheel_vel_out || count < 0) return fail(NUSLAM_ERR_INVALID, "null argument");
    if (count == 0) return NUSLAM_OK;
    CU(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    const double * d_tw = twists;
    double * d_u = wheel_vel_out;
    double * tmp = nullptr;
    if (mem == NUSLAM_HOST)
    {
        CU(cudaMalloc(&tmp, sizeof(double) * count * 5));
        CU(cudaMemcpyAsync(tmp, twists, sizeof(double) * count * 3, cudaMemcpyHostToDevice, st));
        d_tw = tmp;
        d_u = tmp + 3 * count;
    }
    const int threads = 128;
    nuslam::k_diffdrive_convert_twist<<<(unsigned) ((count + threads - 1) / threads), threads, 0, st>>>(wheel_base, wheel_rad, d_tw, d_u, count);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && mem == NUSLAM_HOST)
    {
        e = cudaMemcpyAsync(wheel_vel_out, d_u, sizeof(double) * count * 2, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    if (tmp) cudaFree(tmp);
    if (e != cudaSuccess) return cuda_fail(e, "diffdrive_convert_twist");
    return NUSLAM_OK;
}

int nuslam_scan_set_fit(int mode)
{
    const int prev = nuslam::scan_fit_mode();
    if (mode == NUSLAM_FIT_MOMENT || mode == NUSLAM_FIT_JACOBI) nuslam::scan_fit_mode() = mode;
    return prev;
}

int nuslam_scan_last_fallbacks(int device)
{
    if (cudaSetDevice(device) != cudaSuccess) return -1;
    return nuslam::scan_moment_fallbacks(device);
}

int nuslam_scan_detect(const float * ranges, int64_t n_scans, double min_range, double max_range, int16_t * cluster_of_beam,
                       int32_t * n_clusters, int32_t * n_circles, double * circles, int32_t max_circles, int mem, int device,
                       void * cuda_stream)
{
    if (!ranges || !n_clusters || !n_circles || !circles || n_scans < 0 || max_circles < 1)
        return fail(NUSLAM_ERR_INVALID, "null argument or bad sizes");
    if (n_scans == 0) return NUSLAM_OK;
    CU(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    const float * d_ranges = ranges;
    int16_t * d_cob = cluster_of_beam;
    int32_t * d_ncl = n_clusters;
    int32_t * d_nci = n_circles;
    double * d_circ = circles;
    char * tmp = nullptr;
    const size_t b_r = sizeof(float) * 360 * n_scans, b_cob = sizeof(int16_t) * 360 * n_scans;
    const size_t b_n = sizeof(int32_t) * n_scans, b_c = sizeof(double) * 4 * max_circles * n_scans;
    if (mem == NUSLAM_HOST)
    {
        auto al = [](size_t v) { return (v + 255) & ~(size_t) 255; };
        CU(cudaMalloc(&tmp, al(b_r) + al(b_cob) + 2 * al(b_n) + al(b_c)));
        char * q = tmp;
        d_ranges = reinterpret_cast<float *>(q);
        q += al(b_r);
        d_cob = reinterpret_cast<int16_t *>(q);
        q += al(b_cob);
        d_ncl = reinterpret_cast<int32_t *>(q);
        q += al(b_n);
        d_nci = reinterpret_cast<int32_t *>(q);
        q += al(b_n);
        d_circ = reinterpret_cast<double *>(q);
        CU(cudaMemcpyAsync(const_cast<float *>(d_ranges), ranges, b_r, cudaMemcpyHostToDevice, st));
    }
    int sm_count = 0;
    cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device);
    cudaError_t e = (nuslam::scan_fit_mode() == nuslam::kFitMoment ? nuslam::launch_scan_moment : nuslam::launch_scan_detect)(
        d_ranges, n_scans, min_range, max_range, cluster_of_beam ? d_cob : nullptr, d_ncl, d_nci, d_circ, max_circles, NUSLAM_SCAN_UB, device,
        sm_count > 0 ? sm_count : 148, st);
    if (e == cudaSuccess && mem == NUSLAM_HOST)
    {
        if (cluster_of_beam) e = cudaMemcpyAsync(cluster_of_beam, d_cob, b_cob, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(n_clusters, d_ncl, b_n, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(n_circles, d_nci, b_n, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(circles, d_circ, b_c, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    if (tmp) cudaFree(tmp);
    if (e != cudaSuccess) return cuda_fail(e, "scan_detect");
    return NUSLAM_OK;
}

int nuslam_classify_and_fit(const double * px, const double * py, const int32_t * offsets, int64_t n_clusters, int32_t * is_circle,
                            double * fit, int mem, int device, void * cuda_stream)
{
    if (!px || !py || !offsets || !is_circle || !fit || n_clusters < 0) return fail(NUSLAM_ERR_INVALID, "null argument");
    if (n_clusters == 0) return NUSLAM_OK;
    CU(cudaSetDevice(device));
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    const double * d_px = px;
    const double * d_py = py;
    const int32_t * d_off = offsets;
    int32_t * d_is = is_circle;
    double * d_fit = fit;
    char * tmp = nullptr;
    if (mem == NUSLAM_HOST)
    {
        const int64_t npts = offsets[n_clusters];
        auto al = [](size_t v) { return (v + 255) & ~(size_t) 255; };
        const size_t b_p = al(sizeof(double) * npts), b_o = al(sizeof(int32_t) * (n_clusters + 1));
        const size_t b_i = al(sizeof(int32_t) * n_clusters), b_f = al(sizeof(double) * 4 * n_clusters);
        CU(cudaMalloc(&tmp, 2 * b_p + b_o + b_i + b_f));
        char * q = tmp;
        CU(cudaMemcpyAsync(q, px, sizeof(double) * npts, cudaMemcpyHostToDevice, st));
        d_px = reinterpret_cast<double *>(q);
        q += b_p;
        CU(cudaMemcpyAsync(q, py, sizeof(double) * npts, cudaMemcpyHostToDevice, st));
        d_py = reinterpret_cast<double *>(q);
        q += b_p;
        CU(cudaMemcpyAsync(q, offsets, sizeof(int32_t) * (n_clusters + 1), cudaMemcpyHostToDevice, st));
        d_off = reinterpret_cast<int32_t *>(q);
        q += b_o;
        d_is = reinterpret_cast<int32_t *>(q);
        q += b_i;
        d_fit = reinterpret_cast<double *>(q);
    }
    // work matrices of the Jacobi SVD: 4 doubles per point
    int32_t npts_total = 0;
    if (mem == NUSLAM_HOST) npts_total = offsets[n_clusters];
    else CU(cudaMemcpyAsync(&npts_total, offsets + n_clusters, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (mem != NUSLAM_HOST) CU(cudaStreamSynchronize(st));
    double * scratch = nullptr;
    CU(cudaMalloc(&scratch, sizeof(double) * 4 * (size_t) (npts_total > 0 ? npts_total : 1)));
    const int threads = 128;
    const int64_t blocks = (n_clusters + threads - 1) / threads;
    nuslam::k_classify_and_fit<<<(unsigned) blocks, threads, 0, st>>>(d_px, d_py, d_off, n_clusters, d_is, d_fit, scratch);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && mem != NUSLAM_HOST) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess && mem == NUSLAM_HOST)
    {
        e = cudaMemcpyAsync(is_circle, d_is, sizeof(int32_t) * n_clusters, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(fit, d_fit, sizeof(double) * 4 * n_clusters, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    if (tmp) cudaFree(tmp);
    if (scratch) cudaFree(scratch);
    if (e != cudaSuccess) return cuda_fail(e, "classify_and_fit");
    return NUSLAM_OK;
}

}   // extern "C"
