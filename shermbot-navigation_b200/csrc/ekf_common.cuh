// ekf_common.cuh -- shared device helpers of the batched EKF-SLAM kernels (sm_100a).
//
// Reference semantics restated here (paths relative to the reference repo):
//   nuslam/src/slam_library.cpp:16-22    cartesian2polar
//   nuslam/src/slam_library.cpp:150-186  computeTheoreticalMeasurement / linearizedMeasurementModel
//   rigid2d/src/rigid2d.cpp:9-13         normalize_angle = atan2(sin, cos)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace nuslam
{

constexpr int kWarp = 32;
constexpr double kLandmarkPrior = 2147483647.0;   // INT_MAX, slam_library.cpp:30
// a landmark whose variance is still above this is "untouched": (I-KH)Sigma cancels catastrophically
// and only the reference's own operation order reproduces its result (SURVEY.md Appendix B)
constexpr double kFirstTouchVariance = 1.0e6;

// status bits / sentinel: keep in sync with include/nuslam_b200.h
constexpr int kStatusMapFull = 1;
constexpr int kStatusSingular = 2;
constexpr int kStatusBadId = 4;
constexpr int kStatusAssocTruncated = 8;
constexpr int kIdException = -1000;
// opt-in departures from the reference: keep in sync with NUSLAM_OPT_* in include/nuslam_b200.h
constexpr unsigned kOptWrapInnovation = 1u, kOptJoseph = 2u, kOptPreMotionJacobian = 4u, kOptNearestNeighbour = 8u;
constexpr unsigned kOptJointCompatibility = 32u;

// Function attributes and __device__ tables are per DEVICE (per context): one-time setup is remembered per device ordinal, so that
// a process driving several GPUs (one handle each) configures every one of them. Races between host threads are benign (the setup
// is idempotent).
constexpr int kMaxDevices = 64;
inline int device_slot()
{
    int dev = 0;
    cudaGetDevice(&dev);
    return (dev >= 0 && dev < kMaxDevices) ? dev : 0;
}

// unfused IEEE operations: nvcc never contracts these into FMAs, whatever -fmad says
__device__ __forceinline__ double mul_(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add_(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub_(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double div_(double a, double b) { return __ddiv_rn(a, b); }

// rigid2d::normalize_angle (rigid2d.cpp:9-13)
__device__ __forceinline__ double normalize_angle(double rad)
{
    double s, c;
    sincos(rad, &s, &c);
    return atan2(s, c);
}

// the 8 data-dependent entries of H_j (slam_library.cpp:175-183); H(0,0) = 0 and H(1,0) = -1 are constants
struct HEntries
{
    double h01, h02, h0c, h0c1;   // row 0: columns 1, 2, c, c+1
    double h11, h12, h1c, h1c1;   // row 1: columns 1, 2, c, c+1
};

// H_j and z_hat_j at state x; c = 3 + 2(j-1). Exactly the reference's operations: + - * / sqrt are IEEE on
// both sides; sin/cos/atan2 come from the CUDA math library (<= 2 ulp from glibc's).
__device__ __forceinline__ void measurement_model(const double * x, int c, HEntries & H, double & zr, double & zb)
{
    const double dx = sub_(x[c], x[1]);
    const double dy = sub_(x[c + 1], x[2]);
    const double d = add_(mul_(dx, dx), mul_(dy, dy));
    const double sq = sqrt(d);
    H.h01 = div_(-dx, sq);
    H.h11 = div_(dy, d);
    H.h02 = div_(-dy, sq);
    H.h12 = div_(-dx, d);
    H.h0c = div_(dx, sq);
    H.h1c = div_(-dy, d);
    H.h0c1 = div_(dy, sq);
    H.h1c1 = div_(dx, d);
    zr = sq;                                         // cartesian2polar range: sqrt(mx^2 + my^2), same operands
    const double b = normalize_angle(atan2(dy, dx));   // :20
    zb = normalize_angle(sub_(b, x[0]));             // :157
}

// closed-form 2x2 inverse in the oracle's operation order (oracle/shim/armadillo inv()); false when singular
__device__ __forceinline__ bool inv2x2(double p, double q, double r, double s, double & i00, double & i01, double & i10, double & i11)
{
    const double det = sub_(mul_(p, s), mul_(q, r));
    if (det == 0.0) return false;
    i00 = div_(s, det);
    i01 = div_(-q, det);
    i10 = div_(-r, det);
    i11 = div_(p, det);
    return true;
}

// Nearest-neighbour association (NUSLAM_OPT_NEAREST_NEIGHBOUR): candidate (d1, k1) beats (d0, k0) in the lexicographic (d, k) order,
// an exact fp64 comparison with ties to the lower k. k = 0 is "no candidate" (none yet, or a NaN distance), which anything beats.
__device__ __forceinline__ bool nn_better(double d1, int k1, double d0, int k0) { return k1 != 0 && (k0 == 0 || d1 < d0 || (d1 == d0 && k1 < k0)); }

// the (d, k) minimum over a full warp by butterfly shuffles: every lane ends with the same winner, whatever order the lanes run in
__device__ __forceinline__ void nn_warp_min(double & d, int & k)
{
#pragma unroll
    for (int off = kWarp / 2; off > 0; off >>= 1)
    {
        const double od = __shfl_xor_sync(0xffffffffu, d, off);
        const int ok = __shfl_xor_sync(0xffffffffu, k, off);
        if (nn_better(od, ok, d, k))
        {
            d = od;
            k = ok;
        }
    }
}

}   // namespace nuslam
