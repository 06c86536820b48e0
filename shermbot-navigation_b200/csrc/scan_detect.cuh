// scan_detect.cuh -- batched laser-scan clustering + circle classification + Hyper algebraic circle fit (sm_100a).
//
// One warp per 360-beam scan. Reference semantics restated here (paths relative to the reference repo):
//   nuslam/src/circle_fit_library.cpp:136-206  clusterPoints   (sequential state machine over the beams)
//   nuslam/src/circle_fit_library.cpp:208-250  classifyCluster (population std of inscribed angles < 10 deg)
//   nuslam/src/circle_fit_library.cpp:15-134   circleFit       (SVD of Z, eig of Y Hinv Y, solve)
//   nuslam/src/landmarks.cpp:84-109            caller protocol (id < 0 skip, R > 1 skip, detection order)
// Parallel form of clusterPoints (SURVEY.md Appendix A-11): with inr_i = !(r_i > max || r_i < min),
// sim_i = |r_i - r_(i+1 mod 360)| < 0.04, closer_i = inr_i && !sim_i, the cluster of an in-range beam is the number of
// closers before it (warp ballots + popcounts); beams after the last closer form the open cluster the reference
// drops; beam 359 similar to beam 0 is appended to the END of cluster 0 (and the reference indexes clusters[0] of an
// empty vector when there is none: reported as NUSLAM_SCAN_UB); the erase loop's index skipping is a two-state
// walk over the clusters.
// circleFit is the reference's own algorithm, term by term (one-sided Jacobi SVD of the N x 4 data matrix in the
// oracle's sweep order, cyclic Jacobi eig_sym of the symmetrised 4 x 4, Gaussian elimination with partial pivoting;
// see oracle/shim/armadillo for the order the oracle defines), with unfused IEEE multiply/add and IEEE sqrt and
// division, one cluster per lane, its data matrix in shared memory. Only atan2 (classification) comes from the
// CUDA math library. Beam directions cos/sin(deg2rad(i)) (circle_fit_library.cpp:162-163) are a 360-entry
// constant table filled by the host once (host libm, bit-identical to what the reference multiplies with).
#pragma once
#include "ekf_common.cuh"
#include <math.h>
#include <string.h>

namespace nuslam
{

constexpr int kBeams = 360;
constexpr int kScanWarps = 2;   // scans per CTA
constexpr double kPiRef = 3.14159265358979323846;   // rigid2d.hpp:16

// beam directions cos / sin(deg2rad(i)) from the HOST libm (the reference's own values). In global memory, read through the
// read-only path: the lanes of a warp index them with different beams, which the constant cache would serialise.
__device__ double c_beam_cos[kBeams];
__device__ double c_beam_sin[kBeams];

// clustering state of one scan (one warp); the point and work-matrix arrays follow it only in the instantiation that also fits
struct ScanSmemHead
{
    float r[kBeams + 8];
    short cend[kBeams + 2];       // flat position of the last point of pre-erase cluster k
    short cbeam[kBeams + 2];      // beam index of that point (the closer)
    short newidx[kBeams + 2];     // index after the erase loop, -1 when erased
    short kept[kBeams + 2];       // pre-erase index of kept cluster q
    int nk;
    int pad[3];
};
struct ScanSmem : ScanSmemHead
{
    double px[kBeams + 2];        // points in the reference's stored order (flat over the pre-erase clusters); [361] = wrap point
    double py[kBeams + 2];
    double A[4 * (kBeams + 2)];   // Jacobi work matrices of the clusters being fitted (disjoint slices)
};
static_assert(sizeof(ScanSmemHead) % 16 == 0, "per-warp slices stay 16-byte aligned");
// per-warp shared-memory footprint: 4.4 KB for clustering only (22 resident warps per SM, register-bound), 21.8 KB with the fits
template <bool INLINE_FIT>
constexpr size_t scan_smem_stride() { return INLINE_FIT ? sizeof(ScanSmem) : sizeof(ScanSmemHead); }

// view of an m x 4 work matrix: element (i, c) at p[(i + c * ld) * stride] (stride > 1: interleaved over the threads of a CTA)
struct WorkMatrix
{
    double * p;
    int ld, stride;
    __device__ __forceinline__ double & operator()(int i, int c) const { return p[(i + c * ld) * stride]; }
};

// classifyCluster, circle_fit_library.cpp:208-250. Points P(0..n-1) in stored order.
template <typename PX, typename PY>
__device__ __forceinline__ bool classify_cluster(int n, PX X, PY Y)
{
    const double p2x = X(0), p2y = Y(0), p3x = X(n - 1), p3y = Y(n - 1);
    const int na = (n >= 2) ? n - 2 : 0;   // angles.size(): 0 for clusters of 1 or 2 points -> 0/0 = NaN -> not a circle
    double mean = 0.0;
    for (int i = 1; i < n - 1; ++i)
    {
        const double p1x = X(i), p1y = Y(i);
        // num = p2.y*(p1.x-p3.x) + p1.y*(p3.x-p2.x) + p3.y*(p2.x-p1.x); den = (p2.x-p1.x)*(p1.x-p3.x) + (p2.y-p1.y)*(p1.y-p3.y)
        const double num = add_(add_(mul_(p2y, sub_(p1x, p3x)), mul_(p1y, sub_(p3x, p2x))), mul_(p3y, sub_(p2x, p1x)));
        const double den = add_(mul_(sub_(p2x, p1x), sub_(p1x, p3x)), mul_(sub_(p2y, p1y), sub_(p1y, p3y)));
        const double ang = mul_(div_(180.0, kPiRef), atan2(num, den));   // rigid2d::rad2deg, rigid2d.hpp:49-53
        mean = add_(mean, div_(ang, (double) na));
    }
    double sd = 0.0;
    for (int i = 1; i < n - 1; ++i)
    {
        const double p1x = X(i), p1y = Y(i);
        const double num = add_(add_(mul_(p2y, sub_(p1x, p3x)), mul_(p1y, sub_(p3x, p2x))), mul_(p3y, sub_(p2x, p1x)));
        const double den = add_(mul_(sub_(p2x, p1x), sub_(p1x, p3x)), mul_(sub_(p2y, p1y), sub_(p1y, p3y)));
        const double ang = mul_(div_(180.0, kPiRef), atan2(num, den));
        const double dv = sub_(ang, mean);
        sd = add_(sd, mul_(dv, dv));   // pow(angle - mean, 2)
    }
    sd = sqrt(div_(sd, (double) na));   // na == 0 -> 0/0 = NaN -> false
    return sd < 10.0;
}

// one-sided (Hestenes) Jacobi SVD of the m x 4 matrix A (column-major, overwritten): singular values descending in s,
// right singular vectors in V (4 x 4 column-major). oracle/shim/armadillo svd().
__device__ inline void svd_n4(const WorkMatrix A, int m, double * s, double * V)
{
    double W[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) W[k] = (k % 5 == 0) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 60; ++sweep)
    {
        bool rotated = false;
#pragma unroll
        for (int p = 0; p < 3; ++p)
#pragma unroll
            for (int q = p + 1; q < 4; ++q)
            {
                double alpha = 0.0, beta = 0.0, gamma = 0.0;
                for (int i = 0; i < m; ++i)
                {
                    const double ap = A(i, p), aq = A(i, q);
                    alpha = add_(alpha, mul_(ap, ap));
                    beta = add_(beta, mul_(aq, aq));
                    gamma = add_(gamma, mul_(ap, aq));
                }
                const bool skip = (gamma == 0.0) || (fabs(gamma) <= 1e-300) ||
                                  (fabs(gamma) <= mul_(2.220446049250313e-16, sqrt(mul_(alpha, beta))));
                if (!skip)
                {
                    rotated = true;
                    const double zeta = div_(sub_(beta, alpha), mul_(2.0, gamma));
                    const double tt = div_((zeta >= 0.0 ? 1.0 : -1.0), add_(fabs(zeta), sqrt(add_(1.0, mul_(zeta, zeta)))));
                    const double c = div_(1.0, sqrt(add_(1.0, mul_(tt, tt))));
                    const double sn = mul_(c, tt);
                    for (int i = 0; i < m; ++i)
                    {
                        const double ap = A(i, p), aq = A(i, q);
                        A(i, p) = sub_(mul_(c, ap), mul_(sn, aq));
                        A(i, q) = add_(mul_(sn, ap), mul_(c, aq));
                    }
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                    {
                        const double wp = W[i + p * 4], wq = W[i + q * 4];
                        W[i + p * 4] = sub_(mul_(c, wp), mul_(sn, wq));
                        W[i + q * 4] = add_(mul_(sn, wp), mul_(c, wq));
                    }
                }
            }
        if (!rotated) break;
    }
    double norms[4];
#pragma unroll
    for (int j = 0; j < 4; ++j)
    {
        double acc = 0.0;
        for (int i = 0; i < m; ++i) acc = add_(acc, mul_(A(i, j), A(i, j)));
        norms[j] = sqrt(acc);
    }
    // stable insertion sort, descending (a 4-element network with the same tie behaviour); the columns of W travel with their
    // keys by selects -- no index array, so that W and norms stay in registers (a dynamically indexed array lives in local memory)
#pragma unroll
    for (int a = 1; a < 4; ++a)
    {
#pragma unroll
        for (int b = a; b > 0; --b)
        {
            const bool sw = norms[b - 1] < norms[b];
            const double k0 = norms[b - 1], k1 = norms[b];
            norms[b - 1] = sw ? k1 : k0;
            norms[b] = sw ? k0 : k1;
#pragma unroll
            for (int i = 0; i < 4; ++i)
            {
                const double w0 = W[i + (b - 1) * 4], w1 = W[i + b * 4];
                W[i + (b - 1) * 4] = sw ? w1 : w0;
                W[i + b * 4] = sw ? w0 : w1;
            }
        }
    }
#pragma unroll
    for (int jj = 0; jj < 4; ++jj)
    {
        s[jj] = norms[jj];
#pragma unroll
        for (int i = 0; i < 4; ++i) V[i + jj * 4] = W[i + jj * 4];
    }
}

// cyclic two-sided Jacobi on the symmetrised 4 x 4: eigenvalues ascending. oracle/shim/armadillo eig_sym().
__device__ inline void eig_sym4(const double * X, double * val, double * vec)
{
    double A[16], W[16];
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i)
        {
            A[i + j * 4] = mul_(0.5, add_(X[i + j * 4], X[j + i * 4]));
            W[i + j * 4] = (i == j) ? 1.0 : 0.0;
        }
    for (int sweep = 0; sweep < 100; ++sweep)
    {
        double off = 0.0, diag = 0.0;
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i)
            {
                if (i == j) diag = add_(diag, mul_(A[i + j * 4], A[i + j * 4]));
                else off = add_(off, mul_(A[i + j * 4], A[i + j * 4]));
            }
        if (off == 0.0 || off <= mul_(1e-40, diag)) break;
        // The oracle's loop practically never meets its criterion (the lower triangle, which no rotation targets, stalls at
        // ~1e-17 relative) and runs all 100 sweeps. Its OUTPUT is diag(A) and W. Once a whole sweep consists of rotations with
        // c == 1 exactly that leave diag(A) and W bit for bit unchanged, every later sweep does too: the off-diagonal entries
        // only keep shrinking (quadratically), so every later |sn| is smaller and sn * x stays below half an ulp of the entry it
        // would be added to. Stopping there returns exactly what sweep 100 would (checked bit for bit against the oracle).
        bool out_changed = false, all_c1 = true;
#pragma unroll
        for (int p = 0; p < 3; ++p)
#pragma unroll
            for (int q = p + 1; q < 4; ++q)
            {
                const double apq = A[p + q * 4];
                if (apq != 0.0)
                {
                    const double theta = div_(sub_(A[q + q * 4], A[p + p * 4]), mul_(2.0, apq));
                    const double tt = div_((theta >= 0.0 ? 1.0 : -1.0), add_(fabs(theta), sqrt(add_(1.0, mul_(theta, theta)))));
                    const double c = div_(1.0, sqrt(add_(1.0, mul_(tt, tt))));
                    const double sn = mul_(c, tt);
                    all_c1 &= (c == 1.0);
                    const double dpp = A[p + p * 4], dqq = A[q + q * 4];
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                    {
                        const double akp = A[k + p * 4], akq = A[k + q * 4];
                        A[k + p * 4] = sub_(mul_(c, akp), mul_(sn, akq));
                        A[k + q * 4] = add_(mul_(sn, akp), mul_(c, akq));
                    }
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                    {
                        const double apk = A[p + k * 4], aqk = A[q + k * 4];
                        A[p + k * 4] = sub_(mul_(c, apk), mul_(sn, aqk));
                        A[q + k * 4] = add_(mul_(sn, apk), mul_(c, aqk));
                    }
                    out_changed |= !(A[p + p * 4] == dpp) | !(A[q + q * 4] == dqq);
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                    {
                        const double wp = W[k + p * 4], wq = W[k + q * 4];
                        const double n1 = sub_(mul_(c, wp), mul_(sn, wq)), n2 = add_(mul_(sn, wp), mul_(c, wq));
                        out_changed |= !(n1 == wp) | !(n2 == wq);
                        W[k + p * 4] = n1;
                        W[k + q * 4] = n2;
                    }
                }
            }
        if (!out_changed && all_c1) break;
    }
    // ascending stable insertion sort of (eigenvalue, eigenvector column) pairs by selects (no index array: registers only)
    double key[4] = {A[0], A[5], A[10], A[15]};
#pragma unroll
    for (int a = 1; a < 4; ++a)
    {
#pragma unroll
        for (int b = a; b > 0; --b)
        {
            const bool sw = key[b - 1] > key[b];
            const double k0 = key[b - 1], k1 = key[b];
            key[b - 1] = sw ? k1 : k0;
            key[b] = sw ? k0 : k1;
#pragma unroll
            for (int i = 0; i < 4; ++i)
            {
                const double w0 = W[i + (b - 1) * 4], w1 = W[i + b * 4];
                W[i + (b - 1) * 4] = sw ? w1 : w0;
                W[i + b * 4] = sw ? w0 : w1;
            }
        }
    }
#pragma unroll
    for (int jj = 0; jj < 4; ++jj)
    {
        val[jj] = key[jj];
#pragma unroll
        for (int i = 0; i < 4; ++i) vec[i + jj * 4] = W[i + jj * 4];
    }
}

// Gaussian elimination with partial pivoting, 4 x 4. oracle/shim/armadillo solve(). false when singular.
__device__ inline bool solve4(const double * Ain, const double * b, double * x)
{
    double A[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) A[k] = Ain[k];
#pragma unroll
    for (int k = 0; k < 4; ++k) x[k] = b[k];
#pragma unroll
    for (int c = 0; c < 4; ++c)
    {
        // partial pivoting without a dynamic row index (registers only): the first row of maximal |A(r, c)|, then a select-swap
        int piv = c;
        double best = fabs(A[c + c * 4]);
#pragma unroll
        for (int r = c + 1; r < 4; ++r)
        {
            const double v = fabs(A[r + c * 4]);
            const bool gt = v > best;
            piv = gt ? r : piv;
            best = gt ? v : best;
        }
        if (best == 0.0) return false;
#pragma unroll
        for (int r = c + 1; r < 4; ++r)
        {
            const bool sw = (piv == r);
#pragma unroll
            for (int k = 0; k < 4; ++k)
            {
                const double t0 = A[r + k * 4], t1 = A[c + k * 4];
                A[r + k * 4] = sw ? t1 : t0;
                A[c + k * 4] = sw ? t0 : t1;
            }
            const double u0 = x[r], u1 = x[c];
            x[r] = sw ? u1 : u0;
            x[c] = sw ? u0 : u1;
        }
#pragma unroll
        for (int r = c + 1; r < 4; ++r)
        {
            const double fct = div_(A[r + c * 4], A[c + c * 4]);
            if (fct != 0.0)
            {
#pragma unroll
                for (int k = c; k < 4; ++k) A[r + k * 4] = sub_(A[r + k * 4], mul_(fct, A[c + k * 4]));
                x[r] = sub_(x[r], mul_(fct, x[c]));
            }
        }
    }
#pragma unroll
    for (int ii = 3; ii >= 0; --ii)
    {
        double acc = x[ii];
#pragma unroll
        for (int j = ii + 1; j < 4; ++j) acc = sub_(acc, mul_(A[ii + j * 4], x[j]));
        x[ii] = div_(acc, A[ii + ii * 4]);
    }
    return true;
}

__device__ __forceinline__ void mm4(double * C, const double * A, const double * B)
{
    // oracle/shim/armadillo operator*: C(i,j) = sum_k A(i,k) B(k,j), ascending k, unfused
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i)
        {
            double acc = 0.0;
#pragma unroll
            for (int k = 0; k < 4; ++k) acc = add_(acc, mul_(A[i + k * 4], B[k + j * 4]));
            C[i + j * 4] = acc;
        }
}

constexpr int kFitException = -1000;   // solve() on a singular Y: Armadillo throws

// circleFit after the SVD (circle_fit_library.cpp:78-125): A from sigma_4 / the eigenproblem of Y Hinv Y, then centre and radius
__device__ inline int circle_fit_tail(const double * s, const double * V, double z_bar, double x_hat, double y_hat, double * out3)
{
    double Aco[4];
    if (s[3] < 1e-12)   // :78-80
    {
#pragma unroll
        for (int i = 0; i < 4; ++i) Aco[i] = V[i + 12];
    }
    else
    {
        double Hinv[16], D[16], VD[16], Vt[16], Yq[16], YH[16], Q[16];
#pragma unroll
        for (int k = 0; k < 16; ++k)
        {
            Hinv[k] = 0.0;
            D[k] = 0.0;
        }
        Hinv[5] = 1.0;
        Hinv[10] = 1.0;
        Hinv[0 + 3 * 4] = 0.5;
        Hinv[3 + 0 * 4] = 0.5;
        Hinv[15] = mul_(-2.0, z_bar);
#pragma unroll
        for (int i = 0; i < 4; ++i) D[i * 5] = s[i];
        mm4(VD, V, D);   // Y = V * diagmat(s) * V.t() (:82)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i) Vt[i + j * 4] = V[j + i * 4];
        mm4(Yq, VD, Vt);
        mm4(YH, Yq, Hinv);   // Q = Y * Hinv * Y (:83)
        mm4(Q, YH, Yq);
        double eigval[4], eigvec[16];
        eig_sym4(Q, eigval, eigvec);
        int eig_index = 0;
        double eig_max = 2147483647.0;   // INT_MAX (:92)
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (eigval[i] > 0.0 && eigval[i] < eig_max)
            {
                eig_index = i;
                eig_max = eigval[i];
            }
        double Astar[4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
            Astar[i] = (eig_index == 0) ? eigvec[i] : (eig_index == 1) ? eigvec[i + 4] : (eig_index == 2) ? eigvec[i + 8] : eigvec[i + 12];
        if (!solve4(Yq, Astar, Aco)) return kFitException;
    }
    const double a = div_(-Aco[1], mul_(2.0, Aco[0]));
    const double b = div_(-Aco[2], mul_(2.0, Aco[0]));
    const double R2 = div_(sub_(add_(mul_(Aco[1], Aco[1]), mul_(Aco[2], Aco[2])), mul_(mul_(4.0, Aco[0]), Aco[3])),
                           mul_(4.0, mul_(Aco[0], Aco[0])));
    const double tube_radius = sqrt(R2);
    out3[0] = add_(a, x_hat);
    out3[1] = add_(b, y_hat);
    out3[2] = div_(mul_(2.0, tube_radius), 2.0);   // scale.x = 2R (:124); callers read scale.x / 2 (landmarks.cpp:95)
    return 0;
}

// circleFit, circle_fit_library.cpp:15-134. Z (work matrix, N x 4 column-major) lives in shared memory.
// Returns marker.id (0, or -1 when N < 4); out = (pose.x, pose.y, scale.x / 2).
template <typename PX, typename PY>
__device__ inline int circle_fit(int N, PX X, PY Y, const WorkMatrix Z, double * out3)
{
    out3[0] = out3[1] = out3[2] = 0.0;
    double x_hat = 0.0, y_hat = 0.0;
    for (int i = 0; i < N; ++i)
    {
        x_hat = add_(x_hat, div_(X(i), (double) N));   // :23-24, size_t divisor converts to double
        y_hat = add_(y_hat, div_(Y(i), (double) N));
    }
    double z_bar = 0.0;
    for (int j = 0; j < N; ++j)
    {
        const double dx = sub_(X(j), x_hat), dy = sub_(Y(j), y_hat);
        const double z = add_(mul_(dx, dx), mul_(dy, dy));   // pow(x, 2) + pow(y, 2)
        z_bar = add_(z_bar, div_(z, (double) N));
        Z(j, 0) = z;
        Z(j, 1) = dx;
        Z(j, 2) = dy;
        Z(j, 3) = 1.0;
    }
    if (N < 4) return -1;   // s.size() < 4 (:72-76)
    double s[4], V[16];
    svd_n4(Z, N, s, V);
    return circle_fit_tail(s, V, z_bar, x_hat, y_hat, out3);
}

// Work list of the two-stage pipeline: one entry per kept cluster of the chunk of scans in flight
struct ClusterDesc
{
    int32_t scan;          // scan index (global)
    int32_t beams;         // first beam to examine | last beam << 16 (out-of-range beams in between are skipped)
    int32_t n_wrap;        // number of points | wrap flag << 16 (beam 359 appended last)
    int32_t q;             // index among the scan's returned clusters
};
struct ClusterFit
{
    double pub, cx, cy, R;   // pub = 1: published by the landmarks node (classified circle, id >= 0, R <= 1)
};
constexpr int kFitNMax = 32;        // clusters up to this many points are fitted one per THREAD (work matrix interleaved in shared memory)
constexpr int kFitThreads = 64;
constexpr int kBigSmallCtas = 5;    // resident CTAs (of 4 warps) per SM of the first warp-per-cluster class (96 registers per thread; measured best of 4 / 5)
constexpr int kFitBigSmall = 126;   // largest cluster of the first warp-per-cluster class
constexpr int kFitCtas = 8;     // CTAs of the first class per SM
constexpr int kFitSmall = 12;   // largest cluster of the first size class (work matrix kFitSmall x 4 doubles per thread)
constexpr int kMaxFastClusters = 32;   // scans returning more clusters than this take the one-warp-per-scan path

struct ScanPipe
{
    ClusterDesc * desc;      // chunk * kMaxFastClusters
    ClusterFit * fit;        // same
    int32_t * big;           // indices into desc of clusters with more than kFitBigSmall points
    int32_t * big_s;         // indices into desc of clusters with kFitNMax + 1 .. kFitBigSmall points
    int32_t * mid;           // indices into desc of clusters with kFitSmall + 1 .. kFitNMax points
    int32_t * slow;          // scans (global index) with more than kMaxFastClusters clusters
    int32_t * scan_base;     // per scan of the chunk: first entry in desc, -1 for slow / UB scans
    int32_t * counters;      // [0] entries in desc, [1] entries in big, [2] entries in slow, [3] entries in mid, [4] entries in big_s
    int64_t scan0;           // first scan of the chunk
};

// One warp per scan. cluster_of_beam may be null. INLINE_FIT: classification + fit by the same warp, one cluster per lane
// (latency path for a few scans, and the slow path of the pipeline: `list` then names the scans); !INLINE_FIT: stage 1 of the
// pipeline -- clustering only, kept clusters appended to the work list.
template <bool INLINE_FIT>
__global__ void __launch_bounds__(32 * kScanWarps)
k_scan_detect(const float * __restrict__ ranges, int64_t n_scans, double min_range, double max_range, int16_t * __restrict__ cluster_of_beam,
              int32_t * __restrict__ n_clusters, int32_t * __restrict__ n_circles, double * __restrict__ circles, int max_circles, int scan_ub,
              const int32_t * __restrict__ list, const int32_t * __restrict__ list_count, ScanPipe pipe)
{
    extern __shared__ __align__(16) unsigned char scan_smem_raw[];
    // the clustering-only instantiation never touches px / py / A: its slices are ScanSmemHead-sized
    ScanSmem & sm = *reinterpret_cast<ScanSmem *>(scan_smem_raw + (threadIdx.x >> 5) * scan_smem_stride<INLINE_FIT>());
    const int lane = threadIdx.x & 31;
    constexpr unsigned kFull = 0xffffffffu;
    constexpr int kChunks = (kBeams + 31) / 32;   // 12
    const int64_t n_work = list ? (int64_t) *list_count : n_scans;
    for (int64_t w = (int64_t) blockIdx.x * kScanWarps + (threadIdx.x >> 5); w < n_work; w += (int64_t) gridDim.x * kScanWarps)
    {
        const int64_t s = list ? (int64_t) list[w] : (INLINE_FIT ? w : pipe.scan0 + w);
        const float * rs = ranges + s * kBeams;
        for (int i = lane; i < kBeams; i += 32) sm.r[i] = rs[i];
        __syncwarp();
        if (lane == 0) sm.r[kBeams] = sm.r[0];
        __syncwarp();
        // ---- per-beam predicates and their ballots ----
        unsigned inr_m[kChunks], clo_m[kChunks];
        bool wrap = false;
#pragma unroll
        for (int k = 0; k < kChunks; ++k)
        {
            const int i = 32 * k + lane;
            bool inr = false, sim = false;
            if (i < kBeams)
            {
                const float r = sm.r[i];
                inr = !(((double) r > max_range) || ((double) r < min_range));           // :149, NaN counts as in range
                sim = fabs((double) r - (double) sm.r[i + 1]) < 0.04;                    // :166
            }
            inr_m[k] = __ballot_sync(kFull, inr);
            clo_m[k] = __ballot_sync(kFull, inr && !sim);
            if (k == kChunks - 1) wrap = ((inr_m[k] >> ((kBeams - 1) & 31)) & 1u) && !((clo_m[k] >> ((kBeams - 1) & 31)) & 1u);
        }
        // beam 359 in range and similar to beam 0: it is not stored in the flat list but appended to cluster 0
        if (wrap) inr_m[kChunks - 1] &= ~(1u << ((kBeams - 1) & 31));
        int nc = 0;
#pragma unroll
        for (int k = 0; k < kChunks; ++k) nc += __popc(clo_m[k]);
        int64_t sb = s * kBeams;
        if (wrap && nc == 0)
        {
            // clusters[0].push_back on an empty vector (:173): undefined behaviour in the reference
            if (cluster_of_beam)
                for (int i = lane; i < kBeams; i += 32) cluster_of_beam[sb + i] = -1;
            if (lane == 0)
            {
                n_clusters[s] = 0;
                n_circles[s] = scan_ub;
                if (!INLINE_FIT) pipe.scan_base[s - pipe.scan0] = -1;
            }
            __syncwarp();
            continue;
        }
        // ---- flat positions, cluster ends, points ----
        int pos_base = 0, clu_base = 0;
        int my_pos[kChunks], my_clu[kChunks];
        const unsigned lt = (1u << lane) - 1u;
#pragma unroll
        for (int k = 0; k < kChunks; ++k)
        {
            const int i = 32 * k + lane;
            const bool inr = (inr_m[k] >> lane) & 1u, clo = (clo_m[k] >> lane) & 1u;
            my_pos[k] = pos_base + __popc(inr_m[k] & lt);
            my_clu[k] = clu_base + __popc(clo_m[k] & lt);
            if (inr)
            {
                if (INLINE_FIT)
                {
                    const double r = (double) sm.r[i];
                    sm.px[my_pos[k]] = mul_(r, __ldg(&c_beam_cos[i]));   // :162-163
                    sm.py[my_pos[k]] = mul_(r, __ldg(&c_beam_sin[i]));
                }
                if (clo)
                {
                    sm.cend[my_clu[k]] = (short) my_pos[k];
                    sm.cbeam[my_clu[k]] = (short) i;
                }
            }
            pos_base += __popc(inr_m[k]);
            clu_base += __popc(clo_m[k]);
        }
        if (INLINE_FIT && wrap && lane == 0)
        {
            const double r = (double) sm.r[kBeams - 1];
            sm.px[kBeams + 1] = mul_(r, __ldg(&c_beam_cos[kBeams - 1]));
            sm.py[kBeams + 1] = mul_(r, __ldg(&c_beam_sin[kBeams - 1]));
        }
        __syncwarp();
        // ---- erase loop (:198-204): a cluster following an erased one is never examined ----
        if (lane == 0)
        {
            int nk = 0;
            bool unchecked = false;
            int prev_end = -1;
            for (int k = 0; k < nc; ++k)
            {
                const int e = sm.cend[k];
                const int size = e - prev_end + ((k == 0 && wrap) ? 1 : 0);
                prev_end = e;
                if (!unchecked && size < 3)
                {
                    sm.newidx[k] = -1;
                    unchecked = true;
                }
                else
                {
                    sm.newidx[k] = (short) nk;
                    sm.kept[nk] = (short) k;
                    ++nk;
                    unchecked = false;
                }
            }
            sm.nk = nk;
        }
        __syncwarp();
        const int nk = sm.nk;
        if (cluster_of_beam)
        {
#pragma unroll
            for (int k = 0; k < kChunks; ++k)
            {
                const int i = 32 * k + lane;
                if (i < kBeams)
                {
                    const bool inr = (inr_m[k] >> lane) & 1u;
                    int out = -1;
                    if (inr && my_clu[k] < nc) out = sm.newidx[my_clu[k]];
                    if (wrap && i == kBeams - 1) out = sm.newidx[0];
                    cluster_of_beam[sb + i] = (int16_t) out;
                }
            }
        }
        if (!INLINE_FIT)
        {
            // ---- stage 1 of the pipeline: hand the kept clusters to the fitting kernels ----
            int base = -1;
            if (nk > kMaxFastClusters)
            {
                if (lane == 0) pipe.slow[atomicAdd(&pipe.counters[2], 1)] = (int32_t) s;   // cluster_of_beam is final; the rest is redone there
            }
            else
            {
                if (lane == 0) base = atomicAdd(&pipe.counters[0], nk);
                base = __shfl_sync(kFull, base, 0);
                if (lane < nk)
                {
                    const int k = sm.kept[lane];
                    const int start = (k == 0) ? 0 : sm.cend[k - 1] + 1;
                    const bool wr = (k == 0) && wrap;
                    const int n = sm.cend[k] - start + 1 + (wr ? 1 : 0);
                    ClusterDesc d;
                    d.scan = (int32_t) s;
                    d.beams = ((k == 0) ? 0 : sm.cbeam[k - 1] + 1) | ((int) sm.cbeam[k] << 16);
                    d.n_wrap = n | (wr ? 1 << 16 : 0);
                    d.q = lane;
                    pipe.desc[base + lane] = d;
                    if (n > kFitBigSmall) pipe.big[atomicAdd(&pipe.counters[1], 1)] = base + lane;
                    else if (n > kFitNMax) pipe.big_s[atomicAdd(&pipe.counters[4], 1)] = base + lane;
                    else if (n > kFitSmall) pipe.mid[atomicAdd(&pipe.counters[3], 1)] = base + lane;
                }
            }
            if (lane == 0)
            {
                n_clusters[s] = nk;
                n_circles[s] = 0;
                pipe.scan_base[s - pipe.scan0] = (nk > kMaxFastClusters) ? -1 : base;
            }
            __syncwarp();
            continue;
        }
        // ---- classification + circle fit, one kept cluster per lane; publication in detection order ----
        int published = 0;
        double * cout = circles + s * (int64_t) max_circles * 4;
        for (int q0 = 0; q0 < nk; q0 += 32)
        {
            const int q = q0 + lane;
            bool pub = false;
            double fit[3] = {0.0, 0.0, 0.0};
            if (q < nk)
            {
                const int k = sm.kept[q];
                const int start = (k == 0) ? 0 : sm.cend[k - 1] + 1;
                const int nmain = sm.cend[k] - start + 1;
                const bool wr = (k == 0) && wrap;
                const int n = nmain + (wr ? 1 : 0);
                const double * bx = sm.px + start;
                const double * by = sm.py + start;
                const double wx = sm.px[kBeams + 1], wy = sm.py[kBeams + 1];
                auto X = [&](int i) { return (i < nmain) ? bx[i] : wx; };
                auto Y = [&](int i) { return (i < nmain) ? by[i] : wy; };
                if (classify_cluster(n, X, Y))
                {
                    const WorkMatrix Z = {sm.A + 4 * (start + (k > 0 ? 1 : 0)), n, 1};
                    const int id = circle_fit(n, X, Y, Z, fit);
                    pub = (id >= 0) && !(fit[2] > 1.0);   // landmarks.cpp:91-97
                }
            }
            const unsigned pm = __ballot_sync(kFull, pub);
            if (pub)
            {
                const int slot = published + __popc(pm & lt);
                if (slot < max_circles)
                {
                    cout[4 * slot + 0] = fit[0];
                    cout[4 * slot + 1] = fit[1];
                    cout[4 * slot + 2] = fit[2];
                    cout[4 * slot + 3] = (double) q;
                }
            }
            published += __popc(pm);
        }
        if (lane == 0)
        {
            n_clusters[s] = nk;
            n_circles[s] = published;
        }
        __syncwarp();
    }
}

// circle_fit::classifyCluster / circleFit on explicit point lists: one cluster per thread, work matrix in global scratch
__global__ void k_classify_and_fit(const double * __restrict__ px, const double * __restrict__ py, const int32_t * __restrict__ offsets,
                                   int64_t n_clusters, int32_t * __restrict__ is_circle, double * __restrict__ fit, double * __restrict__ scratch)
{
    const int64_t c = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_clusters) return;
    const int o = offsets[c], n = offsets[c + 1] - offsets[c];
    const double * bx = px + o;
    const double * by = py + o;
    auto X = [&](int i) { return bx[i]; };
    auto Y = [&](int i) { return by[i]; };
    is_circle[c] = (n >= 1 && classify_cluster(n, X, Y)) ? 1 : 0;
    double out3[3] = {0.0, 0.0, 0.0};
    int id = -1;
    if (n >= 1) id = circle_fit(n, X, Y, WorkMatrix{scratch + 4 * (int64_t) o, n, 1}, out3);
    fit[4 * c + 0] = (double) id;
    fit[4 * c + 1] = out3[0];
    fit[4 * c + 2] = out3[1];
    fit[4 * c + 3] = out3[2];
}

// host: fill the beam-direction table once per device with the host libm (the reference's own cos / sin)
inline cudaError_t scan_tables_init(int device)
{
    static bool done[64] = {false};
    if (device >= 0 && device < 64 && done[device]) return cudaSuccess;
    double hc[kBeams], hs[kBeams];
    for (int i = 0; i < kBeams; ++i)
    {
        const double rad = (kPiRef / (double) 180) * (double) i;   // rigid2d::deg2rad, rigid2d.hpp:40-44
        hc[i] = cos(rad);
        hs[i] = sin(rad);
    }
    cudaError_t e = cudaMemcpyToSymbol(c_beam_cos, hc, sizeof(hc));
    if (e != cudaSuccess) return e;
    e = cudaMemcpyToSymbol(c_beam_sin, hs, sizeof(hs));
    if (e != cudaSuccess) return e;
    if (device >= 0 && device < 64) done[device] = true;
    return cudaSuccess;
}

// the cluster's points in stored order: in-range beams of [first, last], then beam 359 when the wrap rule appended it
template <typename F>
__device__ __forceinline__ int gather_points(const ClusterDesc & d, const float * __restrict__ ranges, double min_range, double max_range, F store)
{
    const float * rs = ranges + (int64_t) d.scan * kBeams;
    const int first = d.beams & 0xffff, last = d.beams >> 16;
    int i = 0;
    for (int bm = first; bm <= last; ++bm)
    {
        const float r = rs[bm];
        if (((double) r > max_range) || ((double) r < min_range)) continue;
        store(i, mul_((double) r, __ldg(&c_beam_cos[bm])), mul_((double) r, __ldg(&c_beam_sin[bm])));
        ++i;
    }
    if (d.n_wrap >> 16)
    {
        const float r = rs[kBeams - 1];
        store(i, mul_((double) r, __ldg(&c_beam_cos[kBeams - 1])), mul_((double) r, __ldg(&c_beam_sin[kBeams - 1])));
        ++i;
    }
    return i;
}

__device__ __forceinline__ void classify_and_publish(int n, const WorkMatrix Z, ClusterFit & out)
{
    // the points live in columns 1, 2 of the work matrix until circleFit overwrites them (after it has read them)
    auto X = [&](int i) { return Z(i, 1); };
    auto Y = [&](int i) { return Z(i, 2); };
    out.pub = 0.0;
    out.cx = out.cy = out.R = 0.0;
    if (classify_cluster(n, X, Y))
    {
        double fit[3];
        const int id = circle_fit(n, X, Y, Z, fit);
        if ((id >= 0) && !(fit[2] > 1.0))   // landmarks.cpp:91-97
        {
            out.pub = 1.0;
            out.cx = fit[0];
            out.cy = fit[1];
            out.R = fit[2];
        }
    }
}

// stage 2: one THREAD per cluster; work matrices interleaved over the CTA's threads in shared memory. Two instantiations: up to
// kFitSmall = 12 points straight from the work list (most tube clusters; 24 KB per CTA, 8 CTAs = 16 warps per SM: measured best
// of 8 / 10 / 12 / 16) and 13..32 points from their own dense list.
template <int NMAX, bool FROM_LIST>
__global__ void __launch_bounds__(kFitThreads) k_scan_fit_small(const float * __restrict__ ranges, double min_range, double max_range, ScanPipe pipe)
{
    extern __shared__ __align__(16) unsigned char fit_smem_raw[];
    double * base = reinterpret_cast<double *>(fit_smem_raw) + threadIdx.x;
    const WorkMatrix Z = {base, NMAX, kFitThreads};
    const int total = FROM_LIST ? pipe.counters[3] : pipe.counters[0];
    for (int w = blockIdx.x * kFitThreads + threadIdx.x; w < total; w += gridDim.x * kFitThreads)
    {
        const int idx = FROM_LIST ? pipe.mid[w] : w;
        const ClusterDesc d = pipe.desc[idx];
        const int n = d.n_wrap & 0xffff;
        if (n > NMAX) continue;   // a larger size class: another stage's cluster
        gather_points(d, ranges, min_range, max_range, [&](int i, double x, double y) {
            Z(i, 1) = x;
            Z(i, 2) = y;
        });
        ClusterFit out;
        classify_and_publish(n, Z, out);
        pipe.fit[idx] = out;
    }
}

// Warp-cooperative form of svd_n4 for large m: the products and the rotations are spread over the lanes, every SUM is still
// accumulated by lane 0 in ascending row order, so the result is bit-identical to the sequential routine.
__device__ inline void svd_n4_warp(double * A, int m, double * prod, int lane, double * s, double * V)
{
    constexpr unsigned kFull = 0xffffffffu;
    double W[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) W[k] = (k % 5 == 0) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 60; ++sweep)
    {
        bool rotated = false;
#pragma unroll
        for (int p = 0; p < 3; ++p)
#pragma unroll
            for (int q = p + 1; q < 4; ++q)
            {
                for (int i = lane; i < m; i += 32)
                {
                    const double ap = A[i + p * m], aq = A[i + q * m];
                    prod[i] = mul_(ap, ap);
                    prod[m + i] = mul_(aq, aq);
                    prod[2 * m + i] = mul_(ap, aq);
                }
                __syncwarp();
                // the three ordered sums side by side: lane 0 alpha, lane 1 beta, lane 2 gamma (each in the reference's order)
                double acc3 = 0.0;
                if (lane < 3)
                {
                    const double * pr = prod + lane * m;
#pragma unroll 4
                    for (int i = 0; i < m; ++i) acc3 = add_(acc3, pr[i]);
                }
                const double alpha = __shfl_sync(kFull, acc3, 0), beta = __shfl_sync(kFull, acc3, 1), gamma = __shfl_sync(kFull, acc3, 2);
                const bool skip = (gamma == 0.0) || (fabs(gamma) <= 1e-300) ||
                                  (fabs(gamma) <= mul_(2.220446049250313e-16, sqrt(mul_(alpha, beta))));
                if (!skip)
                {
                    rotated = true;
                    const double zeta = div_(sub_(beta, alpha), mul_(2.0, gamma));
                    const double tt = div_((zeta >= 0.0 ? 1.0 : -1.0), add_(fabs(zeta), sqrt(add_(1.0, mul_(zeta, zeta)))));
                    const double c = div_(1.0, sqrt(add_(1.0, mul_(tt, tt))));
                    const double sn = mul_(c, tt);
                    for (int i = lane; i < m; i += 32)
                    {
                        const double ap = A[i + p * m], aq = A[i + q * m];
                        A[i + p * m] = sub_(mul_(c, ap), mul_(sn, aq));
                        A[i + q * m] = add_(mul_(sn, ap), mul_(c, aq));
                    }
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                    {
                        const double wp = W[i + p * 4], wq = W[i + q * 4];
                        W[i + p * 4] = sub_(mul_(c, wp), mul_(sn, wq));
                        W[i + q * 4] = add_(mul_(sn, wp), mul_(c, wq));
                    }
                }
                __syncwarp();
            }
        if (!rotated) break;
    }
    double norms[4];
    {
        // the four column norms side by side: lane j squares and sums column j in the reference's order
        double acc = 0.0;
        if (lane < 4)
        {
            const double * col = A + lane * m;
#pragma unroll 4
            for (int i = 0; i < m; ++i) acc = add_(acc, mul_(col[i], col[i]));
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) norms[j] = sqrt(__shfl_sync(kFull, acc, j));
        __syncwarp();
    }
    // stable insertion sort, descending, by selects (registers only; same permutation as svd_n4)
#pragma unroll
    for (int a = 1; a < 4; ++a)
    {
#pragma unroll
        for (int b = a; b > 0; --b)
        {
            const bool sw = norms[b - 1] < norms[b];
            const double k0 = norms[b - 1], k1 = norms[b];
            norms[b - 1] = sw ? k1 : k0;
            norms[b] = sw ? k0 : k1;
#pragma unroll
            for (int i = 0; i < 4; ++i)
            {
                const double w0 = W[i + (b - 1) * 4], w1 = W[i + b * 4];
                W[i + (b - 1) * 4] = sw ? w1 : w0;
                W[i + b * 4] = sw ? w0 : w1;
            }
        }
    }
#pragma unroll
    for (int jj = 0; jj < 4; ++jj)
    {
        s[jj] = norms[jj];
#pragma unroll
        for (int i = 0; i < 4; ++i) V[i + jj * 4] = W[i + jj * 4];
    }
}

// stage 2b: clusters with more than 32 points (walls, very close tubes): one warp per cluster. classifyCluster's inscribed angles
// (one atan2 each) and the Jacobi SVD's products / rotations are spread over the lanes; every sum is accumulated by lane 0 in the
// reference's order, so the results are bit-identical to the sequential evaluation. The 4 x 4 tail (eig, solve) is replicated.
// Two capacities: up to kFitBigSmall points (7 KB of shared memory per warp: four times the resident warps, which is what hides the
// ordered sums' latency) and up to a whole scan.
template <int CAP, int WARPS, bool SMALL_LIST>
__global__ void __launch_bounds__(32 * WARPS, SMALL_LIST ? kBigSmallCtas : 5) k_scan_fit_big(const float * __restrict__ ranges, double min_range, double max_range, ScanPipe pipe)
{
    __shared__ double zbuf[WARPS][4 * CAP];
    __shared__ double angbuf[WARPS][3 * CAP];
    constexpr unsigned kFull = 0xffffffffu;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int total = SMALL_LIST ? pipe.counters[4] : pipe.counters[1];
    for (int w = blockIdx.x * WARPS + warp; w < total; w += gridDim.x * WARPS)
    {
        const int idx = SMALL_LIST ? pipe.big_s[w] : pipe.big[w];
        const ClusterDesc d = pipe.desc[idx];
        const int n = d.n_wrap & 0xffff;
        double * Zp = zbuf[warp];
        double * tmp = angbuf[warp];
        const WorkMatrix Z = {Zp, n, 1};
        // the cluster's points in stored order (gather_points, spread over the lanes: rank among the in-range beams by ballots)
        {
            const float * rs = ranges + (int64_t) d.scan * kBeams;
            const int first = d.beams & 0xffff, last = d.beams >> 16;
            int count = 0;
            for (int b0 = first; b0 <= last; b0 += 32)
            {
                const int bm = b0 + lane;
                float r = 0.0f;
                bool in = false;
                if (bm <= last)
                {
                    r = rs[bm];
                    in = !(((double) r > max_range) || ((double) r < min_range));
                }
                const unsigned bal = __ballot_sync(kFull, in);
                if (in)
                {
                    const int i = count + __popc(bal & ((1u << lane) - 1u));
                    Z(i, 1) = mul_((double) r, __ldg(&c_beam_cos[bm]));
                    Z(i, 2) = mul_((double) r, __ldg(&c_beam_sin[bm]));
                }
                count += __popc(bal);
            }
            if ((d.n_wrap >> 16) && lane == 0)
            {
                const float r = rs[kBeams - 1];
                Z(count, 1) = mul_((double) r, __ldg(&c_beam_cos[kBeams - 1]));
                Z(count, 2) = mul_((double) r, __ldg(&c_beam_sin[kBeams - 1]));
            }
        }
        __syncwarp();
        // classifyCluster (circle_fit_library.cpp:208-250)
        {
            const double p2x = Z(0, 1), p2y = Z(0, 2), p3x = Z(n - 1, 1), p3y = Z(n - 1, 2);
            for (int i = 1 + lane; i < n - 1; i += 32)
            {
                const double p1x = Z(i, 1), p1y = Z(i, 2);
                const double num = add_(add_(mul_(p2y, sub_(p1x, p3x)), mul_(p1y, sub_(p3x, p2x))), mul_(p3y, sub_(p2x, p1x)));
                const double den = add_(mul_(sub_(p2x, p1x), sub_(p1x, p3x)), mul_(sub_(p2y, p1y), sub_(p1y, p3y)));
                tmp[i] = mul_(div_(180.0, kPiRef), atan2(num, den));
            }
        }
        __syncwarp();
        // mean and population variance (:229-241): the quotients and squares by all lanes, the SUMS by lane 0 in the reference's order
        double * q1 = tmp + CAP;
        double sd = 0.0;
        {
            const int na = n - 2;
            for (int i = 1 + lane; i < n - 1; i += 32) q1[i] = div_(tmp[i], (double) na);
            __syncwarp();
            double mean = 0.0;
            if (lane == 0)
                for (int i = 1; i < n - 1; ++i) mean = add_(mean, q1[i]);
            mean = __shfl_sync(kFull, mean, 0);
            __syncwarp();
            for (int i = 1 + lane; i < n - 1; i += 32)
            {
                const double dv = sub_(tmp[i], mean);
                q1[i] = mul_(dv, dv);
            }
            __syncwarp();
            if (lane == 0)
            {
                for (int i = 1; i < n - 1; ++i) sd = add_(sd, q1[i]);
                sd = sqrt(div_(sd, (double) na));
            }
            sd = __shfl_sync(kFull, sd, 0);
            __syncwarp();
        }
        ClusterFit out;
        out.pub = 0.0;
        out.cx = out.cy = out.R = 0.0;
        if (sd < 10.0)   // warp-uniform
        {
            // circleFit (circle_fit_library.cpp:15-134): centroid and z_bar by lane 0 (sequential sums), Z by all lanes
            double x_hat = 0.0, y_hat = 0.0, z_bar = 0.0;
            double * q2 = tmp + 2 * CAP;
            for (int i = lane; i < n; i += 32)
            {
                q1[i] = div_(Z(i, 1), (double) n);
                q2[i] = div_(Z(i, 2), (double) n);
            }
            __syncwarp();
            {
                double acc = 0.0;
                if (lane < 2)
                {
                    const double * qq = lane == 0 ? q1 : q2;
#pragma unroll 4
                    for (int i = 0; i < n; ++i) acc = add_(acc, qq[i]);
                }
                x_hat = __shfl_sync(kFull, acc, 0);
                y_hat = __shfl_sync(kFull, acc, 1);
            }
            __syncwarp();
            for (int j = lane; j < n; j += 32)
            {
                const double dx = sub_(Z(j, 1), x_hat), dy = sub_(Z(j, 2), y_hat);
                Z(j, 0) = add_(mul_(dx, dx), mul_(dy, dy));
                Z(j, 1) = dx;
                Z(j, 2) = dy;
                Z(j, 3) = 1.0;
            }
            __syncwarp();
            for (int j = lane; j < n; j += 32) q1[j] = div_(Z(j, 0), (double) n);
            __syncwarp();
            if (lane == 0)
                for (int j = 0; j < n; ++j) z_bar = add_(z_bar, q1[j]);
            z_bar = __shfl_sync(kFull, z_bar, 0);
            __syncwarp();
            double sv[4], V[16], fit[3];
            svd_n4_warp(Zp, n, tmp, lane, sv, V);
            const int id = circle_fit_tail(sv, V, z_bar, x_hat, y_hat, fit);
            if ((id >= 0) && !(fit[2] > 1.0))
            {
                out.pub = 1.0;
                out.cx = fit[0];
                out.cy = fit[1];
                out.R = fit[2];
            }
        }
        if (lane == 0) pipe.fit[idx] = out;
        __syncwarp();
    }
}

// stage 3: one thread per scan of the chunk: published circles in detection order (landmarks.cpp:84-109)
__global__ void k_scan_publish(int64_t chunk, int32_t * __restrict__ n_clusters, int32_t * __restrict__ n_circles, double * __restrict__ circles,
                               int max_circles, ScanPipe pipe)
{
    const int64_t w = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= chunk) return;
    const int base = pipe.scan_base[w];
    if (base < 0) return;   // UB scans keep their marker, slow scans are written by the one-warp-per-scan kernel
    const int64_t s = pipe.scan0 + w;
    const int nk = n_clusters[s];
    double * cout = circles + s * (int64_t) max_circles * 4;
    int published = 0;
    for (int q = 0; q < nk; ++q)
    {
        const ClusterFit f = pipe.fit[base + q];
        if (f.pub != 0.0)
        {
            if (published < max_circles)
            {
                cout[4 * published + 0] = f.cx;
                cout[4 * published + 1] = f.cy;
                cout[4 * published + 2] = f.R;
                cout[4 * published + 3] = (double) q;
            }
            ++published;
        }
    }
    n_circles[s] = published;
}

constexpr int64_t kScanChunk = 262144;   // scans per pipeline pass (bounds the scratch: 262144 x 32 x 60 B = 0.5 GB of the 180 GB; fewer, longer launches: measured best of 64 K / 128 K / 256 K)

struct ScanScratch
{
    void * p = nullptr;
    size_t bytes = 0;
};

// side streams of the throughput path: the fits of the three size classes (and the slow-scan list) touch disjoint clusters, so the
// two long-tailed small launches run beside the big one instead of after it
struct ScanSide
{
    cudaStream_t s1 = nullptr, s2 = nullptr;
    cudaEvent_t fork = nullptr, join1 = nullptr, join2 = nullptr;
    cudaError_t ensure()
    {
        if (s1) return cudaSuccess;
        cudaError_t e = cudaStreamCreateWithFlags(&s1, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s2, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&fork, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&join1, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&join2, cudaEventDisableTiming);
        return e;
    }
};

inline cudaError_t launch_scan_detect(const float * ranges, int64_t n_scans, double min_range, double max_range, int16_t * cluster_of_beam,
                                      int32_t * n_clusters, int32_t * n_circles, double * circles, int32_t max_circles, int scan_ub,
                                      int device, int sm_count, cudaStream_t stream)
{
    cudaError_t e = scan_tables_init(device);
    if (e != cudaSuccess) return e;
    const size_t smem = sizeof(ScanSmem) * kScanWarps, smem_cluster = sizeof(ScanSmemHead) * kScanWarps;
    const size_t fit_smem16 = sizeof(double) * 4 * kFitSmall * kFitThreads, fit_smem32 = sizeof(double) * 4 * kFitNMax * kFitThreads;
    static bool configured_dev[kMaxDevices] = {false};
    bool & configured = configured_dev[(device >= 0 && device < kMaxDevices) ? device : 0];
    if (!configured)
    {
        e = cudaFuncSetAttribute(k_scan_detect<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_scan_fit_small<kFitNMax, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) fit_smem32);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    const int64_t resident_cluster = (int64_t) sm_count * 11;   // clustering only: 90 registers x 64 threads, 8.8 KB of shared memory per CTA
    ScanPipe none;
    memset(&none, 0, sizeof(none));
    if (n_scans <= 256)
    {
        // latency path: everything in one launch
        int64_t blocks = (n_scans + kScanWarps - 1) / kScanWarps;
        k_scan_detect<true><<<(unsigned) blocks, 32 * kScanWarps, smem, stream>>>(ranges, n_scans, min_range, max_range, cluster_of_beam, n_clusters,
                                                                               n_circles, circles, max_circles, scan_ub, nullptr, nullptr, none);
        return cudaGetLastError();
    }
    // throughput path: cluster (warp per scan) -> fit (thread per cluster) -> publish (thread per scan), in chunks of scans
    static thread_local ScanScratch scratch[64];
    static thread_local ScanSide sides[64];
    ScanScratch & sc = scratch[(device >= 0 && device < 64) ? device : 0];
    ScanSide & side = sides[(device >= 0 && device < 64) ? device : 0];
    e = side.ensure();
    if (e != cudaSuccess) return e;
    const int64_t chunk_max = n_scans < kScanChunk ? n_scans : kScanChunk;
    const size_t n_desc = (size_t) chunk_max * kMaxFastClusters;
    auto al = [](size_t v) { return (v + 255) & ~(size_t) 255; };
    const size_t need = al(n_desc * sizeof(ClusterDesc)) + al(n_desc * sizeof(ClusterFit)) + 3 * al(n_desc * sizeof(int32_t)) +
                        al((size_t) chunk_max * sizeof(int32_t)) * 2 + 256;
    if (sc.bytes < need)
    {
        if (sc.p) cudaFree(sc.p);
        sc.p = nullptr;
        sc.bytes = 0;
        e = cudaMalloc(&sc.p, need);
        if (e != cudaSuccess) return e;
        sc.bytes = need;
    }
    ScanPipe pipe;
    char * q = static_cast<char *>(sc.p);
    pipe.desc = reinterpret_cast<ClusterDesc *>(q);
    q += al(n_desc * sizeof(ClusterDesc));
    pipe.fit = reinterpret_cast<ClusterFit *>(q);
    q += al(n_desc * sizeof(ClusterFit));
    pipe.big = reinterpret_cast<int32_t *>(q);
    q += al(n_desc * sizeof(int32_t));
    pipe.big_s = reinterpret_cast<int32_t *>(q);
    q += al(n_desc * sizeof(int32_t));
    pipe.mid = reinterpret_cast<int32_t *>(q);
    q += al(n_desc * sizeof(int32_t));
    pipe.slow = reinterpret_cast<int32_t *>(q);
    q += al((size_t) chunk_max * sizeof(int32_t));
    pipe.scan_base = reinterpret_cast<int32_t *>(q);
    q += al((size_t) chunk_max * sizeof(int32_t));
    pipe.counters = reinterpret_cast<int32_t *>(q);
    for (int64_t s0 = 0; s0 < n_scans; s0 += kScanChunk)
    {
        const int64_t chunk = (n_scans - s0 < kScanChunk) ? n_scans - s0 : kScanChunk;
        pipe.scan0 = s0;
        e = cudaMemsetAsync(pipe.counters, 0, 8 * sizeof(int32_t), stream);
        if (e != cudaSuccess) return e;
        int64_t blocks = (chunk + kScanWarps - 1) / kScanWarps;
        if (blocks > resident_cluster) blocks = resident_cluster;
        k_scan_detect<false><<<(unsigned) blocks, 32 * kScanWarps, smem_cluster, stream>>>(ranges, chunk, min_range, max_range, cluster_of_beam, n_clusters,
                                                                                n_circles, circles, max_circles, scan_ub, nullptr, nullptr, pipe);
        e = cudaEventRecord(side.fork, stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(side.s1, side.fork, 0);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(side.s2, side.fork, 0);
        if (e != cudaSuccess) return e;
        k_scan_fit_small<kFitSmall, false><<<(unsigned) (sm_count * kFitCtas), kFitThreads, fit_smem16, stream>>>(ranges, min_range, max_range, pipe);
        k_scan_fit_small<kFitNMax, true><<<(unsigned) (sm_count * 3), kFitThreads, fit_smem32, side.s1>>>(ranges, min_range, max_range, pipe);
        k_scan_fit_big<kFitBigSmall + 2, 4, true><<<(unsigned) (sm_count * kBigSmallCtas), 128, 0, side.s2>>>(ranges, min_range, max_range, pipe);
        k_scan_fit_big<kBeams + 2, 2, false><<<(unsigned) (sm_count * 5), 64, 0, side.s2>>>(ranges, min_range, max_range, pipe);
        // scans with more than kMaxFastClusters clusters: the one-warp-per-scan kernel over their list (it writes those scans' outputs itself)
        k_scan_detect<true><<<(unsigned) sm_count, 32 * kScanWarps, smem, side.s2>>>(ranges, n_scans, min_range, max_range, cluster_of_beam, n_clusters,
                                                                                  n_circles, circles, max_circles, scan_ub, pipe.slow, pipe.counters + 2, pipe);
        e = cudaEventRecord(side.join1, side.s1);
        if (e == cudaSuccess) e = cudaEventRecord(side.join2, side.s2);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(stream, side.join1, 0);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(stream, side.join2, 0);
        if (e != cudaSuccess) return e;
        k_scan_publish<<<(unsigned) ((chunk + 127) / 128), 128, 0, stream>>>(chunk, n_clusters, n_circles, circles, max_circles, pipe);
        e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

}   // namespace nuslam
