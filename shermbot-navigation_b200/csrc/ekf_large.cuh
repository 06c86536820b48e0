// ekf_large.cuh -- LARGE-MAP mode: a few filters whose Sigma does not fit on chip (e.g. 4096 landmarks: len 8195, Sigma 537 MB).
//
// One scan with m measurements costs ONE read + ONE write of Sigma, whatever m is (BASELINE.json config 5):
//   predict   (slam_library.cpp:65-108): A = I + B touches rows/columns 1, 2 only                     -> O(len) kernel
//   updates   (slam_library.cpp:263-282) are DELAYED: with Sigma_i = Sigma_0 - sum_{u<i} K_u W_u  (K_u len x 2, W_u 2 x len),
//             update i needs only rows/columns {th, x, y, c, c+1} of Sigma_i, which are formed on the fly from Sigma_0 and
//             the stored K_u, W_u (O(len * i) per update): W_i = H Sigma_i, P_i = Sigma_i H^T, S = W_i H^T + R,
//             K_i = P_i S^-1, x += K_i dz                                                               -> 2 small kernels / update
//   one pass  Sigma <- Sigma_0 - [K_0 .. K_{m-1}] [W_0; ..; W_{m-1}]: a rank-2m update on the fp64 tensor pipe (DMMA m8n8k4,
//             accumulators initialised from Sigma, 32 x 32 tile per warp), HBM-bound: 16 len^2 bytes.
// The same kernels with m = 1 give the immediate (sequential) form used for the single `update` call and as the in-engine
// cross-check of the delayed form. Arithmetic: fp64 with FMAs; H and z_hat through the FAST kernel's short-chain helpers; parity
// <= 1e-9 after the first touch of a landmark (the first touch itself cancels catastrophically in the reference, SURVEY.md
// Appendix B).
// The NUSLAM_OPT_* variants are compile-time variants of the same kernels (template arguments; options == 0 instantiates the
// reference's kernels unchanged): PRE_MOTION_JACOBIAN in k_large_predict_pose, WRAP_INNOVATION in the update, the association and
// the oracle-order tail, JOSEPH as a symmetric factor form of the delayed updates (large_update) and a symmetric pass
// (k_large_rank_update_sym: Sigma <- Sigma_bar_0 - [K | A][A | K]^T, rank 4m).
#pragma once
#include "ekf_strict.cuh"
#include "fastmath.cuh"
#include <cooperative_groups.h>

namespace nuslam
{

constexpr int kLargeMMax = 16;   // measurements per delayed pass (rank 32)

struct LargeParams
{
    int64_t batch;
    int len, n;
    double * x;        // B x len (current)
    double * x2;       // B x len (ping-pong)
    double * sigma;    // B x len x len
    double * U;        // B x (2 kLargeMMax) x len : K_u columns, U[(2u+a) * len + j] = K_u(j, a)
    double * V;        // B x (2 kLargeMMax) x len : W_u rows,    V[(2u+a) * len + j] = W_u(a, j)
    double * P;        // B x 2 x len              : P_i = Sigma_i H^T of the update in flight
    int32_t * status;
    int32_t * strict_from;   // B or null: per filter, the first measurement slot of the pass in flight that the oracle-order tail takes
                             // (k_large_strict_tail: a landmark's first touch / initializeLandmark); >= the pass's count: none
    const int32_t * m_valid; // B or null: filter b uses only measurement slots i < m_valid[b] of the step (fused scan step; read by the
                             // unknown-correspondence kernels, the known-id path never receives one)
    int32_t * applied;       // B: per filter, non-zero once an update of the pass in flight went into U / V (read under JOSEPH only:
                             // the symmetric pass leaves a filter without one untouched)
    unsigned options;        // NUSLAM_OPT_* (0 = the reference's behaviour); the kernels take the bits as template arguments
    double Q[9], R[4];
};

// predict, part 1: pose and the two Jacobian entries (predictEstimate :71-94, getA :127-148 with theta AFTER the motion
// update; kPreMotion, NUSLAM_OPT_PRE_MOTION_JACOBIAN: theta BEFORE it, as WarpFilter::predict), one thread per filter; b10, b20 go to
// the head of the P scratch.
template <bool kPreMotion>
__global__ void k_large_predict_pose(const LargeParams p, const double * __restrict__ twists)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= p.batch) return;
    double * x = p.x + (int64_t) b * p.len;
    double * scratch = p.P + (int64_t) b * 2 * p.len;
    if (p.status[b] & (kStatusMapFull | kStatusSingular))
    {
        // the reference process died on an earlier scan: the filter stays as it was (zero Jacobian entries = identity covariance step)
        scratch[0] = 0.0;
        scratch[1] = 0.0;
        scratch[2] = 1.0;   // frozen marker: no process noise either
        return;
    }
    scratch[2] = 0.0;
    const double dth = twists[3 * b], dx = twists[3 * b + 1];
    const double theta = x[0];
    double s0, c0, th1, x1, y1, b10, b20;
    sincos(theta, &s0, &c0);
    if (dth == 0.0)
    {
        th1 = add_(theta, 0.0);
        x1 = add_(x[1], mul_(dx, c0));
        y1 = add_(x[2], mul_(dx, s0));
        b10 = mul_(-dx, s0);
        b20 = mul_(dx, c0);
    }
    else
    {
        const double q = div_(dx, dth);
        double s1, c1;
        th1 = add_(theta, dth);
        sincos(th1, &s1, &c1);
        x1 = add_(x[1], add_(mul_(-q, s0), mul_(q, s1)));
        y1 = add_(x[2], sub_(mul_(q, c0), mul_(q, c1)));
        if (kPreMotion)
        {
            // thJ = theta: cos(thJ), cos(thJ + dth) are c0, c1 (th1 = theta + dth, the same rounding as WarpFilter's add_(thJ, dth))
            b10 = add_(mul_(-q, c0), mul_(q, c1));
            b20 = add_(mul_(-q, s0), mul_(q, s1));
        }
        else
        {
            double s3, c3;
            sincos(add_(th1, dth), &s3, &c3);
            b10 = add_(mul_(-q, c1), mul_(q, c3));
            b20 = add_(mul_(-q, s1), mul_(q, s3));
        }
    }
    x[0] = th1;
    x[1] = x1;
    x[2] = y1;
    scratch[0] = b10;
    scratch[1] = b20;
}

// predict, part 2: Sigma <- A Sigma A^T + Q_bar in the oracle's operation order; only rows / columns 1, 2 change. Thread j >= 3
// owns entries (1, j), (2, j), (j, 1), (j, 2); thread 0 the 3 x 3 robot block (T = A Sigma, then U = T A^T, then + Q).
__global__ void k_large_predict_cov(const LargeParams p)
{
    const int b = blockIdx.y;
    const int len = p.len;
    double * S = p.sigma + (int64_t) b * len * len;
    const double * scratch = p.P + (int64_t) b * 2 * len;
    const double b10 = scratch[0], b20 = scratch[1];
    if (scratch[2] != 0.0) return;   // frozen filter (k_large_predict_pose): covariance untouched
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= 3 && j < len)
    {
        const double t0 = S[0 + (int64_t) j * len];
        S[1 + (int64_t) j * len] = add_(mul_(b10, t0), S[1 + (int64_t) j * len]);
        S[2 + (int64_t) j * len] = add_(mul_(b20, t0), S[2 + (int64_t) j * len]);
        const double u0 = S[j];
        S[j + (int64_t) len] = add_(mul_(u0, b10), S[j + (int64_t) len]);
        S[j + 2 * (int64_t) len] = add_(mul_(u0, b20), S[j + 2 * (int64_t) len]);
    }
    if (j == 0)
    {
        double B3[3][3];
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) B3[r][c] = S[r + (int64_t) c * len];
        for (int c = 0; c < 3; ++c)
        {
            B3[1][c] = add_(mul_(b10, B3[0][c]), B3[1][c]);
            B3[2][c] = add_(mul_(b20, B3[0][c]), B3[2][c]);
        }
        for (int r = 0; r < 3; ++r)
        {
            B3[r][1] = add_(mul_(B3[r][0], b10), B3[r][1]);
            B3[r][2] = add_(mul_(B3[r][0], b20), B3[r][2]);
        }
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) S[r + (int64_t) c * len] = add_(B3[r][c], p.Q[r + 3 * c]);
    }
}

inline cudaError_t launch_large_predict(const LargeParams & p, const double * twists, cudaStream_t st)
{
    if (p.options & kOptPreMotionJacobian) k_large_predict_pose<true><<<(unsigned) ((p.batch + 63) / 64), 64, 0, st>>>(p, twists);
    else k_large_predict_pose<false><<<(unsigned) ((p.batch + 63) / 64), 64, 0, st>>>(p, twists);
    k_large_predict_cov<<<dim3((p.len + 255) / 256, (unsigned) p.batch), 256, 0, st>>>(p);
    return cudaGetLastError();
}

// H entries and z_hat at state x for landmark slot c (reference expressions)
struct LargeModel
{
    double h[2][5];   // H(a, q) at q = {0, 1, 2, c, c+1}
    double zr, zb;
};
// the five state entries H depends on: (theta, x, y, mx, my). When the step protocol initialises the landmark for this very
// measurement (id above the scan's seen snapshot, slam.cpp:295-297), (mx, my) are what initializeLandmark (slam_library.cpp:255-261)
// would have written just before the update -- a pure function of the pose and z, so no separate pass over x is needed.
__device__ __forceinline__ bool large_local_state(const double * x, int c, int id, const double * z2, const int32_t * seen_snapshot, int b, double * xl)
{
    xl[0] = x[0];
    xl[1] = x[1];
    xl[2] = x[2];
    const bool init = seen_snapshot != nullptr && id > seen_snapshot[b];
    if (init)
    {
        double sn, cs;
        sincos(add_(z2[1], xl[0]), &sn, &cs);
        xl[3] = add_(xl[1], mul_(z2[0], cs));
        xl[4] = add_(xl[2], mul_(z2[0], sn));
    }
    else
    {
        xl[3] = x[c];
        xl[4] = x[c + 1];
    }
    return init;
}

// Every thread of the two update kernels needs H and z_hat; evaluated with the short-chain helpers of the FAST kernel
// (rsqrt / table atan2 / branch-free wrap, ~80 instructions, 1-2 ulp) instead of the libm chain of the reference's expressions
// (sincos + 3 atan2 + 8 divisions, ~800 instructions per thread, which dominated the update time of a large map).
__device__ __forceinline__ LargeModel large_model(const double * xl)
{
    LargeModel mdl;
    const double dx = xl[3] - xl[1], dy = xl[4] - xl[2];
    const double d = fma(dx, dx, dy * dy);
    const double rs = rsqrt_fast(d);
    double sq = d * rs;
    sq = fma(fma(-sq, sq, d), 0.5 * rs, sq);   // sqrt(d) to ~1 ulp
    const double id = rs * rs;                 // 1 / d
    mdl.h[0][0] = 0.0;
    mdl.h[0][1] = -dx * rs;
    mdl.h[0][2] = -dy * rs;
    mdl.h[0][3] = dx * rs;
    mdl.h[0][4] = dy * rs;
    mdl.h[1][0] = -1.0;
    mdl.h[1][1] = dy * id;
    mdl.h[1][2] = -dx * id;
    mdl.h[1][3] = -dy * id;
    mdl.h[1][4] = dx * id;
    mdl.zr = sq;
    mdl.zb = wrap_angle(atan2_fast(dy, dx) - xl[0]);   // normalize(normalize(atan2) - theta), slam_library.cpp:20,157
    return mdl;
}

// One delayed update (slot i of the pass), thread j owns state index j: W_i = H Sigma_i (row j of V), P_i = Sigma_i H^T, the 2 x 2
// innovation covariance, K_i = P_i S^-1 (row j of U) and x_new = x + K_i dz (slam_library.cpp:263-276) in ONE phase. Sigma_i is the
// current covariance, formed on the fly from Sigma_0 and the earlier updates of the pass (rows / columns {theta, x, y, c, c+1}
// only). The 2 x 2 part needs W_i at those five columns, i.e. the 5 x 5 sub-block of Sigma_i: every block forms it for itself
// (25 entries, same operation order as the owner threads use, so the values are bit-identical), which removes the grid-wide
// hand-over between "W, P" and "K, x" -- one grid barrier (or kernel boundary) per measurement instead of two.
// shared-memory copies the cooperative single-launch pass makes BEFORE its chain of dependent updates starts (known correspondence: the ids
// of the whole pass, hence every row / column of Sigma_0 it will read, are known up front): with them an update waits for one round trip
// to L2 (the earlier updates' K_u / W_u at its five indices, and the state) instead of three dependent ones
struct LargePre
{
    const double * rc;    // [(6 + 4 cnt)][blockDim.x]: this thread's Sigma_0 entries -- rows 0, 1, 2, columns 0, 1, 2, then per update rows c, c + 1, columns c, c + 1
    const double * blk;   // [cnt][25]: the 5 x 5 sub-block of Sigma_0 of every update
    const int * id;       // [cnt]
    const double * z;     // [cnt][2]
};

//
// JOSEPH (NUSLAM_OPT_JOSEPH): every update ends in the symmetric part of (I - K H) Sigma (I - K H)^T + K R K^T. With P = Sigma H^T,
// W = H Sigma, S = H Sigma H^T + R and the symmetric parts Sigma_bar, P_bar = (P + W^T) / 2, S_bar, that is, for any K,
//     Sigma_bar - K A^T - A K^T,   A = P_bar - K S_bar / 2,
// so the pass stays one low-rank update: V holds A_u instead of W_u (U keeps K_u) and every consumer forms
//     Sigma_i = Sigma_bar_0 - sum_{u<i} (K_u A_u^T + A_u K_u^T),
// symmetric by construction (row and column of an index are one value, P = W^T, P_bar = P); the pass is k_large_rank_update_sym.
// WRAP (NUSLAM_OPT_WRAP_INNOVATION): the bearing innovation is wrapped with normalize_angle, as in WarpFilter::update.
template <unsigned OPT>
__device__ __forceinline__ void large_update(const LargeParams & p, const double * __restrict__ z, const int32_t * __restrict__ ids, int m, int i,
                                             const double * __restrict__ x_old, double * __restrict__ x_new,
                                             const int32_t * __restrict__ seen_snapshot, int32_t * __restrict__ seen, double * own = nullptr,
                                             const LargePre * pre = nullptr)
{
    // own (cooperative single-launch pass only): this block's shared-memory copy of ITS threads' entries of the pass's K_u / W_u,
    // own[(2 r + {0: W, 1: K}) * blockDim.x + threadIdx.x] -- the correction loop then reads no global memory at all; the global U / V
    // rows are still written (the other blocks read five entries of them, the rank update all of them). JOSEPH: A_u in place of W_u.
    constexpr bool kJoseph = (OPT & kOptJoseph) != 0, kWrap = (OPT & kOptWrapInnovation) != 0;
    const int b = blockIdx.y;
    const int len = p.len;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int id = pre ? pre->id[i] : ids[b * m + i];
    const double z2[2] = {pre ? pre->z[2 * i] : z[(int64_t) (b * m + i) * 2], pre ? pre->z[2 * i + 1] : z[(int64_t) (b * m + i) * 2 + 1]};
    const double * x = x_old + (int64_t) b * len;
    double * xo = x_new + (int64_t) b * len;
    const double * S = p.sigma + (int64_t) b * len * len;
    double * U = p.U + (int64_t) b * 2 * kLargeMMax * len;
    double * V = p.V + (int64_t) b * 2 * kLargeMMax * len;
    const bool to_tail = p.strict_from != nullptr && i >= p.strict_from[b];   // this and every later measurement of the pass: oracle-order tail
    if (to_tail || id < 1 || id > p.n || (p.status[b] & (kStatusMapFull | kStatusSingular)))   // block-uniform
    {
        // (a filter the reference's process would have died on stays frozen, as in the STRICT and FAST kernels)
        // no measurement in this slot: K = 0, W = 0 contribute nothing to the pass (U, V of the slot were cleared at its start)
        if (j < len) xo[j] = x[j];
        if (own)
            for (int a = 0; a < 4; ++a) own[(4 * i + a) * blockDim.x + threadIdx.x] = 0.0;
        if (j == 0 && !to_tail && id > p.n && !(p.status[b] & (kStatusMapFull | kStatusSingular))) p.status[b] |= kStatusBadId;
        return;
    }
    const int c = 3 + 2 * (id - 1);
    const int idx[5] = {0, 1, 2, c, c + 1};
    // this thread's entries of the five rows / columns of Sigma_0 and its local state: issued first, so that their latency overlaps
    // the staging of the shared operands below (the strided row gather is the longest load of the update)
    double row[5], col[5];   // Sigma_i(idx[q], j) and Sigma_i(j, idx[q])
    if (pre)
    {
        const double * rc = pre->rc + threadIdx.x;
#pragma unroll
        for (int q = 0; q < 3; ++q)
        {
            row[q] = rc[q * blockDim.x];
            col[q] = rc[(3 + q) * blockDim.x];
        }
#pragma unroll
        for (int q = 0; q < 2; ++q)
        {
            row[3 + q] = rc[(6 + 4 * i + q) * blockDim.x];
            col[3 + q] = rc[(8 + 4 * i + q) * blockDim.x];
        }
    }
    else if (j < len)
    {
#pragma unroll
        for (int q = 0; q < 5; ++q)
        {
            row[q] = S[idx[q] + (int64_t) j * len];
            col[q] = S[j + (int64_t) idx[q] * len];
        }
    }
    if (kJoseph && (pre || j < len))
    {
        // Sigma_bar_0: row and column of each index are one value from here on (col is not read again)
#pragma unroll
        for (int q = 0; q < 5; ++q) row[q] = 0.5 * (row[q] + col[q]);
    }
    double xl[5];
    const bool init = large_local_state(x, c, id, z2, seen_snapshot, b, xl);
    const double x_own = (j < len) ? x[j] : 0.0;
    // K_u at the five rows and W_u at the five columns of every earlier update of the pass, and the 5 x 5 sub-block of Sigma_0
    __shared__ double ku[2 * kLargeMMax][5], wu[2 * kLargeMMax][5], blk[5][5];
    for (int k = threadIdx.x; k < 2 * i * 5; k += blockDim.x)
    {
        const int r = k / 5, q = k % 5;
        ku[r][q] = U[(int64_t) r * len + idx[q]];
        wu[r][q] = V[(int64_t) r * len + idx[q]];
    }
    if (threadIdx.x < 25)
    {
        const int r = threadIdx.x / 5, q = threadIdx.x % 5;
        blk[r][q] = pre ? pre->blk[25 * i + threadIdx.x] : S[idx[r] + (int64_t) idx[q] * len];
    }
    __syncthreads();
    if constexpr (!kJoseph)
    {
        if (threadIdx.x < 25)
        {
            // Sigma_i(idx[r], idx[q]): what the owner of column idx[q] computes as row[r] below, term for term
            const int r = threadIdx.x / 5, q = threadIdx.x % 5;
            double v = blk[r][q];
            for (int u = 0; u < 2 * i; ++u) v = fma(-ku[u][r], wu[u][q], v);
            blk[r][q] = v;
        }
    }
    else
    {
        // the same under JOSEPH: Sigma_bar_0 (read before any thread writes), then K_u A_u^T + A_u K_u^T (wu holds A_u)
        const int r = threadIdx.x / 5, q = threadIdx.x % 5;
        double v = 0.0;
        if (threadIdx.x < 25) v = 0.5 * (blk[r][q] + blk[q][r]);
        __syncthreads();
        if (threadIdx.x < 25)
        {
            for (int u = 0; u < 2 * i; ++u)
            {
                v = fma(-ku[u][r], wu[u][q], v);
                v = fma(-wu[u][r], ku[u][q], v);
            }
            blk[r][q] = v;
        }
    }
    __syncthreads();
    const LargeModel mdl = large_model(xl);
    // S = W_i[:, idx] H^T + R from the block's copy of the sub-block
    double s[2][2];
    {
        double w5[2][5];
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int q = 0; q < 5; ++q)
            {
                double w = 0.0;
#pragma unroll
                for (int r = 0; r < 5; ++r) w = fma(mdl.h[a][r], blk[r][q], w);
                w5[a][q] = w;
            }
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int e = 0; e < 2; ++e)
            {
                double acc = 0.0;
#pragma unroll
                for (int q = 0; q < 5; ++q) acc = fma(w5[a][q], mdl.h[e][q], acc);
                s[a][e] = acc + p.R[a + 2 * e];
            }
    }
    if (j >= len) return;
    const double xj = (init && j == c) ? xl[3] : (init && j == c + 1) ? xl[4] : x_own;   // x after initializeLandmark
    if (j == 0 && seen && id > seen[b]) seen[b] = id;                                      // what associateLandmark would have done to `seen`
    if constexpr (!kJoseph)
    {
#pragma unroll 4
        for (int r = 0; r < 2 * i; ++r)
        {
            const double wj = own ? own[(2 * r) * blockDim.x + threadIdx.x] : V[(int64_t) r * len + j];
            const double kj = own ? own[(2 * r + 1) * blockDim.x + threadIdx.x] : U[(int64_t) r * len + j];
#pragma unroll
            for (int q = 0; q < 5; ++q)
            {
                row[q] = fma(-ku[r][q], wj, row[q]);
                col[q] = fma(-kj, wu[r][q], col[q]);
            }
        }
    }
    else
    {
        // twice the shared-memory operands per update of the loop above: unrolled by 2 (by 4, ptxas spills k_large_update<JOSEPH>)
#pragma unroll 2
        for (int r = 0; r < 2 * i; ++r)
        {
            const double aj = own ? own[(2 * r) * blockDim.x + threadIdx.x] : V[(int64_t) r * len + j];   // A_r(j)
            const double kj = own ? own[(2 * r + 1) * blockDim.x + threadIdx.x] : U[(int64_t) r * len + j];
#pragma unroll
            for (int q = 0; q < 5; ++q)
            {
                row[q] = fma(-ku[r][q], aj, row[q]);
                row[q] = fma(-wu[r][q], kj, row[q]);
            }
        }
    }
    double pj[2];
#pragma unroll
    for (int a = 0; a < 2; ++a)
    {
        double w = 0.0, pp = 0.0;
#pragma unroll
        for (int q = 0; q < 5; ++q)
        {
            w = fma(mdl.h[a][q], row[q], w);
            if (!kJoseph) pp = fma(col[q], mdl.h[a][q], pp);
        }
        if constexpr (!kJoseph)
        {
            V[(int64_t) (2 * i + a) * len + j] = w;
            if (own) own[(2 * (2 * i + a)) * blockDim.x + threadIdx.x] = w;
            pj[a] = pp;
        }
        else pj[a] = w;   // P = W^T: the formed Sigma_i is symmetric
    }
    const double det = s[0][0] * s[1][1] - s[0][1] * s[1][0];
    if (det == 0.0)
    {
        U[(int64_t) (2 * i) * len + j] = 0.0;
        U[(int64_t) (2 * i + 1) * len + j] = 0.0;
        if (own) own[(2 * (2 * i) + 1) * blockDim.x + threadIdx.x] = own[(2 * (2 * i + 1) + 1) * blockDim.x + threadIdx.x] = 0.0;
        if constexpr (kJoseph)
        {
            // the pass reads both factors in both roles: both are zero
            V[(int64_t) (2 * i) * len + j] = 0.0;
            V[(int64_t) (2 * i + 1) * len + j] = 0.0;
            if (own) own[(2 * (2 * i)) * blockDim.x + threadIdx.x] = own[(2 * (2 * i + 1)) * blockDim.x + threadIdx.x] = 0.0;
        }
        xo[j] = xj;
        if (j == 0) p.status[b] |= kStatusSingular;
        return;
    }
    const double i00 = s[1][1] / det, i01 = -s[0][1] / det, i10 = -s[1][0] / det, i11 = s[0][0] / det;
    const double k0 = pj[0] * i00 + pj[1] * i10, k1 = pj[0] * i01 + pj[1] * i11;
    U[(int64_t) (2 * i) * len + j] = k0;
    U[(int64_t) (2 * i + 1) * len + j] = k1;
    if (own)
    {
        own[(2 * (2 * i) + 1) * blockDim.x + threadIdx.x] = k0;
        own[(2 * (2 * i + 1) + 1) * blockDim.x + threadIdx.x] = k1;
    }
    if constexpr (kJoseph)
    {
        // A(j, :) = P_bar(j, :) - K(j, :) S_bar / 2
        const double sb01 = 0.5 * (s[0][1] + s[1][0]);
        const double a0 = pj[0] - 0.5 * (k0 * s[0][0] + k1 * sb01);
        const double a1 = pj[1] - 0.5 * (k0 * sb01 + k1 * s[1][1]);
        V[(int64_t) (2 * i) * len + j] = a0;
        V[(int64_t) (2 * i + 1) * len + j] = a1;
        if (own)
        {
            own[(2 * (2 * i)) * blockDim.x + threadIdx.x] = a0;
            own[(2 * (2 * i + 1)) * blockDim.x + threadIdx.x] = a1;
        }
        if (j == 0) p.applied[b] = 1;
    }
    double dz1 = z2[1] - mdl.zb;   // :272, no wrap unless opted in
    if (kWrap) dz1 = normalize_angle(dz1);
    const double dz0 = z2[0] - mdl.zr;
    double xn = xj + (k0 * dz0 + k1 * dz1);
    if (j == 0) xn = wrap_angle(xn);   // normalize_angle, slam_library.cpp:276
    xo[j] = xn;
}

template <unsigned OPT>
__global__ void __launch_bounds__(256) k_large_update(const LargeParams p, const double * __restrict__ z, const int32_t * __restrict__ ids, int m, int i,
                                                      const double * __restrict__ x_old, double * __restrict__ x_new,
                                                      const int32_t * __restrict__ seen_snapshot, int32_t * __restrict__ seen)
{
    large_update<OPT>(p, z, ids, m, i, x_old, x_new, seen_snapshot, seen);
}

// ---- associateLandmark (slam_library.cpp:188-253) against the CURRENT covariance of a delayed pass ----
// One thread per candidate landmark k <= seen: the 5 x 5 sub-block of Sigma_i at {theta, x, y, c_k, c_k+1} from Sigma_0 and the
// pass's earlier updates, H and z_hat at the current state, the Mahalanobis distance with the unwrapped innovation. The reference's
// in-order early exit ("the first k whose distance decides") becomes an atomicMin over the keys (k << 2 | kind) of the deciding
// candidates. k_large_assoc_finalize then turns the winner into the id of slam.cpp:291 (and into `seen`, the status bits, the id
// slot the update kernel reads). kind: 0 = inv(psi) throws, 1 = match (d < 0.01), 2 = ambiguous (0.01 < d < 60).
// single_call: the single associateLandmark call (kOpAssociate) with i_pass = 0 -- it associates whatever the sticky status says.
// OPT: JOSEPH forms the sub-block as large_update does under it, WRAP wraps the bearing innovation (WarpFilter::mahalanobis).
// NEAREST_NEIGHBOUR: no key goes to `result`; each CTA reduces its candidates to one exact (d, k, singular) triple in nn[b][blockIdx.x]
// (no floating-point atomics: the winner does not depend on the order in which CTAs finish) and k_large_assoc_finalize scans them.
// A full map still evaluates its candidates there: a match succeeds, only a new landmark throws.
struct LargeNNSlot
{
    double d;       // smallest distance of the CTA's candidates
    int32_t k;      // its candidate (lowest k on ties); 0: none (every distance NaN)
    int32_t singular;
};

template <unsigned OPT>
__global__ void __launch_bounds__(128) k_large_associate(const LargeParams p, const double * __restrict__ z, int m, int i_meas, int i_pass,
                                                         const double * __restrict__ x_cur, const int32_t * __restrict__ seen,
                                                         int32_t * __restrict__ result, double amin, double amax, bool single_call,
                                                         LargeNNSlot * __restrict__ nn)
{
    constexpr bool kNN = (OPT & kOptNearestNeighbour) != 0;
    const int b = blockIdx.y;
    const int len = p.len;
    const int sn = seen[b];
    if (!single_call && (p.status[b] & (kStatusMapFull | kStatusSingular))) return;   // the reference process died on an earlier measurement
    if (p.m_valid && i_meas >= p.m_valid[b]) return;                 // past this filter's measurement count
    if (p.strict_from && p.strict_from[b] <= i_pass) return;         // this filter's measurements from i_pass on: oracle-order tail
    if (sn == 0 || (!kNN && 3 + 2 * sn >= len)) return;              // first landmark / full map: decided without any candidate
    if (kNN && (int) (blockIdx.x * blockDim.x) >= sn) return;         // a CTA without candidates writes no slot
    const double * S = p.sigma + (int64_t) b * len * len;
    const double * U = p.U + (int64_t) b * 2 * kLargeMMax * len;
    const double * V = p.V + (int64_t) b * 2 * kLargeMMax * len;
    const double * x = x_cur + (int64_t) b * len;
    // robot rows / columns of the earlier updates: shared by every candidate
    __shared__ double ku3[2 * kLargeMMax][3], wu3[2 * kLargeMMax][3];
    for (int t = threadIdx.x; t < 2 * i_pass * 3; t += blockDim.x)
    {
        ku3[t / 3][t % 3] = U[(int64_t) (t / 3) * len + t % 3];
        wu3[t / 3][t % 3] = V[(int64_t) (t / 3) * len + t % 3];
    }
    __syncthreads();
    const int k = blockIdx.x * blockDim.x + threadIdx.x + 1;
    if (!kNN && k > sn) return;
    const int c = 3 + 2 * ((kNN && k > sn ? sn : k) - 1);   // NN: every thread takes part in the CTA's reduction (past `seen`: a valid slot, no candidate)
    const int idx[5] = {0, 1, 2, c, c + 1};
    constexpr bool kJoseph = (OPT & kOptJoseph) != 0;
    double B5[5][5];
#pragma unroll
    for (int r = 0; r < 5; ++r)
#pragma unroll
        for (int q = 0; q < 5; ++q) B5[r][q] = S[idx[r] + (int64_t) idx[q] * len];
    if (kJoseph)
    {
#pragma unroll
        for (int r = 0; r < 5; ++r)
#pragma unroll
            for (int q = r + 1; q < 5; ++q) B5[r][q] = B5[q][r] = 0.5 * (B5[r][q] + B5[q][r]);   // Sigma_bar_0
    }
    for (int u = 0; u < 2 * i_pass; ++u)
    {
        const double kc = U[(int64_t) u * len + c], kc1 = U[(int64_t) u * len + c + 1];
        const double wc = V[(int64_t) u * len + c], wc1 = V[(int64_t) u * len + c + 1];
        const double kr[5] = {ku3[u][0], ku3[u][1], ku3[u][2], kc, kc1};
        const double wq[5] = {wu3[u][0], wu3[u][1], wu3[u][2], wc, wc1};   // JOSEPH: A_u
#pragma unroll
        for (int r = 0; r < 5; ++r)
#pragma unroll
            for (int q = 0; q < 5; ++q)
            {
                B5[r][q] = fma(-kr[r], wq[q], B5[r][q]);
                if (kJoseph) B5[r][q] = fma(-wq[r], kr[q], B5[r][q]);
            }
    }
    const double xl[5] = {x[0], x[1], x[2], x[c], x[c + 1]};
    const LargeModel mdl = large_model(xl);
    double w5[2][5];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int q = 0; q < 5; ++q)
        {
            double w = 0.0;
#pragma unroll
            for (int r = 0; r < 5; ++r) w = fma(mdl.h[a][r], B5[r][q], w);
            w5[a][q] = w;
        }
    double psi[2][2];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int e = 0; e < 2; ++e)
        {
            double acc = 0.0;
#pragma unroll
            for (int q = 0; q < 5; ++q) acc = fma(w5[a][q], mdl.h[e][q], acc);
            psi[a][e] = acc + p.R[a + 2 * e];
        }
    const double det = psi[0][0] * psi[1][1] - psi[0][1] * psi[1][0];
    const double z0 = z[(int64_t) (b * m + i_meas) * 2], z1 = z[(int64_t) (b * m + i_meas) * 2 + 1];
    int kind = -1;
    double dnn = 0.0;
    if (det == 0.0 || !(fabs(det) < 1.0e300) || !(fabs(1.0 / det) < 1.0e300)) kind = 0;
    else
    {
        const double i00 = psi[1][1] / det, i01 = -psi[0][1] / det, i10 = -psi[1][0] / det, i11 = psi[0][0] / det;
        const double dz0 = z0 - mdl.zr;
        double dz1 = z1 - mdl.zb;   // no angle wrap (:229-231) unless opted in
        if (OPT & kOptWrapInnovation) dz1 = normalize_angle(dz1);
        const double t0 = dz0 * i00 + dz1 * i10, t1 = dz0 * i01 + dz1 * i11;
        const double d = t0 * dz0 + t1 * dz1;
        if (kNN) dnn = d;
        else if (d < amin) kind = 1;
        else if (d > amin && d < amax) kind = 2;
    }
    if (kNN)
    {
        const bool active = k <= sn;
        double d = dnn;
        int kd = (active && kind != 0 && dnn == dnn) ? k : 0;
        nn_warp_min(d, kd);
        const bool sing = __ballot_sync(0xffffffffu, active && kind == 0) != 0u;
        __shared__ double wd[4];
        __shared__ int wk[4], ws[4];
        const int warp = threadIdx.x / kWarp;
        if (threadIdx.x % kWarp == 0)
        {
            wd[warp] = d;
            wk[warp] = kd;
            ws[warp] = sing;
        }
        __syncthreads();
        if (threadIdx.x == 0)
        {
            int s = ws[0];
            for (int w = 1; w < 4; ++w)
            {
                s |= ws[w];
                if (nn_better(wd[w], wk[w], d, kd))
                {
                    d = wd[w];
                    kd = wk[w];
                }
            }
            nn[(int64_t) b * gridDim.x + blockIdx.x] = LargeNNSlot{d, kd, s};
        }
        return;
    }
    if (kind >= 0) atomicMin(&result[b], (k << 2) | kind);
}

// slam.cpp:291 for every filter: the id associateLandmark returns, its side effect on `seen`, and the status bits where it throws.
// ids_slot: B x m scratch the update kernel reads (id <= 0: no update); ids_out: B x m or null.
// kNN (NUSLAM_OPT_NEAREST_NEIGHBOUR): one warp per filter; the winner is the (d, k) minimum over the ceil(seen / 128) CTA slots
// k_large_associate wrote (lane s reads slot s: one memory round trip instead of one per slot), and lane 0 decides.
template <bool kNN>
__global__ void k_large_assoc_finalize(const LargeParams p, int m, int i_meas, int i_pass, int32_t * __restrict__ seen, int32_t * __restrict__ result,
                                       int32_t * __restrict__ ids_slot, int32_t * __restrict__ ids_out, bool single_call,
                                       const LargeNNSlot * __restrict__ nn, double amin, double amax)
{
    const int b = kNN ? (int) blockIdx.x : (int) (blockIdx.x * blockDim.x + threadIdx.x);
    if (b >= p.batch) return;
    double dn = 0.0;
    int kn = 0;
    bool sing = false;
    if (kNN)
    {
        // (the slots are read whatever the checks below decide; only the branch that follows an associate launch uses them)
        const int slots = (p.n + 127) / 128, used = (seen[b] + 127) / 128;
        int sg = 0;
        for (int s = threadIdx.x; s < used; s += kWarp)   // ascending k within a lane: a later slot wins only with a smaller distance
        {
            const LargeNNSlot e = nn[(int64_t) b * slots + s];
            sg |= e.singular;
            if (nn_better(e.d, e.k, dn, kn))
            {
                dn = e.d;
                kn = e.k;
            }
        }
        nn_warp_min(dn, kn);
        sing = __any_sync(0xffffffffu, sg != 0);
        if (threadIdx.x != 0) return;
    }
    if (p.m_valid && i_meas >= p.m_valid[b])   // no measurement in this slot (k_large_associate left `result` untouched)
    {
        ids_slot[(int64_t) b * m + i_meas] = 0;
        if (ids_out) ids_out[(int64_t) b * m + i_meas] = 0;
        return;
    }
    if (p.strict_from && p.strict_from[b] <= i_pass)   // already handed to the oracle-order tail (it writes ids_out itself)
    {
        result[b] = 0x7fffffff;
        ids_slot[(int64_t) b * m + i_meas] = 0;
        return;
    }
    int id;
    bool tail = false;   // the measurement opens a landmark or touches one for the first time: only the oracle's operation order reproduces
                         // the reference there (SURVEY.md Appendix B), so this and the pass's later measurements go to k_large_strict_tail
    const int st = p.status[b];
    const int sn = seen[b];
    if (!single_call && (st & (kStatusMapFull | kStatusSingular))) id = 0;
    else if (sn == 0)
    {
        id = 1;   // :196-200
        tail = true;
    }
    else if (!kNN && 3 + 2 * sn >= p.len)
    {
        p.status[b] = st | kStatusMapFull;   // temp(3 + 2 seen) out of bounds: Armadillo throws (:204-207)
        id = kIdException;
    }
    else if (kNN)
    {
        if (sing)
        {
            p.status[b] = st | kStatusSingular;
            id = kIdException;
        }
        else if (kn != 0 && dn < amin) id = kn;
        else if (kn != 0 && dn < amax) id = -1;
        else if (3 + 2 * sn >= p.len)   // no slot left for the new landmark
        {
            p.status[b] = st | kStatusMapFull;
            id = kIdException;
        }
        else
        {
            id = sn + 1;
            tail = true;
        }
    }
    else
    {
        const int r = result[b];
        if (r >= 0x7f000000)   // untouched (any fill above the largest key (n << 2 | 3))
        {
            id = sn + 1;   // no candidate decided: a new landmark (:251)
            tail = true;
        }
        else if ((r & 3) == 0)
        {
            p.status[b] = st | kStatusSingular;
            id = kIdException;
        }
        else id = ((r & 3) == 1) ? (r >> 2) : -1;
    }
    if (!tail && id > 0 && p.strict_from)
    {
        const int c = 3 + 2 * (id - 1);
        const double * S = p.sigma + (int64_t) b * p.len * p.len;
        tail = S[c + (int64_t) c * p.len] > kFirstTouchVariance || S[c + 1 + (int64_t) (c + 1) * p.len] > kFirstTouchVariance;
    }
    result[b] = 0x7fffffff;
    if (tail && p.strict_from)
    {
        p.strict_from[b] = i_pass;   // `seen`, ids_out: the tail repeats this association in the oracle's order
        ids_slot[(int64_t) b * m + i_meas] = 0;
        return;
    }
    if (tail) seen[b] = id;   // (no tail scratch: the delayed path opens the landmark itself, as before)
    ids_slot[(int64_t) b * m + i_meas] = id;
    if (ids_out) ids_out[(int64_t) b * m + i_meas] = id;
}

// known correspondence: the first measurement slot of the pass [i0, i0 + cnt) that is a landmark's first touch (its variance still carries the
// INT_MAX prior) or, under the step protocol, an initializeLandmark (id above the scan's `seen` snapshot, slam.cpp:295-297). ids == null
// (unknown correspondence): none yet -- k_large_assoc_finalize finds it measurement by measurement.
__global__ void k_large_first_touch(const LargeParams p, const int32_t * __restrict__ ids, int m, int i0, int cnt, const int32_t * __restrict__ seen_snapshot)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= p.batch) return;
    int sf = cnt;
    if (ids && !(p.status[b] & (kStatusMapFull | kStatusSingular)))
    {
        const double * S = p.sigma + (int64_t) b * p.len * p.len;
        // the variances of every measured landmark are read first (independent loads: one DRAM latency for the pass instead of one
        // per measurement -- 17 us of the 400 us of an m = 12 scan at 4 096 landmarks), then the first hit decides
        double d0[kLargeMMax], d1[kLargeMMax];
#pragma unroll
        for (int i = 0; i < kLargeMMax; ++i)
        {
            const int id = (i < cnt) ? ids[(int64_t) b * m + i0 + i] : 0;
            const bool ok = id >= 1 && id <= p.n;
            const int c = ok ? 3 + 2 * (id - 1) : 0;
            d0[i] = ok ? S[c + (int64_t) c * p.len] : 0.0;
            d1[i] = ok ? S[c + 1 + (int64_t) (c + 1) * p.len] : 0.0;
        }
#pragma unroll
        for (int i = kLargeMMax - 1; i >= 0; --i)
        {
            const int id = (i < cnt) ? ids[(int64_t) b * m + i0 + i] : 0;
            if (id < 1 || id > p.n) continue;
            if ((seen_snapshot && id > seen_snapshot[b]) || d0[i] > kFirstTouchVariance || d1[i] > kFirstTouchVariance) sf = i;
        }
    }
    p.strict_from[b] = sf;
}

// The oracle-order tail of a pass: one warp per filter replays measurements [strict_from, cnt) of the pass with the STRICT arithmetic of
// ekf_strict.cuh (WarpFilter working directly on the filter's Sigma in HBM; its 14 len doubles of scratch are the pass's U rows, free
// once the rank update has run) -- associateLandmark / initializeLandmark / update exactly as EKFSlam::main_loop orders them
// (slam.cpp:279-319). It exists for parity (a first touch costs one warp a full sweep over Sigma: ~30 ms at 4096 landmarks), the
// steady state of a built map never takes it. OPT: the NUSLAM_OPT_* bits of the handle, as in the STRICT kernels.
template <unsigned OPT>
__global__ void __launch_bounds__(32) k_large_strict_tail(const LargeParams p, const double * __restrict__ z, const int32_t * __restrict__ ids, int m, int i0,
                                                          int cnt, double * __restrict__ x_cur, const int32_t * __restrict__ seen_snapshot,
                                                          int32_t * __restrict__ seen, double amin, double amax, int32_t * __restrict__ ids_out)
{
    const int b = blockIdx.x, lane = threadIdx.x;
    const int sf = p.strict_from[b];
    if (sf >= cnt) return;
    WarpFilter f;
    f.len = p.len;
    f.n = p.n;
    f.lane = lane;
    f.opt = OPT | (p.options & kOptNearestNeighbour);   // the pass's template bits do not carry the association rule
    f.S = p.sigma + (int64_t) b * p.len * p.len;
    f.x = x_cur + (int64_t) b * p.len;
    double * scratch = p.U + (int64_t) b * 2 * kLargeMMax * p.len;
    f.R5 = scratch;
    f.M5 = scratch + 5 * (int64_t) p.len;
    f.G = scratch + 10 * (int64_t) p.len;
    f.K = scratch + 12 * (int64_t) p.len;
    int status = p.status[b];
    int sn = seen ? seen[b] : p.n;
    const int snap = seen_snapshot ? seen_snapshot[b] : 0x7fffffff;   // no step protocol: never an initializeLandmark
    const int64_t mb = (int64_t) b * m + i0;
    const int end = p.m_valid ? min(cnt, p.m_valid[b] - i0) : cnt;   // this filter's measurements in the pass
    for (int i = sf; i < end; ++i)
    {
        if (status & (kStatusMapFull | kStatusSingular)) break;   // the reference process has died
        const double z0 = z[2 * (mb + i)], z1 = z[2 * (mb + i) + 1];
        int id;
        if (ids)
        {
            id = ids[mb + i];
            if (id <= 0) continue;
            if (id > p.n)
            {
                status |= kStatusBadId;
                continue;
            }
            if (id > sn) sn = id;
        }
        else
        {
            id = f.associate(z0, z1, sn, status, p.R, amin, amax);   // slam.cpp:291
            if (ids_out && lane == 0) ids_out[mb + i] = id;
            if (id == kIdException)
            {
                if (ids_out)
                    for (int r = i + 1 + lane; r < cnt; r += kWarp) ids_out[mb + r] = 0;
                break;
            }
        }
        if (id > snap) f.init_landmark(z0, z1, id, status);   // slam.cpp:295-297
        else if (id < 0) continue;                            // slam.cpp:298-300
        f.update(z0, z1, id, status, p.R);                    // slam.cpp:318
    }
    __syncwarp();
    if (lane == 0)
    {
        if (seen) seen[b] = sn;
        p.status[b] = status;
    }
}

// all `cnt` delayed updates of a pass in ONE cooperative launch: consecutive updates are separated by a grid barrier (~2 us) instead
// of a kernel boundary (~12 us of dependent-launch latency). x ping-pongs between p.x and p.x2.
template <unsigned OPT>
__global__ void __launch_bounds__(64) k_large_updates_coop(const LargeParams p, const double * __restrict__ z, const int32_t * __restrict__ ids, int m, int cnt,
                                                          const int32_t * __restrict__ seen_snapshot, int32_t * __restrict__ seen)
{
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    __shared__ double own[4 * kLargeMMax * 64];   // 32 KB: this block's entries of the pass's W_u / K_u (large_update)
    __shared__ int pre_id[kLargeMMax];
    __shared__ double pre_z[2 * kLargeMMax];
    extern __shared__ double large_dyn[];           // [(6 + 4 cnt) x 64] rows / columns of Sigma_0, then [cnt x 25] sub-blocks (LargePre)
    double * pre_rc = large_dyn;
    double * pre_blk = large_dyn + (6 + 4 * cnt) * 64;
    const double * xc = p.x;
    double * xn = p.x2;
    // known correspondence: every update of the pass reads five rows and five columns of Sigma_0 whose indices are known now -- they are
    // loaded into shared memory before the chain of dependent updates starts (the strided row gather from DRAM was its longest step;
    // round 2, session 3: loads instead of the L2 prefetches of session 2, which still left an L2 round trip per update in the chain)
    {
        const int b = blockIdx.y, len = p.len;
        const int j = blockIdx.x * blockDim.x + threadIdx.x;
        const int jj = j < len ? j : len - 1;   // the last block's spare threads load a valid entry they never use
        const double * S = p.sigma + (int64_t) b * len * len;
        if (threadIdx.x < cnt)
        {
            pre_id[threadIdx.x] = ids[b * m + threadIdx.x];
            pre_z[2 * threadIdx.x] = z[(int64_t) (b * m + threadIdx.x) * 2];
            pre_z[2 * threadIdx.x + 1] = z[(int64_t) (b * m + threadIdx.x) * 2 + 1];
        }
#pragma unroll
        for (int q = 0; q < 3; ++q)
        {
            pre_rc[q * 64 + threadIdx.x] = S[q + (int64_t) jj * len];
            pre_rc[(3 + q) * 64 + threadIdx.x] = S[jj + (int64_t) q * len];
        }
        for (int k = 0; k < cnt; ++k)
        {
            const int id = ids[b * m + k];
            if (id < 1 || id > p.n) continue;   // block-uniform; large_update returns before it reads the slot
            const int c = 3 + 2 * (id - 1);
            pre_rc[(6 + 4 * k) * 64 + threadIdx.x] = S[c + (int64_t) jj * len];
            pre_rc[(7 + 4 * k) * 64 + threadIdx.x] = S[c + 1 + (int64_t) jj * len];
            pre_rc[(8 + 4 * k) * 64 + threadIdx.x] = S[jj + (int64_t) c * len];
            pre_rc[(9 + 4 * k) * 64 + threadIdx.x] = S[jj + (int64_t) (c + 1) * len];
            if (threadIdx.x < 25)
            {
                const int idx[5] = {0, 1, 2, c, c + 1};
                const int r = threadIdx.x / 5, q = threadIdx.x % 5;
                pre_blk[25 * k + threadIdx.x] = S[idx[r] + (int64_t) idx[q] * len];
            }
        }
        __syncthreads();
    }
    const LargePre pre = {pre_rc, pre_blk, pre_id, pre_z};
    for (int k = 0; k < cnt; ++k)
    {
        large_update<OPT>(p, z, ids, m, k, xc, xn, seen_snapshot, seen, own, &pre);
        grid.sync();
        const double * t = xc;
        xc = xn;
        xn = const_cast<double *>(t);
    }
}

// empty the first `nslots` update slots of the pass (skipped / singular measurements and the rank padding contribute nothing)
__global__ void k_large_clear_w(const LargeParams p, int nslots)
{
    const int b = blockIdx.y;
    const int64_t e = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (int64_t) 2 * nslots * p.len) return;
    (p.V + (int64_t) b * 2 * kLargeMMax * p.len)[e] = 0.0;
    (p.U + (int64_t) b * 2 * kLargeMMax * p.len)[e] = 0.0;
}

__device__ __forceinline__ void dmma884_large(double & c0, double & c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// Sigma <- Sigma - K W with K = U^T (len x 2m), W = V (2m x len): CTA tile 64 x 64 (4 warps of 32 x 32), operands staged in
// shared memory, accumulators initialised from Sigma. kk = padded 2m (multiple of 4).
constexpr int kLargeTile = 64;
constexpr int kRankCtas = 4;   // resident CTAs per SM the register allocation aims at (3 at 148 registers: measured slower at rank >= 24)
__global__ void __launch_bounds__(128, kRankCtas) k_large_rank_update(const LargeParams p, int kk)
{
    __shared__ double su[2 * kLargeMMax][kLargeTile + 1];   // -K: su[k][r]
    __shared__ double sv[2 * kLargeMMax][kLargeTile + 1];   //  W: sv[k][c]
    const int b = blockIdx.z;
    const int len = p.len;
    const int r0 = blockIdx.x * kLargeTile, c0 = blockIdx.y * kLargeTile;
    double * S = p.sigma + (int64_t) b * len * len;
    const double * U = p.U + (int64_t) b * 2 * kLargeMMax * len;
    const double * V = p.V + (int64_t) b * 2 * kLargeMMax * len;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, t = lane & 3;
    const int wr = r0 + 32 * (warp >> 1), wc = c0 + 32 * (warp & 1);
    // the accumulators (this warp's 32 x 32 piece of Sigma: the DRAM stream of the pass) are requested FIRST, the operand staging below
    // (kk x 64 entries of K and W each, from L2) runs under their latency
    double C[4][4][2];
#pragma unroll
    for (int br = 0; br < 4; ++br)
#pragma unroll
        for (int bc = 0; bc < 4; ++bc)
#pragma unroll
            for (int e = 0; e < 2; ++e)
            {
                const int row = wr + 8 * br + g, col = wc + 8 * bc + 2 * t + e;
                C[br][bc][e] = (row < len && col < len) ? __ldcs(S + (int64_t) col * len + row) : 0.0;
            }
#pragma unroll 4
    for (int e = threadIdx.x; e < kk * kLargeTile; e += blockDim.x)
    {
        const int k = e / kLargeTile, o = e % kLargeTile;
        su[k][o] = (r0 + o < len) ? -U[(int64_t) k * len + r0 + o] : 0.0;
        sv[k][o] = (c0 + o < len) ? V[(int64_t) k * len + c0 + o] : 0.0;
    }
    __syncthreads();
    for (int k0 = 0; k0 < kk; k0 += 4)
    {
        double a[4], bb[4];
#pragma unroll
        for (int q = 0; q < 4; ++q)
        {
            a[q] = su[k0 + t][32 * (warp >> 1) + 8 * q + g];
            bb[q] = sv[k0 + t][32 * (warp & 1) + 8 * q + g];
        }
#pragma unroll
        for (int br = 0; br < 4; ++br)
#pragma unroll
            for (int bc = 0; bc < 4; ++bc) dmma884_large(C[br][bc][0], C[br][bc][1], a[br], bb[bc]);
    }
#pragma unroll
    for (int br = 0; br < 4; ++br)
#pragma unroll
        for (int bc = 0; bc < 4; ++bc)
#pragma unroll
            for (int e = 0; e < 2; ++e)
            {
                const int row = wr + 8 * br + g, col = wc + 8 * bc + 2 * t + e;
                if (row < len && col < len) __stcs(S + (int64_t) col * len + row, C[br][bc][e]);
            }
}

// The same pass as a persistent, software-pipelined kernel (round 2, session 3). k_large_rank_update above is a load -> compute -> store
// sequence per CTA whose accumulator registers are the only landing zone of the DRAM stream: at rank 24 its DMMA phase (0.8 us per tile)
// keeps a third of the resident warps from having loads in flight and the pass drops from 0.82 to 0.55 of the copy roof (290 us against
// 199 us at rank 4, measured). Here every CTA walks its tiles with the NEXT tile of Sigma on its way into shared memory while the
// current one is in the DMMAs (8-byte cp.async: Sigma's columns are only 8-byte aligned, len is odd; one 64 x 66 stage per CTA, the
// padding makes the fragment reads conflict-free per half-warp), so four resident CTAs keep 128 KB per SM in flight all the time; the
// operands come straight from L2 / L1 in fragment layout (K and W of the pass are 3 MB: no staging phase, no barrier in front of the
// DMMAs). Same DMMA order per accumulator: bit-identical results.
// (Two stages per CTA at three CTAs per SM -- 96 KB in flight -- were measured slower than the plain kernel: 0.28 ms at rank 4.)
constexpr int kRankStageLd = kLargeTile + 2;   // column stride of a stage in doubles (66: 2 x 66 = 4 mod 16, the four t of a half-warp hit disjoint banks)
constexpr int kRankStageDoubles = kLargeTile * kRankStageLd;
constexpr int kRankPipeCtas = 4;   // resident CTAs per SM (3 measured 0.7 % slower)
__global__ void __launch_bounds__(128, kRankPipeCtas) k_large_rank_update_pipe(const LargeParams p, int kk, int tiles)
{
    extern __shared__ __align__(16) double rank_stage[];   // [64 columns][66]
    const int len = p.len;
    const int64_t ntiles = (int64_t) tiles * tiles * p.batch;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, t = lane & 3;
    const int lr = 32 * (warp >> 1), lc = 32 * (warp & 1);
    // tile id -> (filter, column block, row block): consecutive ids walk down a column strip
    auto issue = [&](int64_t tile) {
        const int b = (int) (tile / ((int64_t) tiles * tiles));
        const int rem = (int) (tile % ((int64_t) tiles * tiles));
        const int c0 = (rem / tiles) * kLargeTile, r0 = (rem % tiles) * kLargeTile;
        const double * S = p.sigma + (int64_t) b * len * len;
        // thread -> one row of the tile (threadIdx.x & 63) and every second column: one pointer walking 2 len doubles per copy
        const int row = threadIdx.x & 63, col0 = threadIdx.x >> 6;
        const bool row_ok = r0 + row < len;
        const double * src = S + (int64_t) (c0 + col0) * len + r0 + row;
        const unsigned sa = (unsigned) __cvta_generic_to_shared(rank_stage + col0 * kRankStageLd + row);
        const int ncol = len - c0 - col0;   // columns c0 + col0 + 2 i with 2 i < ncol exist
#pragma unroll
        for (int i = 0; i < kLargeTile / 2; ++i)
        {
            const bool ok = row_ok && 2 * i < ncol;
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(sa + (unsigned) (2 * i * kRankStageLd * 8)), "l"(ok ? src : S), "r"(ok ? 8 : 0)
                         : "memory");   // out of range: zero fill
            src += 2 * (int64_t) len;
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // pull a tile's K / W operands (kk x 64 doubles each) towards L1 one round ahead of its DMMAs (measured: m = 32 scan 0.788 ms with
    // no prefetch, 0.775 prefetched at the top of the tile's own round, 0.768 one round ahead; m = 12 within 1 %)
    auto prefetch_ops = [&](int64_t tl) {
        const int b = (int) (tl / ((int64_t) tiles * tiles));
        const int rem = (int) (tl % ((int64_t) tiles * tiles));
        const int c0 = (rem / tiles) * kLargeTile, r0 = (rem % tiles) * kLargeTile;
        const double * U = p.U + (int64_t) b * 2 * kLargeMMax * len;
        const double * V = p.V + (int64_t) b * 2 * kLargeMMax * len;
        // row k of K / W at the tile's 64 rows / columns: 512 bytes = up to five 128-byte lines each
        for (int e = threadIdx.x; e < kk * 10; e += 128)
        {
            const int k = e / 10, w = e % 10;
            const double * base = (w < 5 ? U + r0 : V + c0) + (int64_t) k * len;
            const int o = 16 * (w % 5);
            if ((w < 5 ? r0 : c0) + o < len) asm volatile("prefetch.global.L1 [%0];" ::"l"(base + o));
        }
    };
    int64_t tile = blockIdx.x;
    if (tile < ntiles) issue(tile);
    for (; tile < ntiles; tile += gridDim.x)
    {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        double C[4][4][2];
#pragma unroll
        for (int br = 0; br < 4; ++br)
#pragma unroll
            for (int bc = 0; bc < 4; ++bc)
#pragma unroll
                for (int e = 0; e < 2; ++e) C[br][bc][e] = rank_stage[(lc + 8 * bc + 2 * t + e) * kRankStageLd + lr + 8 * br + g];
        __syncthreads();   // the stage is free: the next tile starts its way in while this one is in the DMMAs
        if (tile + gridDim.x < ntiles)
        {
            issue(tile + gridDim.x);
            prefetch_ops(tile + gridDim.x);
        }
        const int b = (int) (tile / ((int64_t) tiles * tiles));
        const int rem = (int) (tile % ((int64_t) tiles * tiles));
        const int c0 = (rem / tiles) * kLargeTile, r0 = (rem % tiles) * kLargeTile;
        double * S = p.sigma + (int64_t) b * len * len;
        const double * U = p.U + (int64_t) b * 2 * kLargeMMax * len;
        const double * V = p.V + (int64_t) b * 2 * kLargeMMax * len;
        // operands in fragment layout straight from L2 / L1: a = -K(row, k0 + t), b = W(k0 + t, column); rows / columns beyond len: 0.
        // One k-step's operands are requested at a time: two or three together measured slower (m = 12 scan 0.408 / 0.419 ms against 0.348)
        for (int k0 = 0; k0 < kk; k0 += 4)
        {
            const double * Uk = U + (int64_t) (k0 + t) * len + r0 + lr + g;
            const double * Vk = V + (int64_t) (k0 + t) * len + c0 + lc + g;
            double a[4], bb[4];
#pragma unroll
            for (int q = 0; q < 4; ++q)
            {
                a[q] = (r0 + lr + 8 * q + g < len) ? -__ldg(Uk + 8 * q) : 0.0;
                bb[q] = (c0 + lc + 8 * q + g < len) ? __ldg(Vk + 8 * q) : 0.0;
            }
#pragma unroll
            for (int br = 0; br < 4; ++br)
#pragma unroll
                for (int bc = 0; bc < 4; ++bc) dmma884_large(C[br][bc][0], C[br][bc][1], a[br], bb[bc]);
        }
#pragma unroll
        for (int br = 0; br < 4; ++br)
#pragma unroll
            for (int bc = 0; bc < 4; ++bc)
#pragma unroll
                for (int e = 0; e < 2; ++e)
                {
                    const int row = r0 + lr + 8 * br + g, col = c0 + lc + 8 * bc + 2 * t + e;
                    if (row < len && col < len) __stcs(S + (int64_t) col * len + row, C[br][bc][e]);
                }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

inline cudaError_t launch_large_rank_update(const LargeParams & p, int kk, cudaStream_t st)
{
    const unsigned tiles = (p.len + kLargeTile - 1) / kLargeTile;
    // the plain kernel below rank 16, the pipelined one from there up. Measured at 4 096 landmarks (tools/gpu_round2_ag.sh): rank 4: plain
    // 0.20 ms, pipelined 0.23 ms; rank 24: 0.30 / 0.27 ms; rank 32: 0.37 / 0.33 ms
    constexpr int kPipeMinRank = 16;
    if (kk < kPipeMinRank)
    {
        k_large_rank_update<<<dim3(tiles, tiles, (unsigned) p.batch), 128, 0, st>>>(p, kk);
        return cudaGetLastError();
    }
    static int sms_dev[kMaxDevices] = {0};
    int & sms = sms_dev[device_slot()];
    constexpr int kSmem = kRankStageDoubles * (int) sizeof(double);
    if (sms == 0)
    {
        int dev = 0, n = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        const cudaError_t e = cudaFuncSetAttribute(k_large_rank_update_pipe, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
        if (e != cudaSuccess) return e;
        sms = n > 0 ? n : 1;
    }
    int64_t blocks = (int64_t) tiles * tiles * p.batch;
    if (blocks > kRankPipeCtas * (int64_t) sms) blocks = kRankPipeCtas * (int64_t) sms;
    k_large_rank_update_pipe<<<(unsigned) blocks, 128, kSmem, st>>>(p, kk, (int) tiles);
    return cudaGetLastError();
}

// The JOSEPH pass: Sigma <- Sigma_bar_0 - [K | A] [A | K]^T (rank 2 kk: U holds K_u, V holds A_u, large_update), exactly symmetric.
// The DMMA sums of (r, c) and (c, r) would run in different orders, so one CTA owns a tile PAIR (I <= J): it stages the partner tile
// (J, I) in shared memory, starts the accumulators of tile (I, J) at (T_IJ + T_JI^T) / 2, runs the DMMAs on (I, J) only and stores
// the tile and its transpose (a diagonal tile: its lower triangle, mirrored). Same bytes read and written as the plain pass, the
// DMMAs of a rank-kk pass over all tiles. The operands come in fragment layout straight from L2 / L1 (as in the pipelined kernel),
// so the rank is not bounded by a shared-memory staging area: kk up to 2 kLargeMMax, rank 4 kLargeMMax.
// A filter with no update of the pass in its factors (frozen, or every slot handed to the oracle-order tail) is not touched at all:
// its Sigma leaves the pass bit for bit as it came in, symmetric or not.
constexpr int kSymLd = kLargeTile + 1;
__global__ void __launch_bounds__(128, 4) k_large_rank_update_sym(const LargeParams p, int kk)
{
    __shared__ double tr[kLargeTile][kSymLd];   // tr[rr][cc] = Sigma(c0 + cc, r0 + rr): tile (J, I) transposed, then the result for it
    const int b = blockIdx.y;
    if (!p.applied[b]) return;
    const int len = p.len;
    // pair index -> (I, J), I <= J: pair = J (J + 1) / 2 + I
    const int pair = (int) blockIdx.x;
    int J = (int) ((sqrt(8.0 * pair + 1.0) - 1.0) * 0.5);
    while ((J + 1) * (J + 2) / 2 <= pair) ++J;
    while (J * (J + 1) / 2 > pair) --J;
    const int I = pair - J * (J + 1) / 2;
    const bool diag = I == J;
    const int r0 = I * kLargeTile, c0 = J * kLargeTile;
    double * S = p.sigma + (int64_t) b * len * len;
    const double * U = p.U + (int64_t) b * 2 * kLargeMMax * len;
    const double * V = p.V + (int64_t) b * 2 * kLargeMMax * len;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, t = lane & 3;
    const int lr = 32 * (warp >> 1), lc = 32 * (warp & 1);
    double C[4][4][2];
#pragma unroll
    for (int br = 0; br < 4; ++br)
#pragma unroll
        for (int bc = 0; bc < 4; ++bc)
#pragma unroll
            for (int e = 0; e < 2; ++e)
            {
                const int row = r0 + lr + 8 * br + g, col = c0 + lc + 8 * bc + 2 * t + e;
                C[br][bc][e] = (row < len && col < len) ? __ldcs(S + (int64_t) col * len + row) : 0.0;
            }
#pragma unroll 4
    for (int e = threadIdx.x; e < kLargeTile * kLargeTile; e += blockDim.x)
    {
        const int cc = e % kLargeTile, rr = e / kLargeTile;   // column r0 + rr of Sigma, rows c0 + cc: contiguous in cc
        tr[rr][cc] = (c0 + cc < len && r0 + rr < len) ? __ldcs(S + (int64_t) (r0 + rr) * len + c0 + cc) : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int br = 0; br < 4; ++br)
#pragma unroll
        for (int bc = 0; bc < 4; ++bc)
#pragma unroll
            for (int e = 0; e < 2; ++e) C[br][bc][e] = 0.5 * (C[br][bc][e] + tr[lr + 8 * br + g][lc + 8 * bc + 2 * t + e]);
    __syncthreads();   // tr is reused for the transposed store
    // a = -[K | A](row, k), b = [A | K](k, column); kk is a multiple of 4, so a k-step lies in one half
    for (int k0 = 0; k0 < 2 * kk; k0 += 4)
    {
        const bool second = k0 >= kk;
        const int k = (second ? k0 - kk : k0) + t;
        const double * Ak = (second ? V : U) + (int64_t) k * len + r0 + lr + g;
        const double * Bk = (second ? U : V) + (int64_t) k * len + c0 + lc + g;
        double a[4], bb[4];
#pragma unroll
        for (int q = 0; q < 4; ++q)
        {
            a[q] = (r0 + lr + 8 * q + g < len) ? -__ldg(Ak + 8 * q) : 0.0;
            bb[q] = (c0 + lc + 8 * q + g < len) ? __ldg(Bk + 8 * q) : 0.0;
        }
#pragma unroll
        for (int br = 0; br < 4; ++br)
#pragma unroll
            for (int bc = 0; bc < 4; ++bc) dmma884_large(C[br][bc][0], C[br][bc][1], a[br], bb[bc]);
    }
#pragma unroll
    for (int br = 0; br < 4; ++br)
#pragma unroll
        for (int bc = 0; bc < 4; ++bc)
#pragma unroll
            for (int e = 0; e < 2; ++e)
            {
                const int rl = lr + 8 * br + g, cl = lc + 8 * bc + 2 * t + e;
                if (r0 + rl < len && c0 + cl < len && (!diag || rl >= cl)) __stcs(S + (int64_t) (c0 + cl) * len + r0 + rl, C[br][bc][e]);
                tr[rl][cl] = C[br][bc][e];
            }
    __syncthreads();
#pragma unroll 4
    for (int e = threadIdx.x; e < kLargeTile * kLargeTile; e += blockDim.x)
    {
        const int cc = e % kLargeTile, rr = e / kLargeTile;   // Sigma(c0 + cc, r0 + rr) = C(rr, cc)
        if (c0 + cc < len && r0 + rr < len && (!diag || rr > cc)) __stcs(S + (int64_t) (r0 + rr) * len + c0 + cc, tr[rr][cc]);
    }
}

inline cudaError_t launch_large_rank_update_sym(const LargeParams & p, int kk, cudaStream_t st)
{
    const unsigned tiles = (p.len + kLargeTile - 1) / kLargeTile;
    k_large_rank_update_sym<<<dim3(tiles * (tiles + 1) / 2, (unsigned) p.batch), 128, 0, st>>>(p, kk);
    return cudaGetLastError();
}

// initializeLandmark (slam_library.cpp:255-261) for measurement i of the step when its id exceeds the scan's seen snapshot
// (slam.cpp:295-297), or unconditionally (snapshot == nullptr: the single initializeLandmark call); one thread per filter.
__global__ void k_large_init_landmark(const LargeParams p, const double * __restrict__ z, const int32_t * __restrict__ ids, int m, int i,
                                      const int32_t * __restrict__ seen_snapshot, int32_t * __restrict__ seen)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= p.batch) return;
    const int id = ids[b * m + i];
    if (id < 1) return;
    if (id > p.n)
    {
        p.status[b] |= kStatusBadId;
        return;
    }
    if (seen_snapshot)
    {
        if (id > seen[b]) seen[b] = id;   // what associateLandmark would have done to `seen`
        if (id <= seen_snapshot[b]) return;
    }
    double * x = p.x + (int64_t) b * p.len;
    const int c = 3 + 2 * (id - 1);
    const double z0 = z[(int64_t) (b * m + i) * 2], z1 = z[(int64_t) (b * m + i) * 2 + 1];
    double sn, cs;
    sincos(add_(z1, x[0]), &sn, &cs);
    x[c] = add_(x[1], mul_(z0, cs));
    x[c + 1] = add_(x[2], mul_(z0, sn));
}

// host: one delayed pass over measurements [i0, i0 + cnt) of the step (cnt <= kLargeMMax); x ping-pongs between p.x and p.x2
// association of a pass: unknown correspondence (ids written measurement by measurement into ids_slot by the association kernels)
struct LargeAssoc
{
    int32_t * ids_slot = nullptr;   // B x m
    int32_t * result = nullptr;     // B, initialised to INT_MAX
    int32_t * ids_out = nullptr;    // B x m or null
    LargeNNSlot * nn = nullptr;     // B x ceil(n / 128) (NUSLAM_OPT_NEAREST_NEIGHBOUR only)
    double amin = 0.01, amax = 60.0;
};

// k_large_associate for measurement i_meas of the step (slot i_pass of the pass), one thread per candidate landmark, then
// k_large_assoc_finalize. OPT: the pass's bits (kLargePassOpts); the association rule comes from p.options.
template <unsigned OPT>
inline void launch_large_associate_t(const LargeParams & p, const double * z, int m, int i_meas, int i_pass, const double * x_cur, int32_t * seen,
                                     int32_t * ids_slot, int32_t * ids_out, const LargeAssoc & a, bool single_call, cudaStream_t st)
{
    const dim3 grid((unsigned) ((p.n + 127) / 128), (unsigned) p.batch);
    if (p.options & kOptNearestNeighbour)
    {
        k_large_associate<OPT | kOptNearestNeighbour><<<grid, 128, 0, st>>>(p, z, m, i_meas, i_pass, x_cur, seen, a.result, a.amin, a.amax, single_call,
                                                                          a.nn);
        k_large_assoc_finalize<true><<<(unsigned) p.batch, kWarp, 0, st>>>(p, m, i_meas, i_pass, seen, a.result, ids_slot, ids_out, single_call, a.nn,
                                                                            a.amin, a.amax);
    }
    else
    {
        k_large_associate<OPT><<<grid, 128, 0, st>>>(p, z, m, i_meas, i_pass, x_cur, seen, a.result, a.amin, a.amax, single_call, nullptr);
        k_large_assoc_finalize<false><<<(unsigned) ((p.batch + 63) / 64), 64, 0, st>>>(p, m, i_meas, i_pass, seen, a.result, ids_slot, ids_out,
                                                                                        single_call, nullptr, a.amin, a.amax);
    }
}

// the option bits the pass kernels take as template arguments (PRE_MOTION_JACOBIAN is predict's alone, NEAREST_NEIGHBOUR the
// association's: launch_large_associate_t and k_large_strict_tail read it from p.options)
constexpr unsigned kLargePassOpts = kOptWrapInnovation | kOptJoseph;

// the single associateLandmark call: i_pass = 0, no tail
inline void launch_large_associate(const LargeParams & p, const double * z, int32_t * seen, int32_t * ids_slot, int32_t * id_out, const LargeAssoc & a,
                                   cudaStream_t st)
{
    switch (p.options & kLargePassOpts)
    {
    case 0u: launch_large_associate_t<0u>(p, z, 1, 0, 0, p.x, seen, ids_slot, id_out, a, true, st); break;
    case kOptWrapInnovation: launch_large_associate_t<kOptWrapInnovation>(p, z, 1, 0, 0, p.x, seen, ids_slot, id_out, a, true, st); break;
    case kOptJoseph: launch_large_associate_t<kOptJoseph>(p, z, 1, 0, 0, p.x, seen, ids_slot, id_out, a, true, st); break;
    default: launch_large_associate_t<kLargePassOpts>(p, z, 1, 0, 0, p.x, seen, ids_slot, id_out, a, true, st); break;
    }
}

// OPT: the handle's option bits within kLargePassOpts (every static below is per instantiation: each kernel variant has its own occupancy)
template <unsigned OPT>
inline cudaError_t launch_large_updates_t(LargeParams & p, const double * z, const int32_t * ids, int m, int i0, int cnt,
                                          const int32_t * seen_snapshot, int32_t * seen, cudaStream_t st, const LargeAssoc * assoc)
{
    constexpr bool kJoseph = (OPT & kOptJoseph) != 0;
    const int threads = 64;   // ~130 small blocks at len 8195: every SM takes part in the latency-bound row / column gathers
    const dim3 grid((p.len + threads - 1) / threads, (unsigned) p.batch);
    const int kk = (2 * cnt + 3) & ~3;
    k_large_clear_w<<<dim3((unsigned) (((int64_t) kk * p.len + threads - 1) / threads), (unsigned) p.batch), threads, 0, st>>>(p, kk / 2);
    if (kJoseph)
    {
        const cudaError_t ce = cudaMemsetAsync(p.applied, 0, sizeof(int32_t) * p.batch, st);
        if (ce != cudaSuccess) return ce;
    }
    if (p.strict_from) k_large_first_touch<<<(unsigned) ((p.batch + 63) / 64), 64, 0, st>>>(p, ids, m, i0, cnt, seen_snapshot);
    // after the pass: measurements the delayed path left to the oracle-order tail (first touches; usually none)
    auto tail = [&]() {
        if (p.strict_from)
            k_large_strict_tail<OPT><<<(unsigned) p.batch, 32, 0, st>>>(p, z, ids, m, i0, cnt, p.x, seen_snapshot, seen, assoc ? assoc->amin : 0.0,
                                                                     assoc ? assoc->amax : 0.0, assoc ? assoc->ids_out : nullptr);
    };
    if (assoc)
    {
        // unknown correspondence: per measurement associate (one thread per candidate) -> finalize -> update
        for (int k = 0; k < cnt; ++k)
        {
            launch_large_associate_t<OPT>(p, z, m, i0 + k, k, p.x, seen, assoc->ids_slot, assoc->ids_out, *assoc, false, st);
            k_large_update<OPT><<<grid, threads, 0, st>>>(p, z + 2 * (int64_t) i0, assoc->ids_slot + i0, m, k, p.x, p.x2, seen_snapshot, seen);
            double * tmp = p.x;
            p.x = p.x2;
            p.x2 = tmp;
        }
        const cudaError_t re = kJoseph ? launch_large_rank_update_sym(p, kk, st) : launch_large_rank_update(p, kk, st);
        if (re != cudaSuccess) return re;
        tail();
        return cudaGetLastError();
    }
    // one cooperative launch when the whole grid is co-resident (it is for a few large maps), else two launches per update
    static int coop_dev[kMaxDevices];
    static bool coop_known[kMaxDevices] = {false};
    const int slot = device_slot();
    if (!coop_known[slot]) coop_dev[slot] = -1;
    coop_known[slot] = true;
    int & coop_blocks_per_sm = coop_dev[slot];
    if (coop_blocks_per_sm < 0)
    {
        int dev = 0, sms = 0, nb = 0, can = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&can, cudaDevAttrCooperativeLaunch, dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        const size_t dyn_max = ((size_t) (6 + 4 * kLargeMMax) * 64 + 25 * kLargeMMax) * sizeof(double);
        if (cudaFuncSetAttribute(k_large_updates_coop<OPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) dyn_max) != cudaSuccess) can = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_large_updates_coop<OPT>, threads, dyn_max);
        coop_blocks_per_sm = can ? nb * sms : 0;
    }
    if ((int64_t) grid.x * grid.y <= coop_blocks_per_sm)
    {
        const double * zz = z + 2 * (int64_t) i0;
        const int32_t * ii = ids + i0;
        void * args[] = {(void *) &p, (void *) &zz, (void *) &ii, (void *) &m, (void *) &cnt, (void *) &seen_snapshot, (void *) &seen};
        const size_t dyn = ((size_t) (6 + 4 * cnt) * 64 + 25 * cnt) * sizeof(double);   // LargePre
        cudaError_t ce = cudaLaunchCooperativeKernel((const void *) k_large_updates_coop<OPT>, grid, dim3(threads), args, dyn, st);
        if (ce != cudaSuccess) return ce;
        if (cnt & 1)
        {
            double * tmp = p.x;
            p.x = p.x2;
            p.x2 = tmp;
        }
    }
    else
    for (int k = 0; k < cnt; ++k)
    {
        // slot k of the pass holds measurement i0 + k: the kernels index ids / z with (b * m + k) from the shifted base pointers
        k_large_update<OPT><<<grid, threads, 0, st>>>(p, z + 2 * (int64_t) i0, ids + i0, m, k, p.x, p.x2, seen_snapshot, seen);
        double * tmp = p.x;
        p.x = p.x2;
        p.x2 = tmp;
    }
    const cudaError_t re = kJoseph ? launch_large_rank_update_sym(p, kk, st) : launch_large_rank_update(p, kk, st);
    if (re != cudaSuccess) return re;
    tail();
    return cudaGetLastError();
}

inline cudaError_t launch_large_updates(LargeParams & p, const double * z, const int32_t * ids, int m, int i0, int cnt,
                                        const int32_t * seen_snapshot, int32_t * seen, cudaStream_t st, const LargeAssoc * assoc = nullptr)
{
    switch (p.options & kLargePassOpts)
    {
    case 0u: return launch_large_updates_t<0u>(p, z, ids, m, i0, cnt, seen_snapshot, seen, st, assoc);
    case kOptWrapInnovation: return launch_large_updates_t<kOptWrapInnovation>(p, z, ids, m, i0, cnt, seen_snapshot, seen, st, assoc);
    case kOptJoseph: return launch_large_updates_t<kOptJoseph>(p, z, ids, m, i0, cnt, seen_snapshot, seen, st, assoc);
    default: return launch_large_updates_t<kLargePassOpts>(p, z, ids, m, i0, cnt, seen_snapshot, seen, st, assoc);
    }
}

}   // namespace nuslam
