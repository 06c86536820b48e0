// ekf_strict.cuh -- STRICT arithmetic: one warp per filter, Sigma resident in shared memory.
//
// Reproduces, term by term, the operation order of the reference's dense Armadillo expressions
// (ascending k, one rounded multiply then one rounded add per term, chained products left to right;
// see oracle/shim/armadillo for the order the oracle defines) while visiting only the structurally
// non-zero terms:
//   predict : A = I + B has B(1,0), B(2,0) only (slam_library.cpp:133-146), so A*Sigma*A.t() + Q_bar
//             (:104) touches rows 1,2 then columns 1,2 then the 3x3 block            -> O(len)
//   update  : H_j has non-zeros in columns {0,1,2,c,c+1} (:175-183), so (I - K*H) has non-zeros on the
//             diagonal and in those 5 columns; (I-KH)*Sigma (:279) is 5 or 6 terms per element -> O(len^2)
// Skipped terms are exact zeros in the oracle (0 * finite), so every finite result is bit-identical
// up to the sign of zero.
#pragma once
#include "ekf_common.cuh"

namespace nuslam
{

// shared-memory footprint of one warp's filter, in doubles
__host__ __device__ constexpr int strict_smem_doubles(int len) { return len * len + 17 * len + 8; }

struct WarpFilter
{
    int len, n, lane;
    unsigned opt = 0u;   // NUSLAM_OPT_* (0 = the reference's behaviour)
    double * S;    // len x len, column-major
    double * x;    // len
    double * R5;   // 5 x len: rows {0,1,2,c,c+1} of Sigma before the update, R5[k*len + j]
    double * M5;   // 5 x len: columns {0,1,2,c,c+1} of (I - K*H), M5[k*len + i]
    double * G;    // 2 x len: H*Sigma, G[a*len + j]
    double * K;    // 2 x len (debug / future use)

    __device__ __forceinline__ void carve(double * base, int len_, int n_, int lane_)
    {
        len = len_;
        n = n_;
        lane = lane_;
        S = base;
        x = S + len * len;
        R5 = x + len;
        M5 = R5 + 5 * len;
        G = M5 + 5 * len;
        K = G + 2 * len;
    }

    __device__ __forceinline__ void load(const double * gx, const double * gS)
    {
        for (int e = lane; e < len * len; e += kWarp) S[e] = gS[e];
        for (int e = lane; e < len; e += kWarp) x[e] = gx[e];
        __syncwarp();
    }

    __device__ __forceinline__ void store(double * gx, double * gS, bool sigma)
    {
        __syncwarp();
        if (sigma)
            for (int e = lane; e < len * len; e += kWarp) gS[e] = S[e];
        for (int e = lane; e < len; e += kWarp) gx[e] = x[e];
    }

    // ExtendedKalman::predict, slam_library.cpp:65-69
    __device__ void predict(double dth, double dx, const double * Q)
    {
        // predictEstimate :71-94 (every lane evaluates the same scalars)
        const double theta = x[0];
        double dq_th, dq_x, dq_y;
        if (dth == 0.0)
        {
            dq_th = 0.0;
            dq_x = mul_(dx, cos(theta));
            dq_y = mul_(dx, sin(theta));
        }
        else
        {
            const double q = div_(dx, dth);
            dq_th = dth;
            dq_x = add_(mul_(-q, sin(theta)), mul_(q, sin(add_(theta, dth))));
            dq_y = sub_(mul_(q, cos(theta)), mul_(q, cos(add_(theta, dth))));
        }
        const double th1 = add_(theta, dq_th);
        const double x1 = add_(x[1], dq_x);
        const double y1 = add_(x[2], dq_y);
        __syncwarp();
        if (lane == 0)
        {
            x[0] = th1;
            x[1] = x1;
            x[2] = y1;
        }
        // getA :127-148 -- theta read AFTER predictEstimate (:129); the opt-in variant linearises where the motion started
        const double thJ = (opt & kOptPreMotionJacobian) ? theta : th1;
        double b10, b20;
        if (dth == 0.0)
        {
            b10 = mul_(-dx, sin(thJ));
            b20 = mul_(dx, cos(thJ));
        }
        else
        {
            const double q = div_(dx, dth);
            b10 = add_(mul_(-q, cos(thJ)), mul_(q, cos(add_(thJ, dth))));
            b20 = add_(mul_(-q, sin(thJ)), mul_(q, sin(add_(thJ, dth))));
        }
        // T = A * Sigma: rows 1 and 2 (k = 0 term first, then the unit diagonal term)
        for (int j = lane; j < len; j += kWarp)
        {
            const double s0 = S[0 + j * len];
            S[1 + j * len] = add_(mul_(b10, s0), S[1 + j * len]);
            S[2 + j * len] = add_(mul_(b20, s0), S[2 + j * len]);
        }
        __syncwarp();
        // U = T * A.t(): columns 1 and 2
        for (int i = lane; i < len; i += kWarp)
        {
            const double t0 = S[i + 0 * len];
            S[i + 1 * len] = add_(mul_(t0, b10), S[i + 1 * len]);
            S[i + 2 * len] = add_(mul_(t0, b20), S[i + 2 * len]);
        }
        __syncwarp();
        // + Q_bar (expanded_process_noise :110-125): only the robot block is non-zero
        if (lane < 9)
        {
            const int r = lane % 3, cc = lane / 3;
            S[r + cc * len] = add_(S[r + cc * len], Q[r + 3 * cc]);
        }
        __syncwarp();
    }

    // ExtendedKalman::initializeLandmark, slam_library.cpp:255-261
    __device__ void init_landmark(double z0, double z1, int id, int & status)
    {
        if (id < 1 || id > n)
        {
            status |= kStatusBadId;
            return;
        }
        const int c = 3 + 2 * (id - 1);
        const double a = add_(z1, x[0]);
        const double mx = add_(x[1], mul_(z0, cos(a)));
        const double my = add_(x[2], mul_(z0, sin(a)));
        __syncwarp();
        if (lane == 0)
        {
            x[c] = mx;
            x[c + 1] = my;
        }
        __syncwarp();
    }

    // Mahalanobis distance of z to landmark k at the current state: slam_library.cpp:212-232
    __device__ double mahalanobis(double z0, double z1, int k, const double * R, bool & singular)
    {
        const int c = 3 + 2 * (k - 1);
        HEntries H;
        double zr, zb;
        measurement_model(x, c, H, zr, zb);
        const int cols[5] = {0, 1, 2, c, c + 1};
        double g0[5], g1[5];   // (H*Sigma) at the 5 columns where H is non-zero
#pragma unroll
        for (int q = 0; q < 5; ++q)
        {
            const int j = cols[q];
            const double s0 = S[0 + j * len], s1 = S[1 + j * len], s2 = S[2 + j * len];
            const double sc = S[c + j * len], sc1 = S[c + 1 + j * len];
            double a0 = mul_(H.h01, s1);
            a0 = add_(a0, mul_(H.h02, s2));
            a0 = add_(a0, mul_(H.h0c, sc));
            a0 = add_(a0, mul_(H.h0c1, sc1));
            double a1 = -s0;
            a1 = add_(a1, mul_(H.h11, s1));
            a1 = add_(a1, mul_(H.h12, s2));
            a1 = add_(a1, mul_(H.h1c, sc));
            a1 = add_(a1, mul_(H.h1c1, sc1));
            g0[q] = a0;
            g1[q] = a1;
        }
        // psi = (H*Sigma)*H.t() + R
        double p00 = mul_(g0[1], H.h01);
        p00 = add_(p00, mul_(g0[2], H.h02));
        p00 = add_(p00, mul_(g0[3], H.h0c));
        p00 = add_(p00, mul_(g0[4], H.h0c1));
        double p10 = mul_(g1[1], H.h01);
        p10 = add_(p10, mul_(g1[2], H.h02));
        p10 = add_(p10, mul_(g1[3], H.h0c));
        p10 = add_(p10, mul_(g1[4], H.h0c1));
        double p01 = -g0[0];
        p01 = add_(p01, mul_(g0[1], H.h11));
        p01 = add_(p01, mul_(g0[2], H.h12));
        p01 = add_(p01, mul_(g0[3], H.h1c));
        p01 = add_(p01, mul_(g0[4], H.h1c1));
        double p11 = -g1[0];
        p11 = add_(p11, mul_(g1[1], H.h11));
        p11 = add_(p11, mul_(g1[2], H.h12));
        p11 = add_(p11, mul_(g1[3], H.h1c));
        p11 = add_(p11, mul_(g1[4], H.h1c1));
        p00 = add_(p00, R[0]);
        p10 = add_(p10, R[1]);
        p01 = add_(p01, R[2]);
        p11 = add_(p11, R[3]);
        double i00, i01, i10, i11;
        if (!inv2x2(p00, p01, p10, p11, i00, i01, i10, i11))
        {
            singular = true;
            return 0.0;
        }
        double dz1 = sub_(z1, zb);   // no angle wrap (:229-231) unless opted in
        if (opt & kOptWrapInnovation) dz1 = normalize_angle(dz1);
        const double dz0 = sub_(z0, zr);
        // (dz.t() * psi.i()) * dz
        const double t0 = add_(mul_(dz0, i00), mul_(dz1, i10));
        const double t1 = add_(mul_(dz0, i01), mul_(dz1, i11));
        return add_(mul_(t0, dz0), mul_(t1, dz1));
    }

    // ExtendedKalman::associateLandmark, slam_library.cpp:188-253. One candidate landmark per lane; the
    // reference's in-order early exit becomes "lowest lane whose distance decides".
    __device__ int associate(double z0, double z1, int & seen, int & status, const double * R, double amin, double amax)
    {
        if (seen == 0)
        {
            seen = 1;
            return 1;
        }
        if (opt & kOptNearestNeighbour) return associate_nn(z0, z1, seen, status, R, amin, amax);
        if (3 + 2 * seen >= len)   // temp(3+2*seen) out of bounds: Armadillo throws (:206)
        {
            status |= kStatusMapFull;
            return kIdException;
        }
        for (int base = 0; base < seen; base += kWarp)
        {
            const int k = base + lane + 1;
            const bool active = k <= seen;
            bool singular = false;
            double d = 0.0;
            if (active) d = mahalanobis(z0, z1, k, R, singular);
            const unsigned sing = __ballot_sync(0xffffffffu, active && singular);
            const unsigned hitA = __ballot_sync(0xffffffffu, active && !singular && (d < amin));
            const unsigned hitB = __ballot_sync(0xffffffffu, active && !singular && (d > amin) && (d < amax));
            const unsigned any = hitA | hitB | sing;
            if (any)
            {
                const int first = __ffs(any) - 1;
                if ((sing >> first) & 1u)
                {
                    status |= kStatusSingular;
                    return kIdException;
                }
                if ((hitA >> first) & 1u) return base + first + 1;
                return -1;
            }
        }
        seen += 1;
        return seen;
    }

    // NUSLAM_OPT_NEAREST_NEIGHBOUR (seen >= 1): every candidate k = 1..seen is evaluated; a singular psi anywhere throws, as the
    // reference's inv would once it reached that candidate. The smallest distance (lowest k on ties; a NaN distance is no candidate)
    // is a match below amin, ambiguous below amax, and otherwise the measurement opens a landmark -- which throws on a full map,
    // where a match still succeeds. Each lane keeps its running minimum over the chunks of 32, then one warp-wide (d, k) reduction.
    __device__ int associate_nn(double z0, double z1, int & seen, int & status, const double * R, double amin, double amax)
    {
        double best = 0.0;
        int kbest = 0;
        for (int base = 0; base < seen; base += kWarp)
        {
            const int k = base + lane + 1;
            bool singular = false;
            double d = 0.0;
            if (k <= seen) d = mahalanobis(z0, z1, k, R, singular);
            if (__ballot_sync(0xffffffffu, singular))
            {
                status |= kStatusSingular;
                return kIdException;
            }
            if (k <= seen && d == d && nn_better(d, k, best, kbest))
            {
                best = d;
                kbest = k;
            }
        }
        nn_warp_min(best, kbest);
        if (kbest != 0 && best < amin) return kbest;
        if (kbest != 0 && best < amax) return -1;
        if (3 + 2 * seen >= len)   // no slot left for the new landmark
        {
            status |= kStatusMapFull;
            return kIdException;
        }
        seen += 1;
        return seen;
    }

    // ExtendedKalman::update, slam_library.cpp:263-282
    __device__ void update(double z0, double z1, int id, int & status, const double * R)
    {
        if (id < 1 || id > n)
        {
            status |= kStatusBadId;
            return;
        }
        const int c = 3 + 2 * (id - 1);
        HEntries H;
        double zr, zb;
        measurement_model(x, c, H, zr, zb);
        // G = H * Sigma (2 x len); keep the 5 rows of Sigma the update reads
        for (int j = lane; j < len; j += kWarp)
        {
            const double s0 = S[0 + j * len], s1 = S[1 + j * len], s2 = S[2 + j * len];
            const double sc = S[c + j * len], sc1 = S[c + 1 + j * len];
            R5[0 * len + j] = s0;
            R5[1 * len + j] = s1;
            R5[2 * len + j] = s2;
            R5[3 * len + j] = sc;
            R5[4 * len + j] = sc1;
            double a0 = mul_(H.h01, s1);
            a0 = add_(a0, mul_(H.h02, s2));
            a0 = add_(a0, mul_(H.h0c, sc));
            a0 = add_(a0, mul_(H.h0c1, sc1));
            double a1 = -s0;
            a1 = add_(a1, mul_(H.h11, s1));
            a1 = add_(a1, mul_(H.h12, s2));
            a1 = add_(a1, mul_(H.h1c, sc));
            a1 = add_(a1, mul_(H.h1c1, sc1));
            G[0 * len + j] = a0;
            G[1 * len + j] = a1;
        }
        __syncwarp();
        // psi = G * H.t() + R, inverse
        double p00 = mul_(G[1], H.h01);
        p00 = add_(p00, mul_(G[2], H.h02));
        p00 = add_(p00, mul_(G[c], H.h0c));
        p00 = add_(p00, mul_(G[c + 1], H.h0c1));
        double p10 = mul_(G[len + 1], H.h01);
        p10 = add_(p10, mul_(G[len + 2], H.h02));
        p10 = add_(p10, mul_(G[len + c], H.h0c));
        p10 = add_(p10, mul_(G[len + c + 1], H.h0c1));
        double p01 = -G[0];
        p01 = add_(p01, mul_(G[1], H.h11));
        p01 = add_(p01, mul_(G[2], H.h12));
        p01 = add_(p01, mul_(G[c], H.h1c));
        p01 = add_(p01, mul_(G[c + 1], H.h1c1));
        double p11 = -G[len + 0];
        p11 = add_(p11, mul_(G[len + 1], H.h11));
        p11 = add_(p11, mul_(G[len + 2], H.h12));
        p11 = add_(p11, mul_(G[len + c], H.h1c));
        p11 = add_(p11, mul_(G[len + c + 1], H.h1c1));
        p00 = add_(p00, R[0]);
        p10 = add_(p10, R[1]);
        p01 = add_(p01, R[2]);
        p11 = add_(p11, R[3]);
        double i00, i01, i10, i11;
        if (!inv2x2(p00, p01, p10, p11, i00, i01, i10, i11))
        {
            status |= kStatusSingular;   // arma::inv throws; the update never happens
            __syncwarp();
            return;
        }
        double dz1 = sub_(z1, zb);   // :272, no wrap unless opted in
        if (opt & kOptWrapInnovation) dz1 = normalize_angle(dz1);
        const double dz0 = sub_(z0, zr);
        // P = Sigma * H.t(); K = P * inv(psi); x += K * dz; columns of M = I - K*H
        for (int i = lane; i < len; i += kWarp)
        {
            const double s0 = S[i + 0 * len], s1 = S[i + 1 * len], s2 = S[i + 2 * len];
            const double sc = S[i + c * len], sc1 = S[i + (c + 1) * len];
            double pa = mul_(s1, H.h01);
            pa = add_(pa, mul_(s2, H.h02));
            pa = add_(pa, mul_(sc, H.h0c));
            pa = add_(pa, mul_(sc1, H.h0c1));
            double pb = -s0;
            pb = add_(pb, mul_(s1, H.h11));
            pb = add_(pb, mul_(s2, H.h12));
            pb = add_(pb, mul_(sc, H.h1c));
            pb = add_(pb, mul_(sc1, H.h1c1));
            const double k0 = add_(mul_(pa, i00), mul_(pb, i10));
            const double k1 = add_(mul_(pa, i01), mul_(pb, i11));
            x[i] = add_(x[i], add_(mul_(k0, dz0), mul_(k1, dz1)));   // :275
            if (opt & kOptJoseph)
            {
                K[0 * len + i] = k0;
                K[1 * len + i] = k1;
            }
            // (K*H)(i,j) = K(i,0)*H(0,j) + K(i,1)*H(1,j);  M = eye - K*H
            const double kh0 = -k1;   // K(i,0)*0 + K(i,1)*(-1)
            const double kh1 = add_(mul_(k0, H.h01), mul_(k1, H.h11));
            const double kh2 = add_(mul_(k0, H.h02), mul_(k1, H.h12));
            const double khc = add_(mul_(k0, H.h0c), mul_(k1, H.h1c));
            const double khc1 = add_(mul_(k0, H.h0c1), mul_(k1, H.h1c1));
            M5[0 * len + i] = sub_((i == 0) ? 1.0 : 0.0, kh0);
            M5[1 * len + i] = sub_((i == 1) ? 1.0 : 0.0, kh1);
            M5[2 * len + i] = sub_((i == 2) ? 1.0 : 0.0, kh2);
            M5[3 * len + i] = sub_((i == c) ? 1.0 : 0.0, khc);
            M5[4 * len + i] = sub_((i == c + 1) ? 1.0 : 0.0, khc1);
        }
        __syncwarp();
        if (lane == 0) x[0] = normalize_angle(x[0]);   // :276
        // Sigma = M * Sigma (:279): ascending-k merge of {0,1,2,c,c+1} with the unit diagonal term k = i. Every element is an
        // independent expression, so the traversal is free: lane = row i (its five M entries stay in registers), loop over the
        // columns j (the five R5 entries of a column are one broadcast read each) -- a third of the shared-memory traffic of a
        // flat element loop, the same arithmetic per element.
        const int len2 = len * len;
        for (int i0 = 0; i0 < len; i0 += kWarp)
        {
            const int i = i0 + lane;
            if (i < len)
            {
                const double m0 = M5[0 * len + i], m1 = M5[1 * len + i], m2 = M5[2 * len + i], m3 = M5[3 * len + i], m4 = M5[4 * len + i];
                const bool mid = i >= 3 && i < c, hi = i > c + 1;
                for (int j = 0; j < len; ++j)
                {
                    const int e = i + j * len;
                    double acc = mul_(m0, R5[0 * len + j]);
                    acc = add_(acc, mul_(m1, R5[1 * len + j]));
                    acc = add_(acc, mul_(m2, R5[2 * len + j]));
                    if (mid) acc = add_(acc, S[e]);
                    acc = add_(acc, mul_(m3, R5[3 * len + j]));
                    acc = add_(acc, mul_(m4, R5[4 * len + j]));
                    if (hi) acc = add_(acc, S[e]);
                    S[e] = acc;
                }
            }
        }
        __syncwarp();
        if (opt & kOptJoseph)
        {
            // Joseph form on top of T = (I - K H) Sigma (now in S): Sigma' = T (I - K H)^T + K R K^T = T - (T H^T) K^T + K R K^T,
            // then the symmetric part. T H^T (len x 2) goes to the first two rows of R5 (dead after the pass above).
            for (int i = lane; i < len; i += kWarp)
            {
                const double t0 = S[i + 0 * len], t1 = S[i + 1 * len], t2 = S[i + 2 * len];
                const double tc = S[i + c * len], tc1 = S[i + (c + 1) * len];
                R5[0 * len + i] = fma(t1, H.h01, fma(t2, H.h02, fma(tc, H.h0c, tc1 * H.h0c1)));
                R5[1 * len + i] = fma(t1, H.h11, fma(t2, H.h12, fma(tc, H.h1c, fma(tc1, H.h1c1, -t0))));
            }
            __syncwarp();
            for (int e = lane; e < len2; e += kWarp)
            {
                const int j = e / len;
                const int i = e - j * len;
                const double k0j = K[0 * len + j], k1j = K[1 * len + j];
                const double rk0 = fma(R[0], k0j, R[2] * k1j), rk1 = fma(R[1], k0j, R[3] * k1j);   // (R K^T)(:, j), R column-major
                double acc = S[e];
                acc = fma(-R5[0 * len + i], k0j, acc);
                acc = fma(-R5[1 * len + i], k1j, acc);
                acc = fma(K[0 * len + i], rk0, acc);
                acc = fma(K[1 * len + i], rk1, acc);
                S[e] = acc;
            }
            __syncwarp();
            for (int e = lane; e < len2; e += kWarp)
            {
                const int j = e / len;
                const int i = e - j * len;
                if (i < j)
                {
                    const double a = 0.5 * (S[i + j * len] + S[j + i * len]);
                    S[i + j * len] = a;
                    S[j + i * len] = a;
                }
            }
            __syncwarp();
        }
    }
};

// NUSLAM_OPT_JOINT_COMPATIBILITY (joint compatibility branch and bound, Neira & Tardos 2001): measurements per step, and joint tests
// per filter per step before the search stops with the best hypothesis found so far (NUSLAM_FILTER_ASSOC_TRUNCATED)
constexpr int kJcbbMMax = 16;
constexpr int kJcbbMaxTests = 4096;
constexpr int kJcbbRows = 2 * kJcbbMMax;

// JCBB scratch of one warp, behind its WarpFilter slice (JOINT handles only), in doubles
__host__ __device__ constexpr int jcbb_smem_doubles(int n)
{
    return kJcbbMMax * n + 10 * n + kJcbbRows * (kJcbbRows + 1) / 2 + kJcbbRows + 4 * kJcbbMMax + (kJcbbMMax + 1)
         + (kJcbbMMax * n + 6 * kJcbbMMax + 2 * (kJcbbMMax + 1) + 1) / 2;
}

struct JcbbScratch
{
    double * dist;   // m x n: d_ik, the individual distance of measurement i to candidate k (dist[i * n + k - 1])
    double * hc;     // n x 10: H entries (h01 h02 h0c h0c1 h11 h12 h1c h1c1), z_hat (range, bearing) of every candidate
    double * L;      // packed lower Cholesky factor of the hypothesis' joint S, row r at r (r + 1) / 2
    double * y;      // L^-1 nu, the whitened stacked innovation
    double * bx;     // per test: 2 x 2 cross blocks H_new Sigma H_j^T of the pairings j < p, then H_new Sigma H_new^T + R at j = p
    double * d2;     // per depth: D^2 of the hypothesis on entry
    int * cand;      // m x n: the compatible candidates of measurement i in ascending (d_ik, k)
    int * ncand;     // m
    int * jid;       // m: the ids the step applies
    int * hyp;       // per depth: the landmark measurement i is paired with (0: none)
    int * best;      // m: the best hypothesis
    int * pk;        // per pairing: its landmark
    int * it;        // per depth: next position in cand (ncand: the null pairing, ncand + 1: exhausted)
    int * pcnt;      // per depth: pairings on entry

    __device__ __forceinline__ void carve(double * base, int n)
    {
        dist = base;
        hc = dist + kJcbbMMax * n;
        L = hc + 10 * n;
        y = L + kJcbbRows * (kJcbbRows + 1) / 2;
        bx = y + kJcbbRows;
        d2 = bx + 4 * kJcbbMMax;
        cand = reinterpret_cast<int *>(d2 + kJcbbMMax + 1);
        ncand = cand + kJcbbMMax * n;
        jid = ncand + kJcbbMMax;
        hyp = jid + kJcbbMMax;
        best = hyp + kJcbbMMax;
        pk = best + kJcbbMMax;
        it = pk + kJcbbMMax;
        pcnt = it + kJcbbMMax + 1;
    }
};

// One joint test: D^2 of the hypothesis (pairings pk[0..p), D^2 = d2) extended by measurement (z0, z1) paired with landmark k, whose
// individual distance is dik. Appends rows 2p, 2p + 1 to L and y (a sibling overwrites them). The joint S is H Sigma H^T + blockdiag(R)
// at the predicted Sigma; a child whose S is not positive definite comes out NaN or infinite, so it is never accepted. The first
// pairing's D^2 is its individual distance, the same arithmetic as nearest neighbour. Lanes j < p form the cross blocks, lane p the
// diagonal block; lanes 0 and 1 solve L l = cross^T for the two new rows; every lane then forms the same 2 x 2 Schur complement.
__device__ inline double jcbb_joint_test(WarpFilter & f, JcbbScratch & w, double z0, double z1, int k, int p, double dik, double d2,
                                  const double * R)
{
    const int lane = f.lane, len = f.len;
    const double * hq = w.hc + 10 * (k - 1);
    const int cq = 3 + 2 * (k - 1);
    if (lane <= p)
    {
        const int kj = lane < p ? w.pk[lane] : k;
        const double * hj = w.hc + 10 * (kj - 1);
        const int cj = 3 + 2 * (kj - 1);
        const int cols[5] = {0, 1, 2, cj, cj + 1};
        const double hj0[5] = {0.0, hj[0], hj[1], hj[2], hj[3]}, hj1[5] = {-1.0, hj[4], hj[5], hj[6], hj[7]};
        double b00 = 0.0, b01 = 0.0, b10 = 0.0, b11 = 0.0;
#pragma unroll
        for (int t = 0; t < 5; ++t)
        {
            const double * col = f.S + cols[t] * len;
            const double g0 = hq[0] * col[1] + hq[1] * col[2] + hq[2] * col[cq] + hq[3] * col[cq + 1];
            const double g1 = -col[0] + hq[4] * col[1] + hq[5] * col[2] + hq[6] * col[cq] + hq[7] * col[cq + 1];
            b00 += g0 * hj0[t];
            b01 += g0 * hj1[t];
            b10 += g1 * hj0[t];
            b11 += g1 * hj1[t];
        }
        if (lane == p)
        {
            b00 += R[0];
            b10 += R[1];
            b01 += R[2];
            b11 += R[3];
        }
        double * o = w.bx + 4 * lane;   // [a * 2 + b] = (H_new Sigma H_j^T)(a, b)
        o[0] = b00;
        o[1] = b01;
        o[2] = b10;
        o[3] = b11;
    }
    __syncwarp();
    const int P = 2 * p;
    double * l0 = w.L + P * (P + 1) / 2;
    double * l1 = l0 + P + 1;
    if (lane < 2)
    {
        double * lr = lane ? l1 : l0;
        for (int r = 0; r < P; ++r)
        {
            const double * Lr = w.L + r * (r + 1) / 2;
            double v = w.bx[4 * (r >> 1) + 2 * lane + (r & 1)];
            for (int s = 0; s < r; ++s) v -= Lr[s] * lr[s];
            lr[r] = v / Lr[r];
        }
    }
    __syncwarp();
    double s00 = w.bx[4 * p], s10 = w.bx[4 * p + 2], s11 = w.bx[4 * p + 3];
    double n1 = z1 - hq[9];
    if (f.opt & kOptWrapInnovation) n1 = normalize_angle(n1);
    double n0 = z0 - hq[8];
    for (int r = 0; r < P; ++r)
    {
        s00 -= l0[r] * l0[r];
        s10 -= l1[r] * l0[r];
        s11 -= l1[r] * l1[r];
        n0 -= l0[r] * w.y[r];
        n1 -= l1[r] * w.y[r];
    }
    const double a = sqrt(s00), b = s10 / a, e = sqrt(s11 - b * b);
    const double y0 = n0 / a, y1 = (n1 - b * y0) / e;
    __syncwarp();
    if (lane == 0)
    {
        l0[P] = a;
        l1[P] = b;
        l1[P + 1] = e;
        w.y[P] = y0;
        w.y[P + 1] = y1;
    }
    __syncwarp();
    return p == 0 ? dik : d2 + y0 * y0 + y1 * y1;
}

// NUSLAM_OPT_JOINT_COMPATIBILITY: the ids of one step's measurements z[0..mv) (mv <= kJcbbMMax) at the predicted state, into w.jid;
// seen and status as the per-measurement rule would leave them. T[p]: the joint threshold of p pairings (T[1] = amin).
__device__ inline void jcbb_associate(WarpFilter & f, JcbbScratch & w, const double * z, int mv, int & seen, int & status, const double * R,
                               double amin, double amax, const double * T)
{
    const int lane = f.lane, n = f.n, seen0 = seen;
    // individual phase: every (measurement, candidate) pair, spread over the lanes
    for (int k = lane + 1; k <= seen0; k += kWarp)
    {
        HEntries H;
        double zr, zb;
        measurement_model(f.x, 3 + 2 * (k - 1), H, zr, zb);
        double * h = w.hc + 10 * (k - 1);
        h[0] = H.h01;
        h[1] = H.h02;
        h[2] = H.h0c;
        h[3] = H.h0c1;
        h[4] = H.h11;
        h[5] = H.h12;
        h[6] = H.h1c;
        h[7] = H.h1c1;
        h[8] = zr;
        h[9] = zb;
    }
    bool singular = false;
    for (int e = lane; e < mv * seen0; e += kWarp)
    {
        const int i = e / seen0, k = e - i * seen0 + 1;
        bool s = false;
        const double d = f.mahalanobis(z[2 * i], z[2 * i + 1], k, R, s);
        singular |= s;
        w.dist[i * n + k - 1] = d;
    }
    if (__any_sync(0xffffffffu, singular))
    {
        // psi does not depend on the measurement: every measurement has the singular candidate, so the first one throws
        status |= kStatusSingular;
        if (lane == 0) w.jid[0] = kIdException;
        __syncwarp();
        return;
    }
    __syncwarp();
    for (int e = lane; e < mv * seen0; e += kWarp)
    {
        const int i = e / seen0, k = e - i * seen0 + 1;
        const double * di = w.dist + i * n;
        const double d = di[k - 1];
        if (d < amin)
        {
            int r = 0;
            for (int k2 = 1; k2 <= seen0; ++k2)
            {
                const double d2 = di[k2 - 1];
                r += (d2 < amin) && (d2 < d || (d2 == d && k2 < k));
            }
            w.cand[i * n + r] = k;
        }
    }
    if (lane < mv)
    {
        int c = 0;
        for (int k = 1; k <= seen0; ++k) c += w.dist[lane * n + k - 1] < amin;
        w.ncand[lane] = c;
        w.best[lane] = 0;
    }
    __syncwarp();

    // depth-first search over the measurements; every lane runs the same control flow on the same values
    int tests = 0, best_p = 0;
    double best_d2 = 0.0;
    int i = 0, p = 0;
    double d2 = 0.0;
    bool entered = true, running = mv > 0 && seen0 > 0;
    while (running)
    {
        if (entered)
        {
            entered = false;
            if (i < mv && p + (mv - i) >= best_p)
            {
                __syncwarp();
                if (lane == 0)
                {
                    w.it[i] = 0;
                    w.pcnt[i] = p;
                    w.d2[i] = d2;
                }
                __syncwarp();
                continue;
            }
            if (i == mv && (p > best_p || (p == best_p && d2 < best_d2)))
            {
                best_p = p;
                best_d2 = d2;
                __syncwarp();
                if (lane < mv) w.best[lane] = w.hyp[lane];
                __syncwarp();
            }
            --i;   // pruned, or a leaf: back to the parent's next option
            p = w.pcnt[i];
            d2 = w.d2[i];
            continue;
        }
        // node i: its next option
        const int nc = w.ncand[i];
        int pos = w.it[i], k = -1;
        double nd2 = d2;
        while (pos < nc)
        {
            const int kk = w.cand[i * n + pos];
            ++pos;
            bool used = false;
            for (int j = 0; j < p; ++j) used |= w.pk[j] == kk;
            if (used) continue;
            if (tests == kJcbbMaxTests)
            {
                status |= kStatusAssocTruncated;
                running = false;
                break;
            }
            ++tests;
            const double t = jcbb_joint_test(f, w, z[2 * i], z[2 * i + 1], kk, p, w.dist[i * n + kk - 1], d2, R);
            if (t < T[p + 1])
            {
                k = kk;
                nd2 = t;
                break;
            }
        }
        if (!running) break;
        if (k < 0 && pos == nc)   // the null pairing, last
        {
            pos = nc + 1;
            k = 0;
        }
        __syncwarp();
        if (lane == 0)
        {
            w.it[i] = pos;
            if (k >= 0) w.hyp[i] = k;
            if (k > 0) w.pk[p] = k;
        }
        __syncwarp();
        if (k >= 0)
        {
            if (k > 0)
            {
                ++p;
                d2 = nd2;
            }
            ++i;
            entered = true;
        }
        else if (i == 0)
            running = false;
        else
        {
            --i;
            p = w.pcnt[i];
            d2 = w.d2[i];
        }
    }

    // outcome: the best hypothesis' pairings; an unpaired measurement is ambiguous when any candidate lies below amax, and otherwise
    // opens a landmark in measurement order (an exception on a full map, and nothing after it)
    bool full = false;
    for (int r = 0; r < mv; ++r)
    {
        int id = 0;
        if (!full)
        {
            id = w.best[r];
            if (id == 0)
            {
                bool amb = false;
                for (int k = 1; k <= seen0; ++k) amb |= w.dist[r * n + k - 1] < amax;
                if (amb) id = -1;
                else if (seen >= n)
                {
                    status |= kStatusMapFull;
                    full = true;
                    id = kIdException;
                }
                else id = ++seen;
            }
        }
        if (lane == 0) w.jid[r] = id;
    }
    __syncwarp();
}

enum EkfOp
{
    kOpPredict = 0,
    kOpUpdate = 1,
    kOpAssociate = 2,
    kOpInit = 3,
    kOpStep = 4,
    kOpStepJoint = 5   // kOpStep with NUSLAM_OPT_JOINT_COMPATIBILITY and unknown ids
};

struct EkfParams
{
    int64_t batch;
    int len, n, m;
    double * x;          // B x len
    double * sigma;      // B x len x len, column-major per filter
    int32_t * seen;      // B
    int32_t * status;    // B
    const double * twists;   // B x 3
    const double * z;        // B x m x 2
    const int32_t * ids;     // B x m or null
    unsigned options;        // NUSLAM_OPT_* (0 = the reference's behaviour)
    const int32_t * m_valid; // B or null: filter b uses only its first m_valid[b] (<= m) measurements (fused scan step)
    int32_t * ids_out;       // B x m or null
    double * x_snap;         // B x len or null: a second copy of the state vector after the step (pipelined host path: the snapshot the
                             // device -> host copy reads while the next step already runs)
    double Q[9], R[4];
    double amin, amax;
    // launch shape of k_ekf_strict_list for the filters a FAST kernel hands over (strict_tail below); tail_blocks == 0: the host launches it
    int tail_blocks, tail_threads, tail_smem;
    const double * joint_t;  // NUSLAM_OPT_JOINT_COMPATIBILITY: the joint thresholds T[p] of p = 1..kJcbbMMax pairings, or null
};

// per-warp shared memory of the oracle-order kernels, in doubles: the filter, plus the JCBB scratch in the JOINT step
template <int OP>
__host__ __device__ constexpr int strict_warp_doubles(int len, int n)
{
    return OP == kOpStepJoint ? strict_smem_doubles(len) + jcbb_smem_doubles(n) : strict_smem_doubles(len);
}

// One warp replays reference call OP on filter b; Sigma staged through the warp's slice of shared memory.
template <int OP>
__device__ __forceinline__ void strict_filter(const EkfParams & p, const int64_t b, double * smem_warp, const int lane)
{
    WarpFilter f;
    f.carve(smem_warp, p.len, p.n, lane);
    f.opt = p.options;
    double * gx = p.x + b * p.len;
    double * gS = p.sigma + b * (int64_t) p.len * p.len;
    int status = p.status[b];
    int seen = p.seen[b];

    if (OP == kOpInit)
    {
        const int id = p.ids[b];
        if (id <= 0) return;
        for (int e = lane; e < p.len; e += kWarp) f.x[e] = gx[e];
        __syncwarp();
        f.init_landmark(p.z[2 * b], p.z[2 * b + 1], id, status);
        f.store(gx, gS, false);
        if (lane == 0) p.status[b] = status;
        return;
    }

    f.load(gx, gS);
    if (OP == kOpPredict)
    {
        f.predict(p.twists[3 * b], p.twists[3 * b + 1], p.Q);
        f.store(gx, gS, true);
    }
    else if (OP == kOpUpdate)
    {
        const int id = p.ids[b];
        if (id <= 0) return;
        f.update(p.z[2 * b], p.z[2 * b + 1], id, status, p.R);
        f.store(gx, gS, true);
        if (lane == 0) p.status[b] = status;
    }
    else if (OP == kOpAssociate)
    {
        const int id = f.associate(p.z[2 * b], p.z[2 * b + 1], seen, status, p.R, p.amin, p.amax);
        if (lane == 0)
        {
            p.ids_out[b] = id;
            p.seen[b] = seen;
            p.status[b] = status;
        }
    }
    else if (OP == kOpStep || OP == kOpStepJoint)
    {
        // EKFSlam::main_loop, nuslam/src/slam.cpp:262-319
        const int64_t mb = b * p.m;
        if (status & (kStatusMapFull | kStatusSingular))   // the reference process died on an earlier scan
        {
            if (p.ids_out)
                for (int i = lane; i < p.m; i += kWarp) p.ids_out[mb + i] = 0;
            if (p.x_snap)
                for (int e = lane; e < p.len; e += kWarp) p.x_snap[b * p.len + e] = f.x[e];
            return;
        }
        const int seen_snapshot = seen;                               // slam.cpp:251
        f.predict(p.twists[3 * b], p.twists[3 * b + 1], p.Q);         // slam.cpp:269
        const int mv = p.m_valid ? min(p.m, max(0, p.m_valid[b])) : p.m;   // markers this filter received (landmarks.cpp:84-109)
        if (p.ids_out)
            for (int i = mv + lane; i < p.m; i += kWarp) p.ids_out[mb + i] = 0;
        JcbbScratch jw;
        if (OP == kOpStepJoint)
        {
            // every measurement's id at once (the predicted state); the loop below applies them as it would apply associate's
            jw.carve(smem_warp + strict_smem_doubles(p.len), p.n);
            jcbb_associate(f, jw, p.z + 2 * mb, mv, seen, status, p.R, p.amin, p.amax, p.joint_t);
        }
        for (int i = 0; i < mv; ++i)                                  // slam.cpp:279
        {
            const double z0 = p.z[2 * (mb + i)], z1 = p.z[2 * (mb + i) + 1];
            int id;
            if (p.ids)
            {
                id = p.ids[mb + i];
                if (id <= 0)
                {
                    if (p.ids_out && lane == 0) p.ids_out[mb + i] = 0;
                    continue;
                }
                if (id > p.n)
                {
                    // not a landmark of this map: flagged and skipped like the FAST and LARGE paths do, `seen` untouched (the reference
                    // would index its state out of bounds)
                    status |= kStatusBadId;
                    if (p.ids_out && lane == 0) p.ids_out[mb + i] = id;
                    continue;
                }
                if (id > seen) seen = id;
            }
            else
            {
                if (OP == kOpStepJoint) id = jw.jid[i];
                else id = f.associate(z0, z1, seen, status, p.R, p.amin, p.amax);   // slam.cpp:291
                if (id == kIdException)
                {
                    if (p.ids_out)
                        for (int r = i + lane; r < mv; r += kWarp) p.ids_out[mb + r] = (r == i) ? kIdException : 0;
                    break;
                }
            }
            if (p.ids_out && lane == 0) p.ids_out[mb + i] = id;
            if (id > seen_snapshot) f.init_landmark(z0, z1, id, status);   // slam.cpp:295-297
            else if (id < 0) continue;                                      // slam.cpp:298-300
            f.update(z0, z1, id, status, p.R);                              // slam.cpp:318
        }
        f.store(gx, gS, true);
        if (p.x_snap)
            for (int e = lane; e < p.len; e += kWarp) p.x_snap[b * p.len + e] = f.x[e];
        if (lane == 0)
        {
            p.seen[b] = seen;
            p.status[b] = status;
        }
    }
}

// One warp per filter over the whole batch.
template <int OP>
__global__ void __launch_bounds__(128) k_ekf_strict(const EkfParams p)
{
    extern __shared__ double smem[];
    const int warp = threadIdx.x / kWarp, lane = threadIdx.x % kWarp;
    const int64_t b = (int64_t) blockIdx.x * (blockDim.x / kWarp) + warp;
    if (b >= p.batch) return;
    strict_filter<OP>(p, b, smem + (size_t) warp * strict_warp_doubles<OP>(p.len, p.n), lane);
}

// One warp per filter over a device-side work list (the filters the FAST kernel handed over because their step
// contains a landmark's first touch). The last block to finish resets the list for the next launch.
// TU: the translation unit that instantiates it (0 nuslam_b200.cu, whole-program; 1 ekf_fast_tu.cu, relocatable): the two builds of the same
// kernel must not share a name, or the linker would merge their host stubs.
template <int OP, int TU>
__global__ void __launch_bounds__(128) k_ekf_strict_list(const EkfParams p, const int32_t * __restrict__ list, int32_t * count, int32_t * done)
{
    extern __shared__ double smem[];
    const int warps = blockDim.x / kWarp;
    const int warp = threadIdx.x / kWarp, lane = threadIdx.x % kWarp;
    const int n = *reinterpret_cast<volatile int32_t *>(count);
    for (int64_t k = (int64_t) blockIdx.x * warps + warp; k < n; k += (int64_t) gridDim.x * warps)
    {
        strict_filter<OP>(p, list[k], smem + (size_t) warp * strict_smem_doubles(p.len), lane);
        __syncwarp();
    }
    __syncthreads();
    if (threadIdx.x == 0)
    {
        __threadfence();
        if (atomicAdd(done, 1) == (int) gridDim.x - 1)
        {
            *count = 0;
            *done = 0;
            __threadfence();
        }
    }
}

#ifndef NUSLAM_TAIL_LAUNCH
#define NUSLAM_TAIL_LAUNCH 0    // 1: built with -rdc=true + cudadevrt; the FAST kernels launch the list kernel themselves, and only when needed
#endif

// Every warp of a FAST kernel calls this when it has finished its filters. The LAST warp of the grid looks at the work list and, if a
// filter was handed over, launches k_ekf_strict_list into the tail-launch stream: it runs after this grid has completed and before the
// next kernel of the host stream starts. A step without a first touch -- every step of a built map -- is ONE launch.
// wl_count: [0] entries, [1] finished blocks of the list kernel, [2] finished warps of the FAST kernel, [3] sticky device-launch error
__device__ __forceinline__ void strict_tail(const EkfParams & p, const int do_predict, int32_t * worklist, int32_t * wl_count, const int total_warps,
                                            const int lane)
{
#if NUSLAM_TAIL_LAUNCH && defined(NUSLAM_TU_FAST)   // (a device-side launch compiles only as relocatable device code)
    if (p.tail_blocks == 0) return;
    __syncwarp();
    if (lane == 0)
    {
        __threadfence();
        if (atomicAdd(wl_count + 2, 1) == total_warps - 1)
        {
            wl_count[2] = 0;
            __threadfence();
            if (*reinterpret_cast<volatile int32_t *>(wl_count) > 0)
            {
                // (inlined on purpose: an out-of-line launcher takes the parameter block through the stack and costs the kernels registers)
                if (do_predict)
                    k_ekf_strict_list<kOpStep, 1><<<p.tail_blocks, p.tail_threads, p.tail_smem, cudaStreamTailLaunch>>>(p, worklist, wl_count, wl_count + 1);
                else
                    k_ekf_strict_list<kOpUpdate, 1><<<p.tail_blocks, p.tail_threads, p.tail_smem, cudaStreamTailLaunch>>>(p, worklist, wl_count, wl_count + 1);
                const cudaError_t e = cudaGetLastError();
                if (e != cudaSuccess)
                {
                    wl_count[3] = (int32_t) e;   // reported by the next synchronize
                    wl_count[0] = 0;             // the next step must not replay this step's entries
                }
            }
        }
    }
#endif
}

}   // namespace nuslam
