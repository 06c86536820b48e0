// scan_moment.cuh -- the throughput path of the landmark detector: ONE fused kernel, one warp per 360-beam scan.
//
//   clusterPoints (circle_fit_library.cpp:136-206)  ballots + popcounts over the beams, as in scan_detect.cuh: cluster ids are
//                                                   integer work and stay bit-exact, every quirk of SURVEY.md Appendix A-11 included;
//                                                   the erase loop's two-state walk (:198-204) is evaluated in closed form (a run of
//                                                   consecutive small clusters alternates erased / kept, starting with erased)
//   classifyCluster (:208-250)                      one point per lane: inscribed angles, warp-shuffle segmented sums
//   circleFit (:15-134)                             the Hyper algebraic fit (Al-Sharadqah / Chernov) from WARP-SHUFFLE MOMENT REDUCTIONS:
//                                                   centroid, then the six centred moments of (x, y, z = x^2 + y^2), one lane per
//                                                   cluster solves the characteristic polynomial by Newton's iteration from 0 (its
//                                                   smallest non-negative root is the "smallest positive eigenvalue" of :91-101) and
//                                                   forms centre and radius in closed form
//   Landmarks::main_loop (landmarks.cpp:84-109)     id < 0 / R > 1 filters, circles in detection order
//
// The reference reaches the same A = argmin A^T M A / A^T H A through svd -> Y = V S V^T -> eig_sym(Y H^-1 Y) -> solve; on its own
// kind of data the two routes agree to ~1e-13 relative (measured against oracle/_ref on 36 828 fits: worst published circle 8.4e-14,
// no gate decision differs). Where a decision of the reference could hinge on rounding -- the classifier's std within 1e-6 of 10
// degrees, R within 1e-6 of the 1 m gate, a non-finite result, Newton not converging, nearly collinear points that would still be
// published -- the scan is handed to the oracle-order kernels of scan_detect.cuh (one-sided Jacobi SVD etc.) through a work list.
// Tolerance on circles: 1e-9 relative (BASELINE.json north_star); cluster ids, cluster and circle counts: exact.
#pragma once
#include "scan_detect.cuh"
#include "fastmath.cuh"

namespace nuslam
{

constexpr int kMomWarps = 4;          // scans per CTA
constexpr int kMomMaxClusters = 32;   // pre-erase clusters handled by the warp (one per lane); busier scans take the work list
constexpr int kMomSums = 10;          // per cluster: X, Y, XX, YY, XY, XZ, YZ, ZZ about its first point, angle, angle^2

struct __align__(16) MomentSmem
{
    unsigned pb[kBeams + 8];                  // flat position (in-range beams in beam order) -> beam | pre-erase cluster << 16
    double acc[kMomMaxClusters][kMomSums];    // per cluster: the sums above
    double org[kMomMaxClusters][2];           // per cluster: its first point (local origin of the sums)
    short cend[kMomMaxClusters + 8];          // flat position of the cluster's last point
    short nidx[kMomMaxClusters];              // pre-erase cluster -> index among the returned clusters (-1: erased)
};

// the atan2 tables of fastmath.cuh in shared memory (the lanes index them with different entries, which the constant cache serialises)
struct MomentTables
{
    double2 tab[65];
    AtanOctant oct[8];
};

// atan2_fast (fastmath.cuh) on shared-memory tables: ~1e-16 absolute
__device__ __forceinline__ double atan2_tab(double y, double x, const MomentTables & T)
{
    const double ax = fabs(x), ay = fabs(y);
    const bool sw = ay > ax;
    const double mx = sw ? ay : ax, mn = sw ? ax : ay;
    const int idx = (sw ? 1 : 0) | (x < 0.0 ? 2 : 0) | (y < 0.0 ? 4 : 0);
    const float tf = __fdividef((float) mn, (float) mx);
    const int k = max(0, min(64, __float2int_rn(tf * 64.0f)));
    const double tk = (double) k * 0.015625;
    const double2 ak = T.tab[k];
    const AtanOctant oc = T.oct[idx];
    const double num = fma(-tk, mx, mn), den = fma(tk, mn, mx);
    const double rc = rcp_fast(den);
    double r = num * rc;
    r = fma(fma(-den, r, num), rc, r);   // r = num / den to ~1 ulp
    const double u = r * r;
    const double pl = fma(fma(fma(kFastK[0], u, kFastK[1]), u, kFastK[2]), u * r, r);   // atan(r)
    const double a = ak.x + (pl + ak.y);                                              // atan(mn / mx) in [0, pi/4]
    return oc.hi + fma(oc.s, a, oc.lo);
}

struct ScanGate
{
    float max_f, min_f;   // r > max_range <=> r > max_f, r < min_range <=> r < min_f for every float r (the reference compares in double)
};

// largest float <= v / smallest float >= v (host side)
inline float float_below(double v)
{
    float f = (float) v;
    if ((double) f > v) f = nextafterf(f, -INFINITY);
    return f;
}
inline float float_above(double v)
{
    float f = (float) v;
    if ((double) f < v) f = nextafterf(f, INFINITY);
    return f;
}

constexpr int kMomMinBlocks = 8;   // resident CTAs per SM the register allocation aims at (8 x 4 warps: 64 registers)
__global__ void __launch_bounds__(32 * kMomWarps, kMomMinBlocks)
k_scan_moment(const float * __restrict__ ranges, const int64_t n_scans, const double min_range, const double max_range, const ScanGate gate,
              int16_t * __restrict__ cluster_of_beam, int32_t * __restrict__ n_clusters, int32_t * __restrict__ n_circles,
              double * __restrict__ circles, const int max_circles, const int scan_ub, int32_t * __restrict__ slow, int32_t * __restrict__ slow_count)
{
    __shared__ MomentSmem smem_all[kMomWarps];
    __shared__ __align__(16) MomentTables tabs;
    MomentSmem & sm = smem_all[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;
    constexpr unsigned kFull = 0xffffffffu;
    constexpr int kPer = 12;                      // beams per lane in the clustering walk
    static_assert(kBeams % kPer == 0 && kBeams / kPer <= 32 && kPer % 4 == 0, "lane-major walk: 30 lanes x 12 beams");
    const bool vec_ok = (reinterpret_cast<uintptr_t>(ranges) & 15) == 0;
    const unsigned lt = (1u << lane) - 1u;
    for (int k = threadIdx.x; k < 65 + 16; k += blockDim.x)
    {
        if (k < 65) tabs.tab[k] = kAtanTab[k];
        else reinterpret_cast<double2 *>(tabs.oct)[k - 65] = reinterpret_cast<const double2 *>(kAtanOct)[k - 65];
    }
    __syncthreads();
    for (int64_t s = (int64_t) blockIdx.x * kMomWarps + (threadIdx.x >> 5); s < n_scans; s += (int64_t) gridDim.x * kMomWarps)
    {
        const float * rs = ranges + s * kBeams;
        // ---- per-beam predicates (circle_fit_library.cpp:146-190), LANE-MAJOR: lane L owns the kPer = 12 consecutive beams 12 L .. 12 L + 11
        // (lanes 30 and 31 own none), so a beam's successor sits in the same lane's registers (one shuffle per scan for the lane
        // boundary), the in-range / closer predicates become two 12-bit masks per lane, and flat positions and cluster numbers come from
        // ONE warp prefix sum of the two popcounts instead of two ballots and four popcounts per 32 beams ----
        // closer_i = in range and not similar to beam i + 1; the cluster of an in-range beam = closers before it
        const bool own = lane < kBeams / kPer;
        float r[kPer + 1];
        if (vec_ok)   // warp-uniform
        {
            const float4 * r4 = reinterpret_cast<const float4 *>(rs + kPer * (own ? lane : 0));   // 48 B per lane, 16-byte aligned whenever the array is
#pragma unroll
            for (int j = 0; j < kPer / 4; ++j)
            {
                const float4 v = __ldg(r4 + j);
                r[4 * j] = v.x, r[4 * j + 1] = v.y, r[4 * j + 2] = v.z, r[4 * j + 3] = v.w;
            }
        }
        else
        {
#pragma unroll
            for (int k = 0; k < kPer; ++k) r[k] = __ldg(rs + kPer * (own ? lane : 0) + k);
        }
        {
            const float r_first = __shfl_sync(kFull, r[0], 0);
            const float r_up = __shfl_down_sync(kFull, r[0], 1);
            r[kPer] = (lane == kBeams / kPer - 1) ? r_first : r_up;   // the successor of beam 359 is beam 0
        }
        // (lanes 30 and 31 carry a copy of lane 0's beams: `own` masks their predicates)
        unsigned inr_bits = 0u, clo_bits = 0u, risky_bits = 0u;
        const bool big_gate = !(gate.max_f <= 32.0f);   // warp-uniform
#pragma unroll
        for (int k = 0; k < kPer; ++k)
        {
            const float rv = r[k], nb = r[k + 1];
            const bool inr = !(rv > gate.max_f) & !(rv < gate.min_f);   // :149, NaN counts as in range
            // :166 |r_i - r_(i+1)| < 0.04 in double. The float difference is within an ulp of the exact one: decided in float; a scan
            // where it lies within 1e-5 of the threshold (or a range is huge / NaN) goes to the oracle-order kernel, which compares
            // in double like the reference
            const float df = fabsf(rv - nb);
            const bool sim = df < 0.04f;
            const bool near = !(fabsf(df - 0.04f) >= 1e-5f);
            // branch-free on purpose (no short-circuit operators): three predicate instructions per beam instead of a branch ladder
            inr_bits |= inr ? (1u << k) : 0u;
            clo_bits |= (inr & !sim) ? (1u << k) : 0u;
            risky_bits |= (inr & near) ? 1u : 0u;
        }
        if (big_gate)
        {
            // (an in-range beam is below max_f; when that is at most 32 m a neighbour of 64 m or more is nowhere near the threshold, and a
            // NaN fails the first test by itself: the magnitude test is needed only for range gates beyond 32 m)
#pragma unroll
            for (int k = 0; k < kPer; ++k)
                risky_bits |= (((inr_bits >> k) & 1u) && !(fmaxf(fabsf(r[k]), fabsf(r[k + 1])) < 64.0f)) ? 1u : 0u;
        }
        if (!own) inr_bits = clo_bits = risky_bits = 0u;
        const bool risky = risky_bits != 0u;
        // beam 359 in range and similar to beam 0: it is not stored in the flat list but appended to cluster 0 (:170-174)
        constexpr unsigned kLastBit = 1u << (kPer - 1);
        const bool wrap = __shfl_sync(kFull, (int) ((inr_bits & kLastBit) && !(clo_bits & kLastBit)), kBeams / kPer - 1) != 0;
        if (wrap && lane == kBeams / kPer - 1) inr_bits &= ~kLastBit;
        // flat position of this lane's first in-range beam and closers before it: one inclusive prefix sum over (points | closers << 16)
        const unsigned cnt = (unsigned) __popc(inr_bits) | ((unsigned) __popc(clo_bits) << 16);
        unsigned incl = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1)
        {
            const unsigned up = __shfl_up_sync(kFull, incl, d);
            if (lane >= d) incl += up;
        }
        const unsigned total = __shfl_sync(kFull, incl, 31);
        const int npts = (int) (total & 0xffffu), nc = (int) (total >> 16);
        const int pos0 = (int) ((incl - cnt) & 0xffffu), clu0 = (int) ((incl - cnt) >> 16);
        const int64_t sb = s * kBeams;
        if (wrap && nc == 0)
        {
            // clusters[0].push_back on an empty vector (:173): undefined behaviour in the reference
            if (cluster_of_beam)
                for (int i = lane; i < kBeams; i += 32) cluster_of_beam[sb + i] = -1;
            if (lane == 0)
            {
                n_clusters[s] = 0;
                n_circles[s] = scan_ub;
            }
            __syncwarp();
            continue;
        }
        if (nc > kMomMaxClusters || __any_sync(kFull, risky))
        {
            if (lane == 0) slow[atomicAdd(slow_count, 1)] = (int32_t) s;   // the one-warp-per-scan kernel writes every output of this scan
            __syncwarp();
            continue;
        }
        // the flat list of in-range beams (beam | cluster << 16) and the flat position of every cluster's last point
        {
            // running store address, list entry (beam | cluster << 16) and position: one predicated add each per beam
            unsigned * ap = sm.pb + pos0;
            unsigned ent = (unsigned) (kPer * lane) | ((unsigned) clu0 << 16);
            int pos = pos0;
#pragma unroll
            for (int k = 0; k < kPer; ++k)
            {
                const bool in = (inr_bits >> k) & 1u, cl = (clo_bits >> k) & 1u;
                // two independent predicated stores (a closer is in range): no nested branch
                if (in) *ap = ent + (unsigned) k;
                if (cl) sm.cend[(ent >> 16) & (kMomMaxClusters - 1)] = (short) pos;
                ap += in ? 1 : 0;
                pos += in ? 1 : 0;
                ent += cl ? 0x10000u : 0u;
            }
        }
        __syncwarp();
        // ---- one cluster per lane: extent, erase loop (:198-204) in closed form ----
        const int cend = (lane < nc) ? (int) sm.cend[lane] : -1;
        int cstart = __shfl_up_sync(kFull, cend, 1) + 1;
        if (lane == 0) cstart = 0;
        const int csize = (lane < nc) ? cend - cstart + 1 + ((lane == 0 && wrap) ? 1 : 0) : 0;
        const bool small = lane < nc && csize < 3;
        const unsigned small_m = __ballot_sync(kFull, small);
        const unsigned big_below = ~small_m & lt;
        const int run = big_below ? lane - 1 - (31 - __clz((int) big_below)) : lane;   // consecutive small clusters right below this one
        const bool erased = small && !(run & 1);   // a cluster following an erased one is never examined
        const unsigned erased_m = __ballot_sync(kFull, erased);
        const int newidx = (lane < nc && !erased) ? lane - __popc(erased_m & lt) : -1;
        const int nk = nc - __popc(erased_m);
        if (cluster_of_beam)
        {
            // the pre-erase cluster of a beam (closers before it) -> its index among the returned clusters through a 32-entry table; a
            // lane's 12 ids leave as three 8-byte stores (a scan's ids start at a multiple of 8 bytes whenever the array does)
            const int new0 = __shfl_sync(kFull, newidx, 0);
            sm.nidx[lane] = (short) newidx;
            __syncwarp();
            if (own)
            {
                unsigned o[kPer];
                int c = clu0;
#pragma unroll
                for (int k = 0; k < kPer; ++k)
                {
                    // beams out of range, and beams behind the last closer (the open cluster the reference drops): -1
                    const unsigned v = (unsigned) (unsigned short) sm.nidx[c & (kMomMaxClusters - 1)];
                    o[k] = (((inr_bits >> k) & 1u) & (c < nc)) ? v : 0xffffu;
                    c += (clo_bits >> k) & 1u;
                }
                if (wrap && lane == kBeams / kPer - 1) o[kPer - 1] = (unsigned) (unsigned short) new0;   // beam 359 belongs to cluster 0
                int16_t * dst = cluster_of_beam + sb + kPer * lane;
                if ((reinterpret_cast<uintptr_t>(cluster_of_beam) & 7) == 0)
                {
#pragma unroll
                    for (int j = 0; j < kPer / 4; ++j)
                        reinterpret_cast<uint2 *>(dst)[j] = make_uint2(o[4 * j] | (o[4 * j + 1] << 16), o[4 * j + 2] | (o[4 * j + 3] << 16));
                }
                else
                {
#pragma unroll
                    for (int k = 0; k < kPer; ++k) dst[k] = (int16_t) o[k];
                }
            }
        }
        // ---- points: one per lane, ONE pass of segmented warp sums about the cluster's first point: the sums the Hyper fit needs and
        // the inscribed angles of classifyCluster. A cluster is examined when it survives the erase loop and has at least 3 points
        // (fewer: classifyCluster's std is 0/0 = NaN, :229-249)
        const bool examined = lane < nc && !erased && csize >= 3;
        const int ntot = npts + (wrap ? 1 : 0);
#pragma unroll 1
        for (int base = 0; base < ntot; base += 32)
        {
            const int j = base + lane;
            const bool iswrap = wrap && j == npts;
            const unsigned pbv = (j < npts) ? sm.pb[j] : 0u;
            const int beam = iswrap ? kBeams - 1 : (int) (pbv & 0xffffu);
            const int clu = iswrap ? 0 : (int) (pbv >> 16);
            const int src = clu & 31;
            const int cs = __shfl_sync(kFull, cstart, src), ce = __shfl_sync(kFull, cend, src);
            const bool ex = __shfl_sync(kFull, examined ? 1 : 0, src) != 0;
            const bool active = (j < npts || iswrap) && clu < nc && ex;
            const bool wrapped_cluster = wrap && clu == 0;
            const int b2 = active ? (int) (sm.pb[cs] & 0xffffu) : 0;
            const int b3 = !active ? 0 : wrapped_cluster ? kBeams - 1 : (int) (sm.pb[ce] & 0xffffu);
            // points = r (cos, sin)(deg2rad(beam)) (:161-163), relative to the cluster's first point
            const double r1 = (double) __ldg(rs + beam), r2 = (double) __ldg(rs + b2), r3 = (double) __ldg(rs + b3);
            const double x2 = r2 * __ldg(&c_beam_cos[b2]), y2 = r2 * __ldg(&c_beam_sin[b2]);
            const double X = active ? fma(r1, __ldg(&c_beam_cos[beam]), -x2) : 0.0, Y = active ? fma(r1, __ldg(&c_beam_sin[beam]), -y2) : 0.0;
            const double Z = fma(X, X, Y * Y);
            double v[kMomSums];
            v[0] = X;
            v[1] = Y;
            v[2] = X * X;
            v[3] = Y * Y;
            v[4] = X * Y;
            v[5] = X * Z;
            v[6] = Y * Z;
            v[7] = Z * Z;
            // inscribed angle of an interior point P1 over the chord P2 (first) -> P3 (last as stored) (:211-224), in degrees
            const bool last = iswrap || (!wrapped_cluster && j == ce);
            double ang = 0.0;
            if (active && j != cs && !last)
            {
                const double X3 = fma(r3, __ldg(&c_beam_cos[b3]), -x2), Y3 = fma(r3, __ldg(&c_beam_sin[b3]), -y2);
                const double num = fma(Y, X3, -(Y3 * X));
                const double den = -fma(X, X - X3, Y * (Y - Y3));
                ang = (180.0 / kPiRef) * atan2_tab(num, den, tabs);
            }
            v[8] = ang;
            v[9] = ang * ang;
            // segmented inclusive scan: lanes of one cluster are contiguous; as many doubling steps as the longest run in this batch needs
            const int key = active ? (iswrap ? 32 : clu) : -1 - lane;
            const int runpos = (active && !iswrap) ? j - max(cs, base) : 0;
            const int maxrun = __reduce_max_sync(kFull, runpos);
#pragma unroll 1
            for (int d = 1; d <= maxrun; d <<= 1)
            {
                const int kk = __shfl_up_sync(kFull, key, d);
                const bool take = lane >= d && kk == key;
#pragma unroll
                for (int k = 0; k < kMomSums; ++k)
                {
                    const double tv = __shfl_up_sync(kFull, v[k], d);
                    if (take) v[k] += tv;
                }
            }
            const int key_next = __shfl_down_sync(kFull, key, 1);   // (every lane takes part: no collective behind a short-circuit)
            const bool tail = lane == 31 || key_next != key;
            const bool first = cs >= base;   // the cluster's first contribution to its accumulators
            const bool mine = tail && active && !iswrap;
            if (__all_sync(kFull, !mine || first))   // usual case: every cluster of this batch starts in it -- plain stores
            {
                if (mine)
                {
#pragma unroll
                    for (int k = 0; k < kMomSums; ++k) sm.acc[clu][k] = v[k];
                    sm.org[clu][0] = x2;
                    sm.org[clu][1] = y2;
                }
            }
            else if (mine)
            {
#pragma unroll
                for (int k = 0; k < kMomSums; ++k) sm.acc[clu][k] = first ? v[k] : sm.acc[clu][k] + v[k];
                sm.org[clu][0] = x2;
                sm.org[clu][1] = y2;
            }
            __syncwarp();
            if (active && iswrap)
            {
#pragma unroll
                for (int k = 0; k < kMomSums; ++k) sm.acc[0][k] += v[k];
            }
            __syncwarp();
        }
        // ---- one cluster per lane: classification, Hyper fit, gates ----
        bool pub = false, fallback = false;
        double cx = 0.0, cy = 0.0, R = 0.0;
        if (examined)
        {
            const double n = (double) csize, inv_n = rcp_fast(n), inv_na = rcp_fast((double) (csize - 2));
            const double * S = sm.acc[lane];
            const double mean = S[8] * inv_na;
            const double var = fma(-mean, mean, S[9] * inv_na);   // population variance of the angles in degrees (:229-241); one angle: 0
            // std < 10 degrees <=> var < 100 (:243); within 1e-6 degrees of the gate (or not finite): the oracle-order kernel decides
            if (!(fabs(var - 100.0) > 2e-5)) fallback = true;
            const bool circle = var < 100.0;
            if (circle && csize >= 4)   // circleFit rejects N < 4 with id = -1 (:72-76)
            {
                // centroid (relative to the first point) and the centred moments from the sums about the first point
                const double Sx = S[0], Sy = S[1], Sxx = S[2], Syy = S[3], Sxy = S[4], Sxz = S[5], Syz = S[6], Szz = S[7];
                const double a = Sx * inv_n, b = Sy * inv_n, Sz = Sxx + Syy, q = fma(a, a, b * b);
                const double Mxx = fma(-a, a, Sxx * inv_n), Myy = fma(-b, b, Syy * inv_n), Mxy = fma(-a, b, Sxy * inv_n);
                const double Cxz = Sxz - 2.0 * a * Sxx - 2.0 * b * Sxy + q * Sx - a * Sz + 2.0 * a * a * Sx + 2.0 * a * b * Sy - a * q * n;
                const double Cyz = Syz - 2.0 * b * Syy - 2.0 * a * Sxy + q * Sy - b * Sz + 2.0 * b * b * Sy + 2.0 * a * b * Sx - b * q * n;
                const double Czz = Szz - 4.0 * a * Sxz - 4.0 * b * Syz + 2.0 * q * Sz + 4.0 * a * a * Sxx + 8.0 * a * b * Sxy + 4.0 * b * b * Syy -
                                   4.0 * a * q * Sx - 4.0 * b * q * Sy + n * q * q;
                const double Mxz = Cxz * inv_n, Myz = Cyz * inv_n, Mzz = Czz * inv_n;
                const double Mz = Mxx + Myy;
                const double Cov = fma(Mxx, Myy, -Mxy * Mxy);
                const double Var = fma(-Mz, Mz, Mzz);
                // characteristic polynomial of M A = eta H A (Hyper constraint), divided by its trivial factor
                const double A2 = 4.0 * Cov - 3.0 * Mz * Mz - Mzz;
                const double A1 = Var * Mz + 4.0 * Cov * Mz - Mxz * Mxz - Myz * Myz;
                const double A0 = Mxz * (Mxz * Myy - Myz * Mxy) + Myz * (Myz * Mxx - Mxz * Mxy) - Var * Cov;
                const double A22 = A2 + A2;
                double eta = 0.0, yv = A0;
                bool converged = false;
                // Newton from 0 approaches the smallest non-negative root monotonically and needs 4 - 6 steps on a scan's clusters: the first
                // three are taken without looking (a breakdown turns into NaN / inf, which the tested steps below reject)
#pragma unroll
                for (int it = 0; it < 3; ++it)
                {
                    const double Dy = fma(eta, fma(16.0 * eta, eta, A22), A1);
                    eta = fma(-yv, rcp_fast(Dy), eta);
                    yv = fma(eta, fma(eta, fma(4.0 * eta, eta, A2), A1), A0);
                }
#pragma unroll 1
                for (int it = 3; it < 16; ++it)
                {
                    const double Dy = fma(eta, fma(16.0 * eta, eta, A22), A1);
                    const double en = fma(-yv, rcp_fast(Dy), eta);
                    if (!(fabs(en) < 1e300)) break;
                    if (fabs(en - eta) <= 4e-16 * fabs(en))
                    {
                        converged = true;
                        break;
                    }
                    const double yn = fma(en, fma(en, fma(4.0 * en, en, A2), A1), A0);
                    if (fabs(yn) >= fabs(yv))
                    {
                        converged = true;   // the residual no longer shrinks: eta is the root to rounding
                        break;
                    }
                    eta = en;
                    yv = yn;
                }
                const double DET = fma(eta, eta, fma(-eta, Mz, Cov));
                const double hdet = 0.5 * rcp_fast(DET);
                const double hx = (Mxz * (Myy - eta) - Myz * Mxy) * hdet;
                const double hy = (Myz * (Mxx - eta) - Mxz * Mxy) * hdet;
                R = sqrt(fma(hx, hx, fma(hy, hy, Mz - eta - eta)));
                cx = hx + a + sm.org[lane][0];
                cy = hy + b + sm.org[lane][1];
                pub = !(R > 1.0);   // landmarks.cpp:95; a NaN radius would pass the reference's gate: never decided here
                if (!converged || !(fabs(R) < 1e300) || !(fabs(cx) < 1e300) || !(fabs(cy) < 1e300)) fallback = true;
                if (fabs(R - 1.0) < 1e-6) fallback = true;
                if (pub && !(Cov > 1e-9 * Mz * Mz)) fallback = true;   // nearly collinear yet published: conditioning too poor to promise 1e-9
            }
        }
        if (__any_sync(kFull, fallback))
        {
            if (lane == 0) slow[atomicAdd(slow_count, 1)] = (int32_t) s;   // rewrites every output of this scan (cluster_of_beam stays the same)
            __syncwarp();
            continue;
        }
        // ---- publication in detection order (landmarks.cpp:84-109) ----
        const unsigned pm = __ballot_sync(kFull, pub);
        if (pub)
        {
            const int slot = __popc(pm & lt);
            if (slot < max_circles)
            {
                double * cout = circles + (s * (int64_t) max_circles + slot) * 4;
                cout[0] = cx;
                cout[1] = cy;
                cout[2] = R;
                cout[3] = (double) newidx;
            }
        }
        if (lane == 0)
        {
            n_clusters[s] = nk;
            n_circles[s] = __popc(pm);
        }
        __syncwarp();
    }
}

// circle-fit arithmetic of the throughput path: the moment route above (default) or the oracle-order Jacobi pipeline of scan_detect.cuh
constexpr int kFitMoment = 0, kFitJacobi = 1;
inline int & scan_fit_mode()
{
    static int mode = [] {
        const char * e = getenv("NUSLAM_SCAN_FIT");
        return (e && (e[0] == 'j' || e[0] == 'J' || e[0] == '1')) ? kFitJacobi : kFitMoment;
    }();
    return mode;
}

inline ScanScratch & moment_scratch(int device)
{
    static thread_local ScanScratch scratch[64];
    return scratch[(device >= 0 && device < 64) ? device : 0];
}

inline cudaError_t launch_scan_moment(const float * ranges, int64_t n_scans, double min_range, double max_range, int16_t * cluster_of_beam,
                                      int32_t * n_clusters, int32_t * n_circles, double * circles, int32_t max_circles, int scan_ub,
                                      int device, int sm_count, cudaStream_t stream)
{
    cudaError_t e = scan_tables_init(device);
    if (e != cudaSuccess) return e;
    // work list of the scans that need the oracle-order kernel + its counter
    ScanScratch & sc = moment_scratch(device);
    size_t need = ((size_t) n_scans * sizeof(int32_t) + 255) / 256 * 256 + 256;
    if (sc.bytes >= need) need = sc.bytes;   // the counter lives in the last 256 bytes of the allocation
    if (sc.bytes < need)
    {
        if (sc.p) cudaFree(sc.p);
        sc.p = nullptr;
        sc.bytes = 0;
        e = cudaMalloc(&sc.p, need);
        if (e != cudaSuccess) return e;
        sc.bytes = need;
    }
    int32_t * slow = static_cast<int32_t *>(sc.p);
    int32_t * slow_count = reinterpret_cast<int32_t *>(static_cast<char *>(sc.p) + need - 256);
    e = cudaMemsetAsync(slow_count, 0, sizeof(int32_t), stream);
    if (e != cudaSuccess) return e;
    ScanGate gate;
    gate.max_f = float_below(max_range);
    gate.min_f = float_above(min_range);
    int64_t blocks = (n_scans + kMomWarps - 1) / kMomWarps;
    const int64_t resident = (int64_t) sm_count * kMomMinBlocks;
    if (blocks > resident) blocks = resident;
    if (blocks < 1) blocks = 1;
    k_scan_moment<<<(unsigned) blocks, 32 * kMomWarps, 0, stream>>>(ranges, n_scans, min_range, max_range, gate, cluster_of_beam, n_clusters, n_circles,
                                                                 circles, max_circles, scan_ub, slow, slow_count);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    // the scans the moment route does not decide: oracle-order clustering + Jacobi fit, one warp per scan (usually an empty list)
    const size_t smem = sizeof(ScanSmem) * kScanWarps;
    static bool configured_dev[kMaxDevices] = {false};
    bool & configured = configured_dev[(device >= 0 && device < kMaxDevices) ? device : 0];
    if (!configured)
    {
        e = cudaFuncSetAttribute(k_scan_detect<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    ScanPipe none;
    memset(&none, 0, sizeof(none));
    int64_t sblocks = (n_scans + kScanWarps - 1) / kScanWarps;
    if (sblocks > sm_count) sblocks = sm_count;
    k_scan_detect<true><<<(unsigned) sblocks, 32 * kScanWarps, smem, stream>>>(ranges, n_scans, min_range, max_range, cluster_of_beam, n_clusters, n_circles,
                                                                            circles, max_circles, scan_ub, slow, slow_count, none);
    return cudaGetLastError();
}

// number of scans the last launch_scan_moment of this thread on `device` handed to the oracle-order kernel (diagnostics; blocking copy)
inline int scan_moment_fallbacks(int device)
{
    ScanScratch & sc = moment_scratch(device);
    if (!sc.p || sc.bytes < 256) return -1;
    int32_t v = -1;
    if (cudaMemcpy(&v, static_cast<char *>(sc.p) + sc.bytes - 256, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    return (int) v;
}

}   // namespace nuslam
