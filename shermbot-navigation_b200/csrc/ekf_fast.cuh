// ekf_fast.cuh -- FAST arithmetic: fused predict + m sequential updates, one filter per warp, Sigma in REGISTERS.
//
// Roofs (MEASURED on B200, tools/ubench_fp64.cu, profiles/ubench_fp64_r01.txt): the fp64 pipe issues 64 FMA/clk/SM
// for DFMA and for DMMA alike (one pipe: mixing them adds nothing), a dependent DFMA takes 8.7 cycles, shared memory
// returns 256 B/clk/SM (a broadcast LDS.128 costs 2 cycles). A filter-step is ~21 k fp64 FMAs of rank-2 updates
// against 12 352 algorithmic bytes, so the fp64 pipe and HBM (~530 cycles/filter-step/SM at the measured 6.55 TB/s)
// are co-roofs, with the shared-memory pipe close behind; the design below minimises all three per update.
//
// Layout of one filter inside its warp (state order [theta, x, y, m1x, m1y, ...], slam_library.cpp:46-59):
//   * landmark block Sigma(3.., 3..) (2N x 2N): fp64 tensor-core accumulator fragments of mma.m8n8k4 -- block
//     (br, bc), lane (g = lane / 4, t = lane % 4) holds Sigma(3 + 8 br + g, 3 + 8 bc + 2 t + {0, 1}); 18 doubles
//     per lane at N = 12 with no padding waste.
//   * robot rows / columns Sigma({th,x,y}, :) and Sigma(:, {th,x,y}) in VECTOR layout: lane i holds entry i of each
//     of the 6 vectors Rt, Rx, Ry (rows) and Ct, Cx, Cy (columns); the 3 x 3 robot block lives in both (updated
//     with bit-identical operations). predict (slam_library.cpp:65-108) touches only these vectors.
//   * the state x in vector layout (lane i holds x_i); the robot pose (theta, x, y) also replicated in every lane.
// One update (slam_library.cpp:263-282), with H = D Ht, D = diag(1/sqrt d, 1/d), Ht = [0 -dx -dy dx dy; -d dy -dx
// -dy dx] free of divisions:   Sigma' = Sigma - Pt Minv Wt,  x' = x + Pt Minv (sqrt d dz0, d dz1),
//   Pt = Sigma Ht^T (lane i = row i), Wt = Ht Sigma (lane j = column j), M = Wt Ht^T + D^-1 R D^-1.
//   (A) the landmark's two rows and two columns are published from the fragments through shared memory into
//       vector layout; (B) lanes form Pt, Wt and exchange Wt; every lane evaluates the 2 x 2 part (M, one
//       reciprocal, sqrt d from a one-Newton rsqrt, a division-free atan2 of the unit vector, innovation) redundantly -- no
//       cross-warp synchronisation anywhere in the kernel, the 16 resident warps of an SM hide each other's dependency
//       chains; (C) lanes form Kt = Pt Minv, update x, the replicated pose and the 6 robot vectors with plain FMAs;
//   (D) updates are applied to the fragments LAZILY in chunks of 2: the second update of a chunk takes its
//       landmark rows / columns from the stale fragments and corrects them in vector layout with the first update
//       (4 vectors x 2 FMAs), then ONE rank-4 DMMA pass (9 mma.m8n8k4 at N = 12, k = 4 fully used) applies both.
//
// Both triangles of Sigma are kept: the reference's Sigma is NOT symmetric (its INT_MAX first touches leave |Sigma - Sigma^T| at
// ~1e-6 relative and (I - KH) Sigma never restores it), and rows and columns enter the update separately (DESIGN.md 5.1).
// Arithmetic: predict uses the oracle's operation order on the covariance (it is O(len)), one call-free sincos (fastmath.cuh sincos_fast) plus the
// addition theorems for the three angles. A filter-step that contains a landmark's
// FIRST TOUCH (INT_MAX prior, slam_library.cpp:28-31, where only the reference's own operation order reproduces its
// catastrophic cancellation, SURVEY.md Appendix B) or an initializeLandmark is not evaluated here: the filter is
// appended to a work list that the STRICT kernel (ekf_strict.cuh) processes right after on the same stream (launched by this
// kernel itself in the relocatable unit -- strict_tail -- or by the host in the whole-program unit).
// Reference: nuslam/src/slam_library.cpp:65-108 (predict), :263-282 (update), nuslam/src/slam.cpp:262-319.
#pragma once
#include "ekf_fast_api.cuh"
#include "ekf_strict.cuh"
#include "fastmath.cuh"
#include <stdlib.h>

namespace nuslam
{

constexpr int kFastThreads = 32;                   // one warp = one filter in flight per CTA: no cross-warp state at all
#ifndef NUSLAM_FAST_SINGLE_STAGE
#define NUSLAM_FAST_SINGLE_STAGE 0   // 1: one staging buffer per CTA (input image -> exchange area -> output image): half the shared memory
#endif
constexpr bool kFastSingleStage = NUSLAM_FAST_SINGLE_STAGE != 0;
constexpr int kFastCtasPerSm = 16;   // 16 single-warp CTAs / SM at 128 registers (20 at 96 registers spill; measured slower)

// N > 0: the number of landmarks is a compile-time constant (the BASELINE sizes 12 and 6: every index folds). N < 0: a GENERIC
// instantiation for any n with ceil(2 n / 8) = -N fragment blocks per side (n read from the parameters at run time; n <= 4, 8, 12
// for -N = 1, 2, 3), so that FAST mode covers every map of up to 12 landmarks.
template <int N>
struct FastGeom
{
    static constexpr bool FIXED = N > 0;
    static constexpr int NB = FIXED ? (2 * N + 7) / 8 : -N;   // 8 x 8 fragment blocks per side of the landmark block
    static constexpr int NMAX = FIXED ? N : 4 * NB;           // most landmarks this instantiation serves
    static constexpr int LEN = 3 + 2 * NMAX;                  // (largest) state length
    static constexpr int SIG = LEN * LEN;
    static constexpr int TP = 8 * NB;         // padded landmark-block side
    static constexpr int VP = 3 + TP;         // padded vector length (state index space)
    static_assert(VP <= 32, "vector layout needs one lane per state index");
};

__device__ __forceinline__ void prefetch_l2_bulk(const void * src, uint32_t bytes)
{
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}

__device__ __forceinline__ uint32_t smem_u32(const void * p) { return (uint32_t) __cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t * bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t * bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t * bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// bulk async copies (TMA engine, no LSU wavefronts on the global side): global -> shared with mbarrier completion, shared -> global
__device__ __forceinline__ void bulk_g2s(void * dst_smem, const void * src_gmem, uint32_t bytes, uint64_t * bar)
{
    asm volatile("cp.async.bulk.shared::cta.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)), "l"(src_gmem),
                 "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_s2g(void * dst_gmem, const void * src_smem, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// D(8x8) += A(8x4) * B(4x8) on the fp64 tensor pipe; fragment layout in the header comment
__device__ __forceinline__ void dmma884(double & c0, double & c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// per-CTA (= per-warp) shared memory: exchange buffers between the fragment and the vector layout. Every vector has
// 32 + entries, one per lane; entries of lanes that own no state index stay zero.
template <int N>
struct __align__(16) FastSmem
{
    double2 kt[2][36];        // -Kt of the chunk's two updates, kt[s][i] = (-k0, -k1) of state index i < 32; DMMA A operand (slot
                              // stride 72 doubles = 8 (mod 16): the operand loads of the two slots hit disjoint banks)
    double2 wt[2][36];        // Wt of the chunk's two updates; DMMA B operand
    double rho[2][2][40];     // per chunk slot: landmark rows c, c+1 in vector layout, entry j at [j + 1] (index 3 is 16-byte aligned;
                              // row stride = 16 banks (mod 32): the two rows of a landmark are stored without bank conflicts)
    double2 kap[2][32];       // per chunk slot: landmark columns (c, c+1) interleaved, entry i
    double xs[34];            // state broadcast copy, x_i at [i + 1] (the pair (mx, my) is 16-byte aligned)
    double z[2 * kFastMMax];  // this step's measurements
};

#ifdef NUSLAM_TIMING
#define NUSLAM_T(k) { const long long now_ = clock64(); tacc[k] += now_ - tlast; tlast = now_; }
static __device__ long long g_fast_timing[16];
#else
#define NUSLAM_T(k)
#endif

// BULK: Sigma travels HBM <-> shared memory by bulk async copies (buffer A: the NEXT filter's image, prefetched while the
// current one is computed; buffer B: the exchange area during the updates, then the output image), so the global side costs
// no LSU wavefronts and no exposed latency; !BULK: plain per-lane loads / stores (any 8-byte aligned Sigma).
// ASSOC: unknown data association (p.ids == nullptr): every measurement is first associated on the device
// (ExtendedKalman::associateLandmark, slam_library.cpp:188-253: one candidate landmark per lane, Mahalanobis distance from the
// candidate's 5 x 5 block of Sigma, the reference's in-order early exit = lowest deciding lane) and applied at once (rank-2 pass
// per measurement instead of the lazy chunks). A measurement that opens a NEW landmark (or a singular innovation) hands the whole
// filter-step to the strict kernel: nothing has been written back yet, so it restarts from the state in HBM.
// The kernel and its launchers are instantiated in BOTH translation units (ekf_fast_api.cuh): relocatable in ekf_fast_tu.cu (known
// correspondence: the kernel launches the list kernel itself) and whole-program in nuslam_b200.cu (on-device association, where the
// relocatable build costs 3 registers and hand-overs to the list kernel are frequent). Internal linkage there keeps the two apart.
#ifdef NUSLAM_TU_FAST
#define NUSLAM_TU_LOCAL_BEGIN
#define NUSLAM_TU_LOCAL_END
#else
#define NUSLAM_TU_LOCAL_BEGIN namespace {
#define NUSLAM_TU_LOCAL_END }
#endif
NUSLAM_TU_LOCAL_BEGIN

template <int N, bool BULK, bool ASSOC>
__global__ void __launch_bounds__(kFastThreads, kFastCtasPerSm)
k_ekf_fast_step(const EkfParams p, const int do_predict, int32_t * __restrict__ worklist, int32_t * __restrict__ wl_count)
{
    using G = FastGeom<N>;
    constexpr int NB = G::NB;
    // sizes: compile-time constants in a fixed-N instantiation, read from the parameters in a generic one
    const int NL = G::FIXED ? G::NMAX : p.n;            // landmarks
    const int LEN = G::FIXED ? G::LEN : p.len;          // state length
    const int SIG = LEN * LEN;
    constexpr unsigned kFull = 0xffffffffu;
    constexpr int kImgMax = G::SIG * 8;                             // bytes of the largest Sigma this instantiation serves
    constexpr int kWinMax = ((kImgMax + 8 + 15) / 16) * 16;         // 16-byte aligned window that covers it at either alignment
    const int kWin = ((SIG * 8 + 8 + 15) / 16) * 16;
    constexpr int kStage = ((kWinMax > (int) sizeof(FastSmem<N>) ? kWinMax : (int) sizeof(FastSmem<N>)) + 127) / 128 * 128;
    constexpr int kStages = (BULK && !kFastSingleStage) ? 2 : 1;
    __shared__ __align__(128) unsigned char stage[kStages][kStage];
    __shared__ uint64_t full_bar;
    FastSmem<N> & f = *reinterpret_cast<FastSmem<N> *>(stage[kStages - 1]);
    const int lane = threadIdx.x;
    const int g = lane >> 2, t = lane & 3;
    const bool vlane = lane < LEN;      // lane owns a state index
    // zero the exchange buffers once (entries of lanes without a state index stay zero)
    for (int k = lane; k < (int) (sizeof(FastSmem<N>) / 8); k += 32) reinterpret_cast<double *>(&f)[k] = 0.0;
    __syncwarp();
#ifdef NUSLAM_TIMING
    long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long tlast = clock64();
#endif

    // issue the bulk load of filter `b` into buffer A (lane 0 only): the 16-byte aligned window around its Sigma
    auto issue_load = [&](int64_t b) {
        const unsigned char * g0 = reinterpret_cast<const unsigned char *>(p.sigma + b * SIG);
        const uintptr_t lo = reinterpret_cast<uintptr_t>(g0) & ~(uintptr_t) 15;
        uint32_t bytes = kWin;
        // never read past the end of the array: the last filter's window loses its tail, fetched separately below
        const uintptr_t end = reinterpret_cast<uintptr_t>(p.sigma + p.batch * SIG);
        if (lo + bytes > end) bytes = (uint32_t) ((end - lo) & ~(uintptr_t) 15);
        mbar_expect_tx(&full_bar, bytes);
        bulk_g2s(stage[0], reinterpret_cast<const void *>(lo), bytes, &full_bar);
    };
    uint32_t full_parity = 0;
    if (BULK)
    {
        if (lane == 0)
        {
            mbar_init(&full_bar, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            if ((int64_t) blockIdx.x < p.batch) issue_load(blockIdx.x);
        }
        __syncwarp();
    }

    for (int64_t bf = blockIdx.x; bf < p.batch; bf += gridDim.x)
    {
        // ---- load ----
        double C[NB][NB][2];
        double Rt = 0.0, Rx = 0.0, Ry = 0.0, Ct = 0.0, Cx = 0.0, Cy = 0.0, x = 0.0, diag = 0.0;
        // small inputs: plain loads, issued before anything waits
        if (vlane) x = p.x[bf * LEN + lane];
        const int st0 = p.status[bf], seen0 = p.seen[bf];
        // measurements of THIS filter (warp-uniform); ragged counts come with the fused scan step, i.e. with on-device association only
        const int m = (ASSOC && p.m_valid) ? min(p.m, max(0, p.m_valid[bf])) : p.m;
        const int my_id = (!ASSOC && lane < m) ? p.ids[bf * p.m + lane] : 0;
        const double my_z = (lane < 2 * m) ? p.z[bf * p.m * 2 + lane] : 0.0;
        const double my_tw = (do_predict && lane < 2) ? p.twists[bf * 3 + lane] : 0.0;
        if (BULK)
        {
            // image of this filter inside buffer A: offset 0 or 8 (its alignment in HBM)
            const double * img = reinterpret_cast<const double *>(stage[0] + (reinterpret_cast<uintptr_t>(p.sigma + bf * SIG) & 15));
            mbar_wait(&full_bar, full_parity);
            full_parity ^= 1;
            if (bf == p.batch - 1 && lane == 0 && ((reinterpret_cast<uintptr_t>(p.sigma + p.batch * SIG) & 15) != 0))
                const_cast<double *>(img)[SIG - 1] = p.sigma[bf * SIG + SIG - 1];   // tail the clamped window left out
            __syncwarp();
#pragma unroll
            for (int br = 0; br < NB; ++br)
#pragma unroll
                for (int bc = 0; bc < NB; ++bc)
#pragma unroll
                    for (int e = 0; e < 2; ++e)
                    {
                        const int row = 3 + 8 * br + g, col = 3 + 8 * bc + 2 * t + e;
                        C[br][bc][e] = (row < LEN && col < LEN) ? img[col * LEN + row] : 0.0;
                    }
            if (vlane)
            {
                Ct = img[lane];
                Cx = img[LEN + lane];
                Cy = img[2 * LEN + lane];
                Rt = img[lane * LEN];
                Rx = img[lane * LEN + 1];
                Ry = img[lane * LEN + 2];
                diag = img[lane * (LEN + 1)];   // Sigma(lane, lane): first-touch detection
            }
            __syncwarp();
            if (!kFastSingleStage)
            {
                // buffer A is free again: prefetch this CTA's next filter while the current one is computed
                if (lane == 0 && bf + gridDim.x < p.batch) issue_load(bf + gridDim.x);
            }
            else if (lane == 0 && bf + gridDim.x < p.batch)
            {
                // single buffer: it becomes the exchange area now; pull the next image towards L2 meanwhile
                const uintptr_t a0 = reinterpret_cast<uintptr_t>(p.sigma + (bf + gridDim.x) * SIG) & ~(uintptr_t) 15;
                prefetch_l2_bulk(reinterpret_cast<const void *>(a0), (uint32_t) ((sizeof(double) * SIG + 15) & ~15u));
            }
        }
        else
        {
            // pull this warp's next Sigma towards L2 while the current one is computed
            if (lane == 0 && bf + gridDim.x < p.batch)
            {
                const uintptr_t a0 = reinterpret_cast<uintptr_t>(p.sigma + (bf + gridDim.x) * SIG) & ~(uintptr_t) 15;
                prefetch_l2_bulk(reinterpret_cast<const void *>(a0), (uint32_t) ((sizeof(double) * SIG + 15) & ~15u));
            }
            const double * gs = p.sigma + bf * SIG;
#pragma unroll
            for (int br = 0; br < NB; ++br)
#pragma unroll
                for (int bc = 0; bc < NB; ++bc)
#pragma unroll
                    for (int e = 0; e < 2; ++e)
                    {
                        const int row = 3 + 8 * br + g, col = 3 + 8 * bc + 2 * t + e;
                        C[br][bc][e] = (row < LEN && col < LEN) ? __ldcs(gs + col * LEN + row) : 0.0;
                    }
            if (vlane)
            {
                Ct = __ldcs(gs + lane);
                Cx = __ldcs(gs + LEN + lane);
                Cy = __ldcs(gs + 2 * LEN + lane);
                Rt = __ldcs(gs + lane * LEN);
                Rx = __ldcs(gs + lane * LEN + 1);
                Ry = __ldcs(gs + lane * LEN + 2);
                diag = gs[lane * (LEN + 1)];
            }
        }
        // single staging buffer: whoever leaves this iteration must start the next image's copy (nothing is in flight otherwise)
        auto leave = [&]() {
            if (BULK && kFastSingleStage)
            {
                __syncwarp();
                if (lane == 0 && bf + gridDim.x < p.batch) issue_load(bf + gridDim.x);
            }
        };
        // ---- liveness ----
        if (st0 & (kStatusMapFull | kStatusSingular))   // the reference process died on an earlier scan
        {
            if (p.ids_out && lane < p.m) p.ids_out[bf * p.m + lane] = 0;
            if (p.x_snap && vlane) p.x_snap[bf * LEN + lane] = x;
            leave();
            continue;
        }
        if (ASSOC)
        {
            // an empty map: the first measurement opens landmark 1 (slam_library.cpp:196-200); a FULL map: associateLandmark writes
            // temp(3 + 2 seen) out of bounds and Armadillo throws before any candidate is examined (:204-207, SURVEY.md Appendix A-8).
            // Both belong to the strict kernel.
            if (m > 0 && (seen0 == 0 || 3 + 2 * seen0 >= LEN))
            {
                if (lane == 0) worklist[atomicAdd(wl_count, 1)] = (int32_t) bf;
                leave();
                continue;
            }
        }
        else
        {
            const bool idok = (unsigned) (my_id - 1) < (unsigned) NL;
            const int c = idok ? 1 + 2 * my_id : 3;
            const double d0 = __shfl_sync(kFull, diag, c), d1 = __shfl_sync(kFull, diag, c + 1);
            // first touch (INT_MAX prior) or initializeLandmark (slam.cpp:295-297): the strict kernel takes this filter-step
            const bool need = idok && ((do_predict && my_id > seen0) || d0 > kFirstTouchVariance || d1 > kFirstTouchVariance);
            if (__any_sync(kFull, need))
            {
                if (lane == 0) worklist[atomicAdd(wl_count, 1)] = (int32_t) bf;
                leave();
                continue;
            }
        }
        int status = st0;
        // ids_out of the slots this kernel does not associate: the given id (known correspondence), 0 past this filter's last measurement
        if (p.ids_out && lane < p.m && (!ASSOC || lane >= m)) p.ids_out[bf * p.m + lane] = (!ASSOC && my_id > 0) ? my_id : 0;
        if (BULK)
        {
            // buffer B held the previous filter's output image: wait until the bulk store has read it, then restore the zero
            // entries of the exchange vectors that belong to no state index
            if (lane == 0) bulk_wait_read();
            __syncwarp();
            if (lane >= LEN)
            {
#pragma unroll
                for (int s2 = 0; s2 < 2; ++s2)
                {
                    f.rho[s2][0][lane + 1] = 0.0;
                    f.rho[s2][1][lane + 1] = 0.0;
                    f.kap[s2][lane] = make_double2(0.0, 0.0);
                    f.kt[s2][lane] = make_double2(0.0, 0.0);
                    f.wt[s2][lane] = make_double2(0.0, 0.0);
                }
            }
        }
        // known correspondence: the m <= 16 ids as 4-bit codes (0 = no update in that slot) packed into two warp-uniform words by two
        // warp reductions; the update loop shifts them out, no memory round trip. An id above N is flagged here once (the flag is sticky).
        unsigned idlo = 0u, idhi = 0u;
        if (!ASSOC)
        {
            static_assert(G::NMAX <= 15 && kFastMMax <= 16, "4-bit id codes in two 32-bit words");
            const unsigned code = ((unsigned) (my_id - 1) < (unsigned) NL) ? (unsigned) my_id : 0u;
            idlo = __reduce_or_sync(kFull, lane < 8 ? code << (4 * lane) : 0u);
            idhi = __reduce_or_sync(kFull, (lane >= 8 && lane < 16) ? code << (4 * (lane - 8)) : 0u);
            if (__any_sync(kFull, my_id > NL)) status |= kStatusBadId;
        }
        unsigned idw = idlo;
        if (lane < 2 * m) f.z[lane] = my_z;
        // robot pose, replicated in every lane; lanes 0..2 own the same values in x (bit-identical updates)
        double th = __shfl_sync(kFull, x, 0), px = __shfl_sync(kFull, x, 1), py = __shfl_sync(kFull, x, 2);
        NUSLAM_T(0)

        // ---- predict (slam_library.cpp:65-108), oracle operation order, vector layout only ----
        if (do_predict)
        {
            const double dth = __shfl_sync(kFull, my_tw, 0), dxx = __shfl_sync(kFull, my_tw, 1);
            // predictEstimate :71-94, then the two Jacobian entries of getA :127-148 (theta read AFTER the motion update,
            // :129). sin/cos(theta + dth) of :84-85 and of :131 have the same argument: evaluated once.
            double s0, c0, b10, b20;
            sincos_fast(th, &s0, &c0);
            if (dth == 0.0)
            {
                px = add_(px, mul_(dxx, c0));
                py = add_(py, mul_(dxx, s0));
                th = add_(th, 0.0);
                b10 = mul_(-dxx, s0);
                b20 = mul_(dxx, c0);
            }
            else
            {
                const double q = div_fast(dxx, dth);
                // sin / cos of theta + dth and theta + 2 dth by the addition theorems from ONE sincos_fast(theta) and the
                // small-angle series of dth (the oracle calls libm three times; the difference is a few ulp, far inside the tolerance)
                double sd, cd;
                sincos_small(dth, &sd, &cd);
                const double s1 = fma(s0, cd, c0 * sd), c1 = fma(c0, cd, -s0 * sd);
                const double s3 = fma(s1, cd, c1 * sd), c3 = fma(c1, cd, -s1 * sd);
                px = add_(px, add_(mul_(-q, s0), mul_(q, s1)));
                py = add_(py, sub_(mul_(q, c0), mul_(q, c1)));
                th = add_(th, dth);
                b10 = add_(mul_(-q, c1), mul_(q, c3));
                b20 = add_(mul_(-q, s1), mul_(q, s3));
            }
            x = (lane == 0) ? th : (lane == 1) ? px : (lane == 2) ? py : x;
            // T = A * Sigma: rows x, y += b * row theta
            Rx = add_(mul_(b10, Rt), Rx);
            Ry = add_(mul_(b20, Rt), Ry);
            {
                const double t0 = __shfl_sync(kFull, Ct, 0), t1 = __shfl_sync(kFull, Cx, 0), t2 = __shfl_sync(kFull, Cy, 0);
                const double bb = (lane == 1) ? b10 : b20;
                if (lane == 1 || lane == 2)
                {
                    Ct = add_(mul_(bb, t0), Ct);
                    Cx = add_(mul_(bb, t1), Cx);
                    Cy = add_(mul_(bb, t2), Cy);
                }
            }
            // U = T * A.t(): columns x, y += column theta * b
            Cx = add_(mul_(Ct, b10), Cx);
            Cy = add_(mul_(Ct, b20), Cy);
            {
                const double t0 = __shfl_sync(kFull, Rt, 0), t1 = __shfl_sync(kFull, Rx, 0), t2 = __shfl_sync(kFull, Ry, 0);
                const double bb = (lane == 1) ? b10 : b20;
                if (lane == 1 || lane == 2)
                {
                    Rt = add_(mul_(t0, bb), Rt);
                    Rx = add_(mul_(t1, bb), Rx);
                    Ry = add_(mul_(t2, bb), Ry);
                }
            }
            // + Q_bar on the robot block (expanded_process_noise :110-125); Q is column-major
            if (lane < 3)
            {
                Rt = add_(Rt, p.Q[0 + 3 * lane]);
                Rx = add_(Rx, p.Q[1 + 3 * lane]);
                Ry = add_(Ry, p.Q[2 + 3 * lane]);
                Ct = add_(Ct, p.Q[lane + 3 * 0]);
                Cx = add_(Cx, p.Q[lane + 3 * 1]);
                Cy = add_(Cy, p.Q[lane + 3 * 2]);
            }
        }
        f.xs[lane + 1] = x;
        __syncwarp();
        NUSLAM_T(1)

        // ---- m sequential updates in chunks of 2 (slam.cpp:279-319, known correspondence) ----
        bool handed_over = false;
#pragma unroll 1
        for (int i0 = 0; i0 < m; i0 += (ASSOC ? 1 : 2))
        {
            int assoc_id = 0;
            if (ASSOC)
            {
                // ---- associateLandmark(z_i0): one candidate landmark per lane ----
                // exchange: the six robot vectors and the 2 x 2 diagonal blocks of the landmark block (slot 1 of the exchange
                // area is free in this mode: one measurement per pass)
                f.kt[1][lane] = make_double2(Rt, Rx);
                f.wt[1][lane] = make_double2(Ry, Ct);
                f.kap[1][lane] = make_double2(Cx, Cy);
                double2 * dg = reinterpret_cast<double2 *>(&f.rho[1][0][0]);
#pragma unroll
                for (int bb = 0; bb < NB; ++bb)
                    if (t == (g >> 1)) dg[8 * bb + g] = make_double2(C[bb][bb][0], C[bb][bb][1]);
                __syncwarp();
                const bool cand = lane < seen0;
                const int c = cand ? 3 + 2 * lane : 3;
                double Bm[5][5];   // Sigma at rows / columns (theta, x, y, c, c+1)
#pragma unroll
                for (int q = 0; q < 3; ++q)
                {
                    const double2 a = f.kt[1][q], b2 = f.wt[1][q];
                    Bm[0][q] = a.x;
                    Bm[1][q] = a.y;
                    Bm[2][q] = b2.x;
                }
#pragma unroll
                for (int e = 0; e < 2; ++e)
                {
                    const double2 a = f.kt[1][c + e], b2 = f.wt[1][c + e], c2 = f.kap[1][c + e];
                    Bm[0][3 + e] = a.x;    // Sigma(r, c+e) = entry c+e of the row vectors
                    Bm[1][3 + e] = a.y;
                    Bm[2][3 + e] = b2.x;
                    Bm[3 + e][0] = b2.y;   // Sigma(c+e, r) = entry c+e of the column vectors
                    Bm[3 + e][1] = c2.x;
                    Bm[3 + e][2] = c2.y;
                }
                {
                    const int tl = cand ? 2 * lane : 0;
                    const double2 d0 = dg[tl], d1 = dg[tl + 1];
                    Bm[3][3] = d0.x;
                    Bm[3][4] = d0.y;
                    Bm[4][3] = d1.x;
                    Bm[4][4] = d1.y;
                }
                const double2 mxy = *reinterpret_cast<const double2 *>(&f.xs[c + 1]);
                const double2 zz = *reinterpret_cast<const double2 *>(&f.z[2 * i0]);
                const double dx = mxy.x - px, dy = mxy.y - py;
                const double d = fma(dx, dx, dy * dy);
                // psi = Ht B Ht^T + R~ with the division-free rows h0 = (0, -dx, -dy, dx, dy), h1 = (-d, dy, -dx, -dy, dx): written out on the
                // rows' structure (differences of the landmark and robot entries first), 49 operations instead of the 70 FMAs of the dense
                // 5 x 5 products -- the same expressions the update uses for M
                double w0[5], w1[5];
#pragma unroll
                for (int q = 0; q < 5; ++q)
                {
                    const double e = Bm[3][q] - Bm[1][q], g2 = Bm[4][q] - Bm[2][q];
                    w0[q] = fma(dx, e, dy * g2);
                    w1[q] = fma(dx, g2, fma(-dy, e, -d * Bm[0][q]));
                }
                const double e0 = w0[3] - w0[1], f0 = w0[4] - w0[2], e1 = w1[3] - w1[1], f1 = w1[4] - w1[2];
                const double s00 = fma(dx, e0, dy * f0), s01 = fma(dx, f0, fma(-dy, e0, -d * w0[0]));
                const double s10 = fma(dx, e1, dy * f1), s11 = fma(dx, f1, fma(-dy, e1, -d * w1[0]));
                const double rs = rsqrt_1(d);
                double sq = d * rs;
                sq = fma(fma(-sq, sq, d), 0.5 * rs, sq);
                const double dsq = d * sq;
                const double m00 = fma(d, p.R[0], s00), m10 = fma(dsq, p.R[1], s10), m01 = fma(dsq, p.R[2], s01), m11 = fma(d * d, p.R[3], s11);
                const double det = fma(m00, m11, -m01 * m10);
                const double idet = rcp_fast(det);
                double zb = atan2_unit(dy, dx, rs) - th;
                    if (abs_ge_hi(zb, kHiPi)) zb = wrap_angle(zb);   // the identity inside [-pi, pi]
                const double n0 = sq * (zz.x - sq), n1 = d * (zz.y - zb);   // no angle wrap (:229-231)
                const double i00 = m11 * idet, i01 = -m01 * idet, i10 = -m10 * idet, i11 = m00 * idet;
                const double t0 = fma(n0, i00, n1 * i10), t1 = fma(n0, i01, n1 * i11);
                const double dist = fma(t0, n0, t1 * n1);   // (dz^T psi^-1) dz
                const bool sing = cand && abs_ge_hi(idet, kHi1e300);
                const unsigned m_sing = __ballot_sync(kFull, sing);
                const unsigned hitA = __ballot_sync(kFull, cand && !sing && (dist < p.amin));
                const unsigned hitB = __ballot_sync(kFull, cand && !sing && (dist > p.amin) && (dist < p.amax));
                const unsigned any = hitA | hitB | m_sing;
                if (any == 0u || ((m_sing >> (__ffs(any) - 1)) & 1u))
                {
                    // no candidate decides: a NEW landmark (initializeLandmark + first touch), or arma::inv would throw: strict kernel
                    handed_over = true;
                    break;
                }
                assoc_id = ((hitA >> (__ffs(any) - 1)) & 1u) ? __ffs(any) : -1;
                if (assoc_id > 0)
                {
                    // a landmark that is counted in `seen` but still carries the INT_MAX prior (set_state, or associate without update):
                    // its first touch belongs to the oracle-order kernel, exactly as with known correspondence
                    const double d0 = __shfl_sync(kFull, diag, 1 + 2 * assoc_id), d1 = __shfl_sync(kFull, diag, 2 + 2 * assoc_id);
                    if (d0 > kFirstTouchVariance || d1 > kFirstTouchVariance)
                    {
                        handed_over = true;
                        break;
                    }
                }
                if (p.ids_out && lane == 0) p.ids_out[bf * p.m + i0] = assoc_id;
                __syncwarp();
            }
            // (A) publish the chunk's landmark rows / columns from the (stale) fragments into vector layout
            int cc[2];
#pragma unroll
            for (int s = 0; s < 2; ++s)
            {
                int id;
                if (ASSOC)
                    id = (s == 0) ? assoc_id : 0;
                else
                {
                    if (s == 0 && i0 == 8) idw = idhi;
                    id = (int) (idw & 15u);
                    idw >>= 4;
                }
                const bool live = ASSOC ? ((unsigned) (id - 1) < (unsigned) NL) : (id != 0);   // warp-uniform
                cc[s] = live ? 1 + 2 * id : -1;
                if (live)
                {
                    const int c = cc[s];
                    const int tau = c - 3;
                    const int bsel = tau >> 3;
                    const bool rsel = (g >> 1) == ((tau & 7) >> 1);   // this lane holds row c or c+1
                    const bool csel = t == ((tau & 7) >> 1);          // this lane holds columns c, c+1
                    double * const rdst = &f.rho[s][g & 1][4 + 2 * t];
                    double2 * const cdst = &f.kap[s][3 + g];
#define NUSLAM_PUBLISH(b)                                                                                                  \
    if constexpr (NB > b)                                                                                                  \
    {                                                                                                                      \
        _Pragma("unroll") for (int q = 0; q < NB; ++q)                                                                     \
        {                                                                                                                  \
            if (rsel) *reinterpret_cast<double2 *>(rdst + 8 * q) = make_double2(C[b < NB ? b : 0][q][0], C[b < NB ? b : 0][q][1]); \
            if (csel) cdst[8 * q] = make_double2(C[q][b < NB ? b : 0][0], C[q][b < NB ? b : 0][1]);                        \
        }                                                                                                                  \
    }
                    if (bsel == 0)
                    {
                        NUSLAM_PUBLISH(0)
                    }
                    else if (bsel == 1)
                    {
                        NUSLAM_PUBLISH(1)
                    }
                    else if (bsel == 2)
                    {
                        NUSLAM_PUBLISH(2)
                    }
                    else
                    {
                        NUSLAM_PUBLISH(3)
                    }
#undef NUSLAM_PUBLISH
                    const int e = lane - c;
                    if (e == 0 || e == 1)
                    {
                        // robot part of row c+e: Sigma(c+e, {th,x,y}) is entry c+e of the column vectors; of column c+e: entry of the row vectors
                        f.rho[s][e][1] = Ct;
                        f.rho[s][e][2] = Cx;
                        f.rho[s][e][3] = Cy;
                        double * kd = reinterpret_cast<double *>(&f.kap[s][0]) + e;
                        kd[0] = Rt;
                        kd[2] = Rx;
                        kd[4] = Ry;
                    }
                }
            }
            __syncwarp();
            NUSLAM_T(2)
#pragma unroll
            for (int s = 0; s < 2; ++s)
            {
                bool done = false;
                if (cc[s] >= 0)   // warp-uniform (never true for slot 1 in ASSOC mode)
                {
                    const int c = cc[s];
                    // landmark rows c, c+1 (lane = column) and columns c, c+1 (lane = row)
                    double rho0 = f.rho[s][0][lane + 1], rho1 = f.rho[s][1][lane + 1];
                    const double2 kp = f.kap[s][lane];
                    double kap0 = kp.x, kap1 = kp.y;
                    const double2 mxy = *reinterpret_cast<const double2 *>(&f.xs[c + 1]);
                    const double2 zz = *reinterpret_cast<const double2 *>(&f.z[2 * (i0 + s)]);
                    if (s == 1)
                    {
                        // the fragments predate the chunk's first update: bring the four vectors up to date with it
                        const double2 ka = f.kt[0][c], kb = f.kt[0][c + 1], wa2 = f.wt[0][c], wb2 = f.wt[0][c + 1];
                        const double2 pW = f.wt[0][lane], pK = f.kt[0][lane];   // this lane's Wt and -Kt of the chunk's first update
                        rho0 = fma(ka.x, pW.x, fma(ka.y, pW.y, rho0));
                        rho1 = fma(kb.x, pW.x, fma(kb.y, pW.y, rho1));
                        kap0 = fma(pK.x, wa2.x, fma(pK.y, wa2.y, kap0));
                        kap1 = fma(pK.x, wb2.x, fma(pK.y, wb2.y, kap1));
                    }
                    // (B) Pt (row role) and Wt (column role) of this lane
                    const double dx = mxy.x - px, dy = mxy.y - py;
                    const double d = fma(dx, dx, dy * dy);
                    const double pa = kap0 - Cx, pb = kap1 - Cy;
                    const double wa = rho0 - Rx, wb = rho1 - Ry;
                    const double P0 = fma(dx, pa, dy * pb), P1 = fma(dx, pb, fma(-dy, pa, -d * Ct));
                    const double W0 = fma(dx, wa, dy * wb), W1 = fma(dx, wb, fma(-dy, wa, -d * Rt));
                    f.wt[s][lane] = make_double2(W0, W1);
                    __syncwarp();
                    NUSLAM_T(3)
                    // the 2 x 2 part, evaluated by every lane: M = Wt Ht^T + D^-1 R D^-1, Minv, innovation (:150-160, :272 no wrap)
                    const double2 g0 = f.wt[s][0], g1 = f.wt[s][1], g2 = f.wt[s][2], g3 = f.wt[s][c], g4 = f.wt[s][c + 1];
                    const double e0 = g3.x - g1.x, f0 = g4.x - g2.x, e1 = g3.y - g1.y, f1 = g4.y - g2.y;
                    const double s00 = fma(dx, e0, dy * f0), s01 = fma(dx, f0, fma(-dy, e0, -d * g0.x));
                    const double s10 = fma(dx, e1, dy * f1), s11 = fma(dx, f1, fma(-dy, e1, -d * g0.y));
                    const double rs = rsqrt_1(d);
                    double sq = d * rs;
                    sq = fma(fma(-sq, sq, d), 0.5 * rs, sq);   // sqrt(d) to ~1 ulp
                    const double dsq = d * sq;
                    const double m00 = fma(d, p.R[0], s00), m10 = fma(dsq, p.R[1], s10), m01 = fma(dsq, p.R[2], s01), m11 = fma(d * d, p.R[3], s11);
                    const double det = fma(m00, m11, -m01 * m10);
                    const double idet = rcp_fast(det);
                    // the bearing chain (atan2, wrap) is independent of the Minv chain: evaluated before the branch so that the two
                    // dependency chains interleave
                    double zb = atan2_unit(dy, dx, rs) - th;
                    if (abs_ge_hi(zb, kHiPi)) zb = wrap_angle(zb);   // the identity inside [-pi, pi]
                    const double n0 = sq * (zz.x - sq), n1 = d * (zz.y - zb);
                    if (!abs_ge_hi(idet, kHi1e300))   // |idet| < ~1e300: warp-uniform; false for det = 0, inf or nan, where arma::inv throws (slam_library.cpp:270)
                    {
                        done = true;
                        const double i00 = m11 * idet, i01 = -m01 * idet, i10 = -m10 * idet, i11 = m00 * idet;
                        // (C) -Kt = -Pt Minv, x += Kt n
                        const double nk0 = fma(-P0, i00, -P1 * i10), nk1 = fma(-P0, i01, -P1 * i11);
                        f.kt[s][lane] = make_double2(nk0, nk1);
                        __syncwarp();
                        NUSLAM_T(4)
                        const double2 k0 = f.kt[s][0], k1 = f.kt[s][1], k2 = f.kt[s][2];
                        // replicated pose: what lanes 0..2 compute for their own x, evaluated identically by every lane
                        th = fma(-k0.x, n0, fma(-k0.y, n1, th));
                        px = fma(-k1.x, n0, fma(-k1.y, n1, px));
                        py = fma(-k2.x, n0, fma(-k2.y, n1, py));
                        x = fma(-nk0, n0, fma(-nk1, n1, x));
                        if (abs_ge_hi(th, kHiPi)) th = wrap_angle(th);   // slam_library.cpp:275-276 (the identity inside [-pi, pi]); warp-uniform
                        if (lane == 0) x = th;
                        f.xs[lane + 1] = x;
                        // robot rows / columns: Sigma -= Kt Wt restricted to them
                        Rt = fma(k0.x, W0, fma(k0.y, W1, Rt));
                        Rx = fma(k1.x, W0, fma(k1.y, W1, Rx));
                        Ry = fma(k2.x, W0, fma(k2.y, W1, Ry));
                        Ct = fma(nk0, g0.x, fma(nk1, g0.y, Ct));
                        Cx = fma(nk0, g1.x, fma(nk1, g1.y, Cx));
                        Cy = fma(nk0, g2.x, fma(nk1, g2.y, Cy));
                        __syncwarp();
                        NUSLAM_T(5)
                    }
                    else
                        status |= kStatusSingular;
                }
                if (!done)
                {
                    // no measurement in this slot (or a singular one): it contributes nothing to the rank-4 pass
                    f.kt[s][lane] = make_double2(0.0, 0.0);
                    f.wt[s][lane] = make_double2(0.0, 0.0);
                    __syncwarp();
                }
            }
            // (D) one DMMA pass applies the chunk to the fragments: C += (-Kt) Wt, k = (u0, u1, v0, v1). Its operands live in a scope of
            // their own and die with the pass (without the scope the compiler allocates the NB = 1 instantiations' registers differently)
            {
                const double * ka = reinterpret_cast<const double *>(&f.kt[t >> 1][3 + g]) + (t & 1);
                const double * wa = reinterpret_cast<const double *>(&f.wt[t >> 1][3 + g]) + (t & 1);
                double a[NB], b[NB];
#pragma unroll
                for (int bb = 0; bb < NB; ++bb)
                {
                    a[bb] = ka[16 * bb];
                    b[bb] = wa[16 * bb];
                }
#pragma unroll
                for (int br = 0; br < NB; ++br)
#pragma unroll
                    for (int bc = 0; bc < NB; ++bc) dmma884(C[br][bc][0], C[br][bc][1], a[br], b[bc]);
            }
            __syncwarp();
            NUSLAM_T(6)
        }

        if (ASSOC && handed_over)
        {
            if (lane == 0) worklist[atomicAdd(wl_count, 1)] = (int32_t) bf;
            leave();
            continue;
        }
        // ---- write back ----
        if (BULK)
        {
            // registers -> output image in buffer B (the exchange data is dead) -> one bulk store of the 16-byte aligned interior
            // + one plain store of the edge element
            __syncwarp();
            double * gw = p.sigma + bf * SIG;
            const int odd = (int) ((reinterpret_cast<uintptr_t>(gw) >> 3) & 1);   // 1: HBM image starts 8 bytes past a 16-byte boundary
            double * img = reinterpret_cast<double *>(stage[kStages - 1]) + odd;
#pragma unroll
            for (int br = 0; br < NB; ++br)
#pragma unroll
                for (int bc = 0; bc < NB; ++bc)
#pragma unroll
                    for (int e = 0; e < 2; ++e)
                    {
                        const int row = 3 + 8 * br + g, col = 3 + 8 * bc + 2 * t + e;
                        if (row < LEN && col < LEN) img[col * LEN + row] = C[br][bc][e];
                    }
            if (vlane)
            {
                img[lane * LEN] = Rt;
                img[lane * LEN + 1] = Rx;
                img[lane * LEN + 2] = Ry;
                if (lane >= 3)
                {
                    img[lane] = Ct;
                    img[LEN + lane] = Cx;
                    img[2 * LEN + lane] = Cy;
                }
                p.x[bf * LEN + lane] = x;
                if (p.x_snap) p.x_snap[bf * LEN + lane] = x;
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0)
            {
                const int kInner = (SIG - 1) * 8;   // bytes of the aligned interior: SIG = (3 + 2n)^2 is odd, SIG - 1 elements = a multiple of 16 bytes
                static_assert((G::SIG & 1) == 1, "a filter's Sigma is an odd number of doubles");
                bulk_s2g(gw + odd, img + odd, kInner);
                const int edge = odd ? 0 : SIG - 1;
                gw[edge] = img[edge];
                if (status != st0) p.status[bf] = status;
                if (kFastSingleStage)
                {
                    // the buffer is reused for the next input image as soon as the store has read it
                    bulk_wait_read();
                    if (bf + gridDim.x < p.batch) issue_load(bf + gridDim.x);
                }
            }
        }
        else
        {
            double * gw = p.sigma + bf * SIG;
#pragma unroll
            for (int br = 0; br < NB; ++br)
#pragma unroll
                for (int bc = 0; bc < NB; ++bc)
#pragma unroll
                    for (int e = 0; e < 2; ++e)
                    {
                        const int row = 3 + 8 * br + g, col = 3 + 8 * bc + 2 * t + e;
                        if (row < LEN && col < LEN) __stcs(gw + col * LEN + row, C[br][bc][e]);
                    }
            if (vlane)
            {
                __stcs(gw + lane * LEN, Rt);
                __stcs(gw + lane * LEN + 1, Rx);
                __stcs(gw + lane * LEN + 2, Ry);
                if (lane >= 3)
                {
                    __stcs(gw + lane, Ct);
                    __stcs(gw + LEN + lane, Cx);
                    __stcs(gw + 2 * LEN + lane, Cy);
                }
                p.x[bf * LEN + lane] = x;
                if (p.x_snap) p.x_snap[bf * LEN + lane] = x;
            }
            if (lane == 0 && status != st0) p.status[bf] = status;
        }
        NUSLAM_T(7)
    }
    if (BULK && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // shared memory must outlive the last bulk store
    strict_tail(p, do_predict, worklist, wl_count, (int) gridDim.x, lane);
#ifdef NUSLAM_TIMING
    if (blockIdx.x == 0 && lane == 0)
        for (int k = 0; k < 8; ++k) atomicAdd((unsigned long long *) &g_fast_timing[k], (unsigned long long) tacc[k]);
#endif
}


template <int N>
int launch_fast_n(const EkfParams & p, bool do_predict, int sm_count, int32_t * worklist, int32_t * wl_count, cudaStream_t stream)
{
    // persistent: kFastCtasPerSm single-warp CTAs per SM, each striding over the filters
    int64_t blocks = p.batch;
    int ctas_per_sm = kFastCtasPerSm;
#ifdef NUSLAM_TIMING
    if (const char * e = getenv("NUSLAM_FAST_CTAS_PER_SM")) ctas_per_sm = atoi(e);
#endif
    if (blocks > ctas_per_sm * (int64_t) sm_count) blocks = ctas_per_sm * (int64_t) sm_count;
    static bool configured_dev[kMaxDevices] = {false};
    bool & configured = configured_dev[device_slot()];
    if (!configured)
    {
        // 16 CTAs x 11.8 KB of static shared memory per SM: ask for the largest shared-memory carve-out
        cudaFuncSetAttribute(k_ekf_fast_step<N, true, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        cudaFuncSetAttribute(k_ekf_fast_step<N, false, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        cudaFuncSetAttribute(k_ekf_fast_step<N, true, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        cudaFuncSetAttribute(k_ekf_fast_step<N, false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        configured = true;
    }
    const bool bulk = (reinterpret_cast<uintptr_t>(p.sigma) & 15) == 0;
    if (p.ids == nullptr)
    {
        if (bulk) k_ekf_fast_step<N, true, true><<<(unsigned) blocks, kFastThreads, 0, stream>>>(p, do_predict ? 1 : 0, worklist, wl_count);
        else k_ekf_fast_step<N, false, true><<<(unsigned) blocks, kFastThreads, 0, stream>>>(p, do_predict ? 1 : 0, worklist, wl_count);
    }
    else if (bulk)
        k_ekf_fast_step<N, true, false><<<(unsigned) blocks, kFastThreads, 0, stream>>>(p, do_predict ? 1 : 0, worklist, wl_count);
    else
        k_ekf_fast_step<N, false, false><<<(unsigned) blocks, kFastThreads, 0, stream>>>(p, do_predict ? 1 : 0, worklist, wl_count);
    return (int) cudaGetLastError();
}

// returns 0 on success, -1 when this configuration is not covered (caller falls back to the strict kernel), else a cudaError_t
inline int launch_fast(int n, const EkfParams & p, bool do_predict, int sm_count, int32_t * worklist, int32_t * wl_count, cudaStream_t stream)
{
    if (p.m > kFastMMax || p.m < 0) return -1;
    if (p.ids == nullptr && !do_predict) return -1;   // association belongs to the step protocol
    if (p.ids != nullptr && p.m_valid != nullptr) return -1;   // ragged measurement counts with known ids: strict kernel
    if ((reinterpret_cast<uintptr_t>(p.sigma) & 7) || (reinterpret_cast<uintptr_t>(p.x) & 7)) return -1;
    if (n == 12) return launch_fast_n<12>(p, do_predict, sm_count, worklist, wl_count, stream);
    if (n == 6) return launch_fast_n<6>(p, do_predict, sm_count, worklist, wl_count, stream);
    // any other map of up to 12 landmarks: the generic instantiation with the same number of fragment blocks
    if (n >= 1 && n <= 4) return launch_fast_n<-1>(p, do_predict, sm_count, worklist, wl_count, stream);
    if (n <= 8) return launch_fast_n<-2>(p, do_predict, sm_count, worklist, wl_count, stream);
    if (n <= 12) return launch_fast_n<-3>(p, do_predict, sm_count, worklist, wl_count, stream);
    return -1;
}

NUSLAM_TU_LOCAL_END

}   // namespace nuslam
