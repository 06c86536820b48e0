// ekf_res2.cuh -- FAST arithmetic, TWO filters per warp, both Sigma images RESIDENT IN SHARED MEMORY: fused predict + m sequential
// updates with known correspondence (the headline kernel of BASELINE.json configs[1]).
//
// Why two filters per warp (profiles/r02_kernel_iterations.md: what-if builds of the one-filter-per-warp predecessor of this kernel,
// measured on B200): the step is bound by the DISPATCH port of the four warp schedulers -- an fp64 instruction occupies it for two cycles
// (the pipe is 16 lanes wide), everything else for one: 116 fp64 + 195 other warp-instructions per update = 107 of the 150 cycles an update
// costs an SM, whatever the occupancy (12 ... 24 warps: 400 - 415 us) and whatever the shared-memory load (80 % or 66 % of the data pipe).
// HBM traffic is fully hidden (no traffic at all: 389 us). Half of those fp64 instructions are the per-filter scalar chain of an update
// (M, M^-1, sqrt d, atan2, innovation, pose), which every lane of the warp evaluates redundantly. So this kernel
//   * carries filters (2 pr, 2 pr + 1) in one warp: lane (h = lane / 16, q = lane % 16) serves filter h and owns state indices q and
//     16 + q (two vector slots). A scalar statement and every broadcast read is issued ONCE for both filters, each half-warp evaluating
//     its own filter's chain in the same instruction; a vector statement is issued once per slot, i.e. as often per filter as with one
//     filter per warp;
//   * keeps both Sigma images RESIDENT in shared memory (one bulk async copy of the 16-byte aligned 2 x 5 832 B pair in, one out, in
//     place), reads an update's landmark rows / columns straight from the image, delays the updates in chunks of CH and applies a chunk to
//     the landmark block in place on the fp64 tensor pipe (rank-2CH DMMA pass per filter). So no Sigma-sized state is in registers, and
//     two filters per warp do not cost 168 registers as they do when Sigma is held in register fragments (437 - 454 us, latency-starved);
//   * a 64-bit shared-memory access is processed per half-warp, i.e. per filter: both halves see the conflict-free patterns of the
//     one-filter kernel whatever their landmarks are.
// Per filter and update: ~67 fp64 + ~70 other warp-instructions instead of 116 + 195.
// The arithmetic of a filter is ekf_fast.cuh's statement for statement; a filter-step with a first touch / initializeLandmark is handed to
// the strict kernel (work list), and a dead filter or the missing twin of an odd batch keeps its image untouched.
// Reference: nuslam/src/slam_library.cpp:65-108 (predict), :263-282 (update), nuslam/src/slam.cpp:262-319 (caller protocol).
#pragma once
#include "ekf_fast.cuh"

namespace nuslam
{

#ifndef NUSLAM_RES2_CH
#define NUSLAM_RES2_CH 3        // updates per delayed chunk (2, 3 or 4)
#endif
#ifndef NUSLAM_RES2_CTAS
#define NUSLAM_RES2_CTAS (NUSLAM_RES2_CH == 2 ? 12 : NUSLAM_RES2_CH == 3 ? 12 : 11)
#endif
#ifndef NUSLAM_RES2_EXP
#define NUSLAM_RES2_EXP 0       // timing what-ifs (WRONG results): 1 no in-place pass, 2 no atan2, 3 no pending corrections, 5 no updates at all,
#endif                          // 8 in-place pass without its DMMAs
constexpr int kRes2CtasPerSm = NUSLAM_RES2_CTAS;   // one warp (= one pair in flight) per CTA

template <int CH>
struct __align__(16) Res2Smem
{
    // slot stride 28 double2 = 56 doubles = 8 (mod 16): the operand loads of two slots hit disjoint banks; the lanes that own no state
    // index store nothing
    double2 kt[2][CH][28];        // per filter: -Kt of the chunk's updates (DMMA A operand, pending corrections)
    double2 wt[2][CH][28];        // per filter: Wt of the chunk's updates (DMMA B operand)
    double z[2][2 * kFastMMax];   // per filter: this step's measurements
    unsigned slots_of[2][16];     // per filter: landmark (1-based) -> bit mask of this step's measurement slots that carry it
};

template <int N, int CH>
__global__ void __launch_bounds__(32, kRes2CtasPerSm)
k_ekf_res2_step(const EkfParams p, const int do_predict, int32_t * __restrict__ worklist, int32_t * __restrict__ wl_count)
{
    using G = FastGeom<N>;
    static_assert(G::FIXED && 2 * N == 8 * G::NB && G::LEN > 16 && G::LEN <= 32, "pair layout: two slots of 16 state indices, unpadded 8 x 8 tiles");
    static_assert(CH >= 2 && CH <= 4, "chunks of 2, 3 or 4 updates");
    constexpr int KS = (CH + 1) / 2;   // DMMA k-steps of a chunk's pass (an odd chunk leaves half of the last one empty)
    constexpr int NB = G::NB, NL = N, LEN = G::LEN, SIG = G::SIG;
    static_assert(NB == 3, "row permutation written for three row blocks");
    constexpr unsigned kFull = 0xffffffffu;
    constexpr int kImg = SIG * 8, kPairBytes = 2 * kImg;   // a pair is 16-byte aligned in HBM whenever the array is
    // one warp per CTA: [the pair's two images][exchange area][mbarrier]
    extern __shared__ __align__(128) unsigned char res2_dyn[];
    static_assert(kPairBytes % 16 == 0 && sizeof(Res2Smem<CH>) % 16 == 0, "16-byte aligned pieces");
    unsigned char * const stage = res2_dyn;
    Res2Smem<CH> & f = *reinterpret_cast<Res2Smem<CH> *>(stage + kPairBytes);
    uint64_t & full_bar = *reinterpret_cast<uint64_t *>(stage + kPairBytes + sizeof(Res2Smem<CH>));
    const int lane = threadIdx.x & 31;
    const int64_t gw0 = blockIdx.x, gwn = gridDim.x;   // this warp, all warps
    const int h = lane >> 4, q = lane & 15;   // vector / scalar domain: filter of this lane, index inside the half
    const int hb = 16 * h;                    // first lane of this half
    const int g = lane >> 2, t = lane & 3;    // tile domain of the in-place pass
    double * const img = reinterpret_cast<double *>(stage) + h * SIG;   // this lane's filter
    double2(*const ktH)[28] = f.kt[h];
    double2(*const wtH)[28] = f.wt[h];
    // state indices of this lane's two slots; a slot without a state entry re-reads what lanes q = 0..4 read for slot 1 (same address
    // inside the half-warp = broadcast: no bank conflict, no access outside the image); its results are never used
    const bool v1 = 16 + q < LEN;
    const int i1 = v1 ? 16 + q : 5 + q;
    const int rrow0 = 3 + (g & 1) + 8 * ((g >> 1) & 1) + 2 * (g >> 2);
    int rrow[NB];
#pragma unroll
    for (int a = 0; a < NB; ++a) rrow[a] = (a + 1 < NB) ? rrow0 + 4 * a : 3 + 8 * a + g;
    const int64_t npairs = (p.batch + 1) >> 1;
    const int m = p.m;

    auto issue_load = [&](int64_t pr) {   // lane 0 only
        const unsigned char * src = reinterpret_cast<const unsigned char *>(p.sigma + 2 * pr * SIG);
        // the last pair of an odd batch holds one filter: its 16-byte aligned part, the tail element is fetched separately
        const uint32_t bytes = (2 * pr + 1 < p.batch) ? (uint32_t) kPairBytes : (uint32_t) (kImg & ~15);
        mbar_expect_tx(&full_bar, bytes);
        bulk_g2s(stage, src, bytes, &full_bar);
    };
    uint32_t full_parity = 0;
    if (lane == 0)
    {
        mbar_init(&full_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (gw0 < npairs) issue_load(gw0);
    }
    __syncwarp();

    // the small inputs of a pair, carried one iteration ahead
    double nx0 = 0.0, nx1 = 0.0, nz0 = 0.0, nz1 = 0.0, ntw = 0.0;
    int nst = 0, nseen = 0, nid = 0;
    auto load_small = [&](int64_t pr) {
        const int64_t bfn = 2 * pr + h;
        const int64_t b = bfn < p.batch ? bfn : 2 * pr;   // safe addressing for the missing twin of an odd batch
        nx0 = p.x[b * LEN + q];
        nx1 = v1 ? p.x[b * LEN + 16 + q] : 0.0;
        nst = p.status[b];
        nseen = p.seen[b];
        nid = (q < m) ? p.ids[b * m + q] : 0;
        nz0 = (q < m) ? p.z[b * m * 2 + 2 * q] : 0.0;
        nz1 = (q < m) ? p.z[b * m * 2 + 2 * q + 1] : 0.0;
        ntw = (do_predict && q < 2) ? p.twists[b * 3 + q] : 0.0;
    };
    if (gw0 < npairs) load_small(gw0);
    for (int64_t pr = gw0; pr < npairs; pr += gwn)
    {
        const int64_t bf = 2 * pr + h;
        const bool has = bf < p.batch;
        const bool next = pr + gwn < npairs;
        // ---- small inputs: loaded one pair ahead (the loads of the next pair are in flight while this one is computed) ----
        double x[2] = {nx0, nx1};
        const int st0 = nst, seen0 = nseen, my_id = nid;
        const double my_z0 = nz0, my_z1 = nz1, my_tw = ntw;
        if (next) load_small(pr + gwn);
        // robot pose of this lane's filter, replicated over its half; lanes q = 0..2 own the same values in x[0]
        double th = __shfl_sync(kFull, x[0], hb), px = __shfl_sync(kFull, x[0], hb + 1), py = __shfl_sync(kFull, x[0], hb + 2);

        // ---- predict, scalar part (slam_library.cpp:71-94, :127-148): needs the state and the twist only -- evaluated while the bulk copy
        //      of the images is still in flight ----
        double b10 = 0.0, b20 = 0.0;
        const double x0_in = x[0];   // a dead filter's snapshot is the state as it came
        if (do_predict)
        {
            const double dth = __shfl_sync(kFull, my_tw, hb), dxx = __shfl_sync(kFull, my_tw, hb + 1);
            double s0, c0;
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
                const double qq = div_fast(dxx, dth);
                double sd, cd;
                sincos_small(dth, &sd, &cd);
                const double s1 = fma(s0, cd, c0 * sd), c1 = fma(c0, cd, -s0 * sd);
                const double s3 = fma(s1, cd, c1 * sd), c3 = fma(c1, cd, -s1 * sd);
                px = add_(px, add_(mul_(-qq, s0), mul_(qq, s1)));
                py = add_(py, sub_(mul_(qq, c0), mul_(qq, c1)));
                th = add_(th, dth);
                b10 = add_(mul_(-qq, c1), mul_(qq, c3));
                b20 = add_(mul_(-qq, s1), mul_(qq, s3));
            }
            x[0] = (q == 0) ? th : (q == 1) ? px : (q == 2) ? py : x[0];
        }
        mbar_wait(&full_bar, full_parity);
        full_parity ^= 1;
        if (2 * pr + 1 >= p.batch && lane == 0) reinterpret_cast<double *>(stage)[SIG - 1] = p.sigma[2 * pr * SIG + SIG - 1];
        __syncwarp();
        auto leave = [&]() {   // nothing is stored: the buffer is free at once
            __syncwarp();
            if (lane == 0 && next) issue_load(pr + gwn);
        };
        // ---- liveness, first touch ----
        const bool idok = (unsigned) (my_id - 1) < (unsigned) NL;
        bool need;
        {
            const int c = idok ? 1 + 2 * my_id : 3;
            const double d0 = img[c * (LEN + 1)], d1 = img[(c + 1) * (LEN + 1)];
            // first touch (INT_MAX prior) or initializeLandmark (slam.cpp:295-297): the strict kernel takes this filter-step
            need = has && idok && ((do_predict && my_id > seen0) || d0 > kFirstTouchVariance || d1 > kFirstTouchVariance);
        }
        const unsigned need_w = __ballot_sync(kFull, need);
        const unsigned bad_w = __ballot_sync(kFull, q < m && my_id > NL);
        const bool stat_dead = (st0 & (kStatusMapFull | kStatusSingular)) != 0;   // the reference process died on an earlier scan
        const bool to_strict = has && !stat_dead && ((need_w >> hb) & 0xffffu) != 0u;
        const bool dead = !has || stat_dead || to_strict;
        if (has && stat_dead)
        {
            if (p.ids_out && q < m) p.ids_out[bf * m + q] = 0;
            if (p.x_snap)
            {
                p.x_snap[bf * LEN + q] = x0_in;
                if (v1) p.x_snap[bf * LEN + 16 + q] = x[1];
            }
        }
        else if (to_strict && q == 0)
            worklist[atomicAdd(wl_count, 1)] = (int32_t) bf;
        const unsigned dead_w = __ballot_sync(kFull, dead);
        const bool deadA = (dead_w & 1u) != 0u, deadB = (dead_w & 0x10000u) != 0u;
        if (deadA && deadB)
        {
            leave();
            continue;
        }
        int status = st0;
        if (!dead)
        {
            if (p.ids_out && q < m) p.ids_out[bf * m + q] = my_id > 0 ? my_id : 0;
            if ((bad_w >> hb) & 0xffffu) status |= kStatusBadId;
        }
        const int code = (idok && !dead) ? my_id : 0;   // 0: no update in this slot (a dead filter has none at all)
        // this lane's slot as the state index of its landmark (-1: none), and -- once per step -- in which slots the landmarks of this
        // lane's two state indices are measured (index i >= 3 belongs to landmark (i - 1) / 2): the chunk loop then neither decodes ids nor
        // compares indices
        const int cval = code ? 1 + 2 * code : -1;
        f.slots_of[h][q] = 0u;
        __syncwarp();
        if (code) atomicOr(&f.slots_of[h][code], 1u << q);
        if (q < m) *reinterpret_cast<double2 *>(&f.z[h][2 * q]) = make_double2(my_z0, my_z1);
        __syncwarp();
        const unsigned hit0 = (q >= 3) ? f.slots_of[h][(q - 1) >> 1] : 0u;
        const unsigned hit1 = v1 ? f.slots_of[h][(15 + q) >> 1] : 0u;
        // the state-only part of an update: landmark position from the lanes that own it, sqrt d, bearing, innovation (:150-160, :272 no wrap)
        struct StateChain { double dx, dy, d, dsq, n0, n1; };
        auto state_chain = [&](const int c, const int slot) {
            const double xa = (c >= 16) ? x[1] : x[0], xb = (c + 1 >= 16) ? x[1] : x[0];
            const double mxv = __shfl_sync(kFull, xa, hb + (c & 15)), myv = __shfl_sync(kFull, xb, hb + ((c + 1) & 15));
            const double2 zz = *reinterpret_cast<const double2 *>(&f.z[h][2 * (slot & 15)]);
            StateChain o;
            o.dx = mxv - px, o.dy = myv - py;
            o.d = fma(o.dx, o.dx, o.dy * o.dy);
            const double rs = rsqrt_1(o.d);
            double sq = o.d * rs;
            sq = fma(fma(-sq, sq, o.d), 0.5 * rs, sq);   // sqrt(d) to ~1 ulp
            o.dsq = o.d * sq;
#if NUSLAM_RES2_EXP == 2
            double zb = o.dy * rs - th;
#else
            double zb = atan2_unit(o.dy, o.dx, rs) - th;
#endif
            zb = wrap_angle(zb);   // the identity inside [-pi, pi]; branch-free: the update stays ONE basic block, so that the
                                   // state-only chain (rsqrt, atan2) and the covariance chain interleave
            o.n0 = sq * (zz.x - sq), o.n1 = o.d * (zz.y - zb);
            return o;
        };
        // this half's landmark column of a measurement slot (-1: none); a half without a measurement computes on a safe index
        auto col_of_slot = [&](const int slot) {
            const int cv = __shfl_sync(kFull, cval, hb + (slot & 15));
            return (slot < kFastMMax) ? cv : -1;
        };
        // ---- robot rows / columns: image -> registers (vector layout, two slots) ----
        double Ct[2], Cx[2], Cy[2], Rt[2], Rx[2], Ry[2];
        Ct[0] = img[q], Cx[0] = img[LEN + q], Cy[0] = img[2 * LEN + q];
        Rt[0] = img[q * LEN], Rx[0] = img[q * LEN + 1], Ry[0] = img[q * LEN + 2];
        Ct[1] = img[i1], Cx[1] = img[LEN + i1], Cy[1] = img[2 * LEN + i1];
        Rt[1] = img[i1 * LEN], Rx[1] = img[i1 * LEN + 1], Ry[1] = img[i1 * LEN + 2];
        // ---- predict, covariance part (slam_library.cpp:96-108), oracle operation order, vector layout only ----
        if (do_predict)
        {
            // T = A * Sigma: rows x, y += b * row theta
#pragma unroll
            for (int sl = 0; sl < 2; ++sl)
            {
                Rx[sl] = add_(mul_(b10, Rt[sl]), Rx[sl]);
                Ry[sl] = add_(mul_(b20, Rt[sl]), Ry[sl]);
            }
            {
                const double t0 = __shfl_sync(kFull, Ct[0], hb), t1 = __shfl_sync(kFull, Cx[0], hb), t2 = __shfl_sync(kFull, Cy[0], hb);
                const double bb = (q == 1) ? b10 : b20;
                if (q == 1 || q == 2)
                {
                    Ct[0] = add_(mul_(bb, t0), Ct[0]);
                    Cx[0] = add_(mul_(bb, t1), Cx[0]);
                    Cy[0] = add_(mul_(bb, t2), Cy[0]);
                }
            }
            // U = T * A.t(): columns x, y += column theta * b
#pragma unroll
            for (int sl = 0; sl < 2; ++sl)
            {
                Cx[sl] = add_(mul_(Ct[sl], b10), Cx[sl]);
                Cy[sl] = add_(mul_(Ct[sl], b20), Cy[sl]);
            }
            {
                const double t0 = __shfl_sync(kFull, Rt[0], hb), t1 = __shfl_sync(kFull, Rx[0], hb), t2 = __shfl_sync(kFull, Ry[0], hb);
                const double bb = (q == 1) ? b10 : b20;
                if (q == 1 || q == 2)
                {
                    Rt[0] = add_(mul_(t0, bb), Rt[0]);
                    Rx[0] = add_(mul_(t1, bb), Rx[0]);
                    Ry[0] = add_(mul_(t2, bb), Ry[0]);
                }
            }
            // + Q_bar on the robot block (expanded_process_noise :110-125); Q is column-major
            if (q < 3)
            {
                Rt[0] = add_(Rt[0], p.Q[0 + 3 * q]);
                Rx[0] = add_(Rx[0], p.Q[1 + 3 * q]);
                Ry[0] = add_(Ry[0], p.Q[2 + 3 * q]);
                Ct[0] = add_(Ct[0], p.Q[q + 3 * 0]);
                Cx[0] = add_(Cx[0], p.Q[q + 3 * 1]);
                Cy[0] = add_(Cy[0], p.Q[q + 3 * 2]);
            }
        }
        const double r00c = p.R[0], r10c = p.R[1], r01c = p.R[2], r11c = p.R[3];

        // ---- m sequential updates in delayed chunks of CH (slam.cpp:279-319, known correspondence) ----
#pragma unroll 1
        for (int i0 = 0; i0 < (NUSLAM_RES2_EXP == 5 ? 0 : m); i0 += CH)
        {
            int cc[CH];
#pragma unroll
            for (int s = 0; s < CH; ++s)
            {
                cc[s] = col_of_slot(i0 + s);   // this half's landmark column of slot i0 + s; -1: no measurement in this slot of this filter
            }
            const unsigned chunk_bits = ((1u << CH) - 1u) << i0;
            const bool mine0 = (hit0 & chunk_bits) != 0u, mine1 = (hit1 & chunk_bits) != 0u;
            // the image's robot rows / columns are stale (they live in registers): refresh the entries this chunk's landmarks read
            if (mine0)
            {
                img[q] = Ct[0], img[LEN + q] = Cx[0], img[2 * LEN + q] = Cy[0];
                img[q * LEN] = Rt[0], img[q * LEN + 1] = Rx[0], img[q * LEN + 2] = Ry[0];
            }
            if (mine1 && v1)
            {
                img[i1] = Ct[1], img[LEN + i1] = Cx[1], img[2 * LEN + i1] = Cy[1];
                img[i1 * LEN] = Rt[1], img[i1 * LEN + 1] = Rx[1], img[i1 * LEN + 2] = Ry[1];
            }
            __syncwarp();
            double pK0[CH - 1][2], pK1[CH - 1][2], pW0[CH - 1][2], pW1[CH - 1][2];   // this lane's -Kt / Wt of the chunk's earlier updates
#pragma unroll
            for (int s = 0; s < CH; ++s)
            {
                const bool live = cc[s] >= 0;
                double W0[2] = {0.0, 0.0}, W1[2] = {0.0, 0.0}, nk0[2] = {0.0, 0.0}, nk1[2] = {0.0, 0.0};
                if (__any_sync(kFull, live))
                {
                    const int c = live ? cc[s] : 3;   // a half without a measurement in this slot computes on a safe index and drops the result
                    // ---- state-only part: sqrt d, bearing, innovation (:150-160, :272 no wrap) ----
                    const StateChain sc = state_chain(c, i0 + s);
                    const double dx = sc.dx, dy = sc.dy, d = sc.d, dsq = sc.dsq;
                    double n0 = sc.n0, n1 = sc.n1;
                    // ---- landmark rows c, c+1 (lane = column) and columns c, c+1 (lane = row) as of the chunk's start, from the image;
                    //      brought up to date with the chunk's earlier updates (delayed-update algebra); Pt / Wt of this lane's slots ----
                    double rho0[2], rho1[2], kap0[2], kap1[2];
                    rho0[0] = img[q * LEN + c], rho1[0] = img[q * LEN + c + 1];
                    kap0[0] = img[c * LEN + q], kap1[0] = img[(c + 1) * LEN + q];
                    rho0[1] = img[i1 * LEN + c], rho1[1] = img[i1 * LEN + c + 1];
                    kap0[1] = img[c * LEN + i1], kap1[1] = img[(c + 1) * LEN + i1];
#pragma unroll
                    for (int u = 0; u < (NUSLAM_RES2_EXP == 3 ? 0 : s); ++u)
                    {
                        const double2 ka = ktH[u][c], kb = ktH[u][c + 1], wa2 = wtH[u][c], wb2 = wtH[u][c + 1];
#pragma unroll
                        for (int sl = 0; sl < 2; ++sl)
                        {
                            rho0[sl] = fma(ka.x, pW0[u][sl], fma(ka.y, pW1[u][sl], rho0[sl]));
                            rho1[sl] = fma(kb.x, pW0[u][sl], fma(kb.y, pW1[u][sl], rho1[sl]));
                            kap0[sl] = fma(pK0[u][sl], wa2.x, fma(pK1[u][sl], wa2.y, kap0[sl]));
                            kap1[sl] = fma(pK0[u][sl], wb2.x, fma(pK1[u][sl], wb2.y, kap1[sl]));
                        }
                    }
                    double P0[2], P1[2];
#pragma unroll
                    for (int sl = 0; sl < 2; ++sl)
                    {
                        const double pa = kap0[sl] - Cx[sl], pb = kap1[sl] - Cy[sl];
                        const double wa = rho0[sl] - Rx[sl], wb = rho1[sl] - Ry[sl];
                        P0[sl] = fma(dx, pa, dy * pb);
                        P1[sl] = fma(dx, pb, fma(-dy, pa, -d * Ct[sl]));
                        W0[sl] = fma(dx, wa, dy * wb);
                        W1[sl] = fma(dx, wb, fma(-dy, wa, -d * Rt[sl]));
                    }
                    wtH[s][q] = make_double2(W0[0], W1[0]);
                    if (v1) wtH[s][16 + q] = make_double2(W0[1], W1[1]);
                    __syncwarp();
                    // ---- the 2 x 2 part of this lane's filter: M = Wt Ht^T + D^-1 R D^-1, Minv ----
                    const double2 g0 = wtH[s][0], g1 = wtH[s][1], g2 = wtH[s][2], g3 = wtH[s][c], g4 = wtH[s][c + 1];
                    const double e0 = g3.x - g1.x, f0 = g4.x - g2.x, e1 = g3.y - g1.y, f1 = g4.y - g2.y;
                    const double s00 = fma(dx, e0, dy * f0), s01 = fma(dx, f0, fma(-dy, e0, -d * g0.x));
                    const double s10 = fma(dx, e1, dy * f1), s11 = fma(dx, f1, fma(-dy, e1, -d * g0.y));
                    const double m00 = fma(d, r00c, s00), m10 = fma(dsq, r10c, s10), m01 = fma(dsq, r01c, s01), m11 = fma(d * d, r11c, s11);
                    const double det = fma(m00, m11, -m01 * m10);
                    const double idet = rcp_fast(det);
                    // |idet| < ~1e300: false for det = 0, inf or nan, where arma::inv throws (slam_library.cpp:270)
                    const bool ok = live && !abs_ge_hi(idet, kHi1e300);
                    const double i00 = m11 * idet, i01 = -m01 * idet, i10 = -m10 * idet, i11 = m00 * idet;
                    // (C) -Kt = -Pt Minv
#pragma unroll
                    for (int sl = 0; sl < 2; ++sl)
                    {
                        nk0[sl] = fma(-P0[sl], i00, -P1[sl] * i10);
                        nk1[sl] = fma(-P0[sl], i01, -P1[sl] * i11);
                    }
                    if (!__all_sync(kFull, ok))
                    {
                        // a filter without a measurement in this slot (or with a singular one): its update is the identity
                        if (!ok)
                        {
                            if (live) status |= kStatusSingular;
                            n0 = 0.0;
                            n1 = 0.0;
#pragma unroll
                            for (int sl = 0; sl < 2; ++sl) nk0[sl] = nk1[sl] = W0[sl] = W1[sl] = 0.0;
                            wtH[s][q] = make_double2(0.0, 0.0);
                            if (v1) wtH[s][16 + q] = make_double2(0.0, 0.0);
                        }
                    }
                    ktH[s][q] = make_double2(nk0[0], nk1[0]);
                    if (v1) ktH[s][16 + q] = make_double2(nk0[1], nk1[1]);
#pragma unroll
                    for (int sl = 0; sl < 2; ++sl)
                    {
                        // robot columns: Sigma -= Kt Wt restricted to them; state
                        Ct[sl] = fma(nk0[sl], g0.x, fma(nk1[sl], g0.y, Ct[sl]));
                        Cx[sl] = fma(nk0[sl], g1.x, fma(nk1[sl], g1.y, Cx[sl]));
                        Cy[sl] = fma(nk0[sl], g2.x, fma(nk1[sl], g2.y, Cy[sl]));
                        x[sl] = fma(-nk0[sl], n0, fma(-nk1[sl], n1, x[sl]));
                    }
                    __syncwarp();
                    const double2 k0 = ktH[s][0], k1 = ktH[s][1], k2 = ktH[s][2];
                    // replicated pose: what lanes q = 0..2 compute for their own x, evaluated identically by the whole half
                    th = fma(-k0.x, n0, fma(-k0.y, n1, th));
                    px = fma(-k1.x, n0, fma(-k1.y, n1, px));
                    py = fma(-k2.x, n0, fma(-k2.y, n1, py));
                    // slam_library.cpp:275-276 (the identity inside [-pi, pi]), only where this filter had the update: a half with no
                    // measurement in this slot (its partner has one) keeps a heading that predict carried outside [-pi, pi], as the
                    // reference does; wrapping it anyway made the state depend on the partner filter
                    if (ok) th = wrap_angle(th);
                    if (q == 0) x[0] = th;
#pragma unroll
                    for (int sl = 0; sl < 2; ++sl)
                    {
                        // robot rows: Sigma -= Kt Wt restricted to them
                        Rt[sl] = fma(k0.x, W0[sl], fma(k0.y, W1[sl], Rt[sl]));
                        Rx[sl] = fma(k1.x, W0[sl], fma(k1.y, W1[sl], Rx[sl]));
                        Ry[sl] = fma(k2.x, W0[sl], fma(k2.y, W1[sl], Ry[sl]));
                    }
                }
                else
                {
                    // no filter of the pair has a measurement in this slot: it contributes nothing to the pass or to later corrections
                    ktH[s][q] = make_double2(0.0, 0.0);
                    if (v1) ktH[s][16 + q] = make_double2(0.0, 0.0);
                    wtH[s][q] = make_double2(0.0, 0.0);
                    if (v1) wtH[s][16 + q] = make_double2(0.0, 0.0);
                }
                if (s + 1 < CH)
                {
#pragma unroll
                    for (int sl = 0; sl < 2; ++sl)
                    {
                        pK0[s < CH - 1 ? s : 0][sl] = nk0[sl];
                        pK1[s < CH - 1 ? s : 0][sl] = nk1[sl];
                        pW0[s < CH - 1 ? s : 0][sl] = W0[sl];
                        pW1[s < CH - 1 ? s : 0][sl] = W1[sl];
                    }
                    __syncwarp();   // later slots read this slot's Kt / Wt at their landmark's indices
                }
            }
            // (D) one pass per filter applies the chunk to the landmark block of its image in place: tile += (-Kt) Wt
            __syncwarp();
#pragma unroll
            for (int ff = 0; ff < 2; ++ff)
            {
                if (NUSLAM_RES2_EXP != 1 && (ff == 0 ? !deadA : !deadB))   // warp-uniform
                {
                    const double * const ka = reinterpret_cast<const double *>(&f.kt[ff][t >> 1][0]) + (t & 1);
                    const double * const wa = reinterpret_cast<const double *>(&f.wt[ff][t >> 1][3 + g]) + (t & 1);
                    double a[KS][NB], b[KS][NB];
#pragma unroll
                    for (int kk = 0; kk < KS; ++kk)
#pragma unroll
                        for (int bb = 0; bb < NB; ++bb)
                        {
                            const bool used = 2 * kk + 1 < CH || t < 2;   // slot 2 kk + (t >> 1) exists
                            a[kk][bb] = used ? ka[kk * 112 + 2 * rrow[bb]] : 0.0;
                            b[kk][bb] = used ? wa[kk * 112 + 16 * bb] : 0.0;
                        }
                    double * const tbase = reinterpret_cast<double *>(stage) + ff * SIG + (3 + 2 * t) * LEN;
                    double c0[NB][NB], c1[NB][NB];
#pragma unroll
                    for (int bc = 0; bc < NB; ++bc)
#pragma unroll
                        for (int br = 0; br < NB; ++br)
                        {
                            const double * const e0p = tbase + bc * (8 * LEN) + rrow[br];
                            c0[bc][br] = e0p[0];
                            c1[bc][br] = e0p[LEN];
                        }
#pragma unroll
                    for (int kk = 0; kk < KS; ++kk)
#pragma unroll
                        for (int bc = 0; bc < NB; ++bc)
#pragma unroll
                            for (int br = 0; br < NB; ++br)
                            {
#if NUSLAM_RES2_EXP == 8
                                c0[bc][br] += a[kk][br], c1[bc][br] += b[kk][bc];
#else
                                dmma884(c0[bc][br], c1[bc][br], a[kk][br], b[kk][bc]);
#endif
                            }
#pragma unroll
                    for (int bc = 0; bc < NB; ++bc)
#pragma unroll
                        for (int br = 0; br < NB; ++br)
                        {
                            double * const e0p = tbase + bc * (8 * LEN) + rrow[br];
                            e0p[0] = c0[bc][br];
                            e0p[LEN] = c1[bc][br];
                        }
                }
            }
            __syncwarp();
        }

        // ---- write back: robot rows / columns into the image (live filters), the pair to HBM by one bulk store ----
        if (!dead)
        {
            img[q * LEN] = Rt[0], img[q * LEN + 1] = Rx[0], img[q * LEN + 2] = Ry[0];
            if (q >= 3) img[q] = Ct[0], img[LEN + q] = Cx[0], img[2 * LEN + q] = Cy[0];
            p.x[bf * LEN + q] = x[0];
            if (p.x_snap) p.x_snap[bf * LEN + q] = x[0];
            if (v1)
            {
                img[i1 * LEN] = Rt[1], img[i1 * LEN + 1] = Rx[1], img[i1 * LEN + 2] = Ry[1];
                img[i1] = Ct[1], img[LEN + i1] = Cx[1], img[2 * LEN + i1] = Cy[1];
                p.x[bf * LEN + 16 + q] = x[1];
                if (p.x_snap) p.x_snap[bf * LEN + 16 + q] = x[1];
            }
            if (q == 0 && status != st0) p.status[bf] = status;
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0)
        {
            double * gw = p.sigma + 2 * pr * SIG;
            double * im0 = reinterpret_cast<double *>(stage);
            if (2 * pr + 1 < p.batch)
                bulk_s2g(gw, im0, kPairBytes);   // a dead twin's image is untouched: it goes back as it came
            else
            {
                // the single filter of an odd batch's last pair: its 16-byte aligned part + the last element
                bulk_s2g(gw, im0, kImg - 8);
                gw[SIG - 1] = im0[SIG - 1];
            }
            // the buffer receives the next pair as soon as the store has read it
            bulk_wait_read();
            if (next) issue_load(pr + gwn);
        }
        __syncwarp();
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // shared memory must outlive the last bulk store
    strict_tail(p, do_predict, worklist, wl_count, (int) gwn, lane);
}

template <int N>
int launch_res2_n(const EkfParams & p, bool do_predict, int sm_count, int32_t * worklist, int32_t * wl_count, cudaStream_t stream)
{
    int64_t blocks = (p.batch + 1) / 2;   // one pair per warp
    if (blocks > kRes2CtasPerSm * (int64_t) sm_count) blocks = kRes2CtasPerSm * (int64_t) sm_count;
    constexpr int kSmem = 2 * FastGeom<N>::SIG * 8 + (int) sizeof(Res2Smem<NUSLAM_RES2_CH>) + 16;
    static bool configured_dev[kMaxDevices] = {false};
    bool & configured = configured_dev[device_slot()];
    if (!configured)
    {
        cudaFuncSetAttribute(k_ekf_res2_step<N, NUSLAM_RES2_CH>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        const cudaError_t e = cudaFuncSetAttribute(k_ekf_res2_step<N, NUSLAM_RES2_CH>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
        if (e != cudaSuccess) return (int) e;
        configured = true;
    }
    k_ekf_res2_step<N, NUSLAM_RES2_CH><<<(unsigned) blocks, 32, kSmem, stream>>>(p, do_predict ? 1 : 0, worklist, wl_count);
    return (int) cudaGetLastError();
}

// known correspondence, 16-byte aligned Sigma array, the BASELINE map size; everything else stays with ekf_fast.cuh
inline bool res2_supported(int n, const EkfParams & p)
{
    return n == 12 && p.ids != nullptr && p.m_valid == nullptr && p.m >= 0 && p.m <= kFastMMax && p.batch >= 1 &&
           (reinterpret_cast<uintptr_t>(p.sigma) & 15) == 0 && (reinterpret_cast<uintptr_t>(p.x) & 7) == 0;
}

}   // namespace nuslam
