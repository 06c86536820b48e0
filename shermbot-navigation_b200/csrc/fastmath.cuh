// fastmath.cuh -- short-dependency-chain fp64 helpers for the scalar part of the FAST EKF update.
//
// The scalar part of an update (rsqrt, atan2, 2x2 inverse) is a pure latency chain: one lane per filter, nothing
// to overlap it with inside that lane. CUDA's library versions are accurate but long (IEEE division fix-ups,
// Horner polynomials, slow-path calls); these keep ~1-2 ulp accuracy with the minimum number of DEPENDENT steps:
// MUFU seed + two Newton steps, Estrin polynomials. They are used only where the FAST mode is allowed to differ
// from the oracle's libm by rounding (never on a landmark's first touch, see ekf_fast.cuh).
#pragma once
#include <cuda_runtime.h>

namespace nuslam
{

// Sign / magnitude tests on the bit pattern: integer instructions instead of fp64-pipe DADD |x| and DSETP (the fp64 pipe is the
// contended resource of the EKF kernel). abs_bits clears the sign; for non-negative doubles the integer order is the fp order.
__device__ __forceinline__ double abs_bits(double x) { return __hiloint2double(__double2hiint(x) & 0x7fffffff, __double2loint(x)); }
__device__ __forceinline__ bool sign_bit(double x) { return __double2hiint(x) < 0; }
__device__ __forceinline__ bool gt_nonneg(double a, double b) { return __double_as_longlong(a) > __double_as_longlong(b); }
// |x| >= ~bound, decided on the high word alone (bound_hi = high word of the bound); true for inf / nan
__device__ __forceinline__ bool abs_ge_hi(double x, int bound_hi) { return (__double2hiint(x) & 0x7fffffff) >= bound_hi; }
constexpr int kHiPi = 0x400921fb;      // high word of pi: |x| < pi whenever the test fails, and wrapping is the identity up to pi
constexpr int kHi1e300 = 0x7e37e43c;   // high word of 1e300

// 1/x: MUFU.RCP64H seed (~2^-20) + 2 Newton steps -> <= 1 ulp for normal x
__device__ __forceinline__ double rcp_fast(double x)
{
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double e = fma(-x, y, 1.0);
    y = fma(y, e, y);
    e = fma(-x, y, 1.0);
    y = fma(y, e, y);
    return y;
}

// a / b by a reciprocal and one correction: <= 1 ulp for normal operands, no slow path (no call into the device library)
__device__ __forceinline__ double div_fast(double a, double b)
{
    const double y = rcp_fast(b);
    const double q = a * y;
    return fma(fma(-b, q, a), y, q);
}

// 1/sqrt(x): MUFU.RSQ64H seed + 2 Newton steps -> <= 1 ulp for normal x
__device__ __forceinline__ double rsqrt_fast(double x)
{
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double e = fma(-x * y, y, 1.0);
    y = fma(0.5 * y, e, y);
    e = fma(-x * y, y, 1.0);
    y = fma(0.5 * y, e, y);
    return y;
}

// 1/sqrt(x) with ONE Newton step (relative error <= 1.3e-12, worst measured 1.23e-12): enough where a consumer squares the error
// away -- sqrt(x) = x rs refined once is exact to an ulp -- or tolerates it (the unit vector of atan2_unit: <= 1e-14 rad)
__device__ __forceinline__ double rsqrt_1(double x)
{
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double e = fma(-x * y, y, 1.0);
    return fma(0.5 * y, e, y);
}

// atan2(y, x) for finite arguments, not both zero, with ONE division. With mn = min(|x|, |y|), mx = max(|x|, |y|) and
// t_k = k / 64 the table point nearest to mn / mx (k from an fp32 estimate; any neighbouring k works),
//   atan(mn / mx) = atan(t_k) + atan(r),   r = (mn - t_k mx) / (mx + t_k mn),   |r| <= ~1 / 100,
// so a degree-7 odd polynomial (error r^9 / 9 < 1e-19) finishes it; atan(t_k) comes from a 65-entry (hi, lo) table and the
// octant (|y| > |x|, x < 0, y < 0) from an 8-entry table: atan2 = A + S (atan(t_k) + atan(r)) with A = k pi/4 (hi + lo).
// Domain: max(|x|, |y|) in [2^-100, 2^100] (its callers pass metres: the bearing of the large-map model, the circle fit's inscribed
// angles); there the error is <= 2 ulp (worst measured 1.36 ulp). Outside it the fp32 estimate of mn / mx breaks down ((float) mx
// overflows or is denormal, __fdividef returns 0 for a divisor above 2^126), k is wrong, |r| is no longer small and the result is a
// number far from atan2 (NaN for a denormal mx, which rcp_fast flushes to zero); nothing traps. The signs are tested with x < 0 and
// y < 0, so a zero argument counts as +0: atan2_fast(-0, x < 0) = +pi (libm: -pi), atan2_fast(y, -0) = atan2(y, +0).
struct AtanOctant
{
    double hi, lo, s, pad;
};
#define NUSLAM_Q(k) ((k) * 7.85398163397448279e-01), ((k) * 3.06161699786838302e-17)
// index = swap | xneg << 1 | yneg << 2
static __constant__ AtanOctant kAtanOct[8] = {{NUSLAM_Q(0.0), 1.0, 0.0},   {NUSLAM_Q(2.0), -1.0, 0.0},  {NUSLAM_Q(4.0), -1.0, 0.0},  {NUSLAM_Q(2.0), 1.0, 0.0},
                                       {NUSLAM_Q(-0.0), -1.0, 0.0}, {NUSLAM_Q(-2.0), 1.0, 0.0},  {NUSLAM_Q(-4.0), 1.0, 0.0},  {NUSLAM_Q(-2.0), -1.0, 0.0}};
#undef NUSLAM_Q
static __constant__ double2 kAtanTab[65] = {
    {0.0, 0.0},
    {0.015623728620476831, -4.913600136566304e-19},
    {0.031239833430268277, -1.188442711587748e-18},
    {0.046840712915969654, -1.655677442254952e-19},
    {0.06241880999595735, -1.5490756308295046e-18},
    {0.0779666338315423, 5.804551873143357e-18},
    {0.09347678115858947, -6.2844725995420954e-18},
    {0.10894195698986579, 6.8267122072409585e-18},
    {0.12435499454676144, -3.1253241424539383e-18},
    {0.13970887428916365, -2.9579864247315813e-18},
    {0.15499674192394097, 9.585415594114324e-18},
    {0.1702119252854744, -3.541164079802125e-18},
    {0.18534794999569476, 4.180692268843079e-18},
    {0.2003985538258785, 3.1399542871844493e-18},
    {0.21535769969773805, 4.738160130078733e-19},
    {0.23021958727684372, 1.2313404529142703e-17},
    {0.24497866312686414, 1.0698755618734451e-17},
    {0.2596296294082575, 1.9238754924615304e-17},
    {0.2741674511196588, 8.261353575163773e-18},
    {0.2885873618940774, -1.428369957377257e-17},
    {0.3028848683749714, -1.1010827903001369e-17},
    {0.31705575320914703, -1.893928924292642e-17},
    {0.3310960767041321, -7.952610375793799e-18},
    {0.34500217720710513, -2.2938804755578304e-17},
    {0.35877067027057225, -2.4623815582638635e-17},
    {0.3723984466767542, 1.9612311504845653e-17},
    {0.38588266939807375, 2.378822732491941e-17},
    {0.39922076957525254, 2.246598105617042e-17},
    {0.4124104415973873, -1.587652227770689e-17},
    {0.42544963737004227, 2.3315530741892885e-17},
    {0.43833655985795783, -2.494277030626541e-17},
    {0.4510696559885235, -2.2703795229420475e-17},
    {0.4636476090008061, 2.2698777452961687e-17},
    {0.4760693303227612, 1.4654487332256713e-17},
    {0.48833395105640554, -1.1373236189329585e-17},
    {0.5004408131472942, -4.7181675085518756e-17},
    {0.5123894603107377, -2.5462781472855804e-17},
    {0.5241796287829132, 5.520094119641666e-18},
    {0.5358112379604637, -4.0637956834825575e-18},
    {0.5472843809874369, 4.923709671396255e-17},
    {0.5585993153435624, -5.4556305485916264e-18},
    {0.5697564534829784, 1.2255062085054184e-17},
    {0.5807563535676704, -1.441464378193067e-17},
    {0.5915997103351114, 4.920495453686772e-17},
    {0.6022873461349642, 2.950430737228402e-17},
    {0.6128202021652414, -3.1552061848586226e-17},
    {0.6231993299340659, 2.672403885140095e-17},
    {0.6334258829691446, -2.7290767436015276e-17},
    {0.6435011087932844, 1.5834785051444286e-17},
    {0.6534263411807619, 3.5800634857340095e-17},
    {0.6632029927060933, -3.076054864429649e-17},
    {0.6728325475937632, -1.899315009714705e-17},
    {0.6823165548747481, 6.943223671560008e-18},
    {0.6916566218531999, -8.117151192285796e-18},
    {0.7008544078844502, -1.987626234335816e-17},
    {0.7099116184635249, -4.597166450584887e-17},
    {0.7188299996216245, -2.1478388444456983e-17},
    {0.7276113326265107, 2.569325697391839e-18},
    {0.7362574289814281, 3.473937648299457e-17},
    {0.7447701257160751, 3.708315849135547e-17},
    {0.7531512809621944, -2.4256934659182068e-17},
    {0.7614027698055784, 9.850030332752822e-18},
    {0.7695264804056583, -3.704991905602721e-17},
    {0.7775243103733478, -2.6676490951944502e-17},
    {0.7853981633974483, 3.061616997868383e-17}};

// fp64 literals of the per-update scalar chain, kept in the constant bank: an instruction reads them as a c[][] operand, where an
// immediate would be rebuilt in uniform registers (two UMOVs each) on every pass of the update loop
static __constant__ double kFastK[8] = {-1.0 / 7.0, 0.2, -1.0 / 3.0, 6.28318530717958623200, 2.44929359829470641435e-16, 0.15915494309189533577,
                                 1.0e300, 3.14159265358979311600};

static __constant__ double kFastK2[4] = {15.0 / 336.0, 3.0 / 40.0, 1.0 / 6.0, 0.0};   // asin series of atan2_unit

// angle -> [-pi, pi]: what rigid2d::normalize_angle (rigid2d.cpp:9-13) returns, to ~1 ulp, without the
// sin/cos/atan2 round trip; the identity for |a| <= pi, branch-free
__device__ __forceinline__ double wrap_angle(double a)
{
    const double k = rint(a * kFastK[5]);   // 1 / 2 pi; 2 pi = kFastK[3] + kFastK[4]
    return fma(-k, kFastK[4], fma(-k, kFastK[3], a));
}


__device__ __forceinline__ double atan2_fast(double y, double x)
{
    const double ax = fabs(x), ay = fabs(y);
    const bool sw = ay > ax;
    const double mx = sw ? ay : ax, mn = sw ? ax : ay;
    const int idx = (sw ? 1 : 0) | (x < 0.0 ? 2 : 0) | (y < 0.0 ? 4 : 0);
    const AtanOctant oc = kAtanOct[idx];
    // table point: fp32 estimate of 64 mn / mx (the fp32 pipe is idle in this kernel)
    const float tf = __fdividef((float) mn, (float) mx);
    const int k = max(0, min(64, __float2int_rn(tf * 64.0f)));
    const double tk = (double) k * 0.015625;
    const double2 ak = kAtanTab[k];
    const double num = fma(-tk, mx, mn), den = fma(tk, mn, mx);
    const double rc = rcp_fast(den);
    double r = num * rc;
    r = fma(fma(-den, r, num), rc, r);   // r = num / den to ~1 ulp
    const double u = r * r;
    const double pl = fma(fma(fma(kFastK[0], u, kFastK[1]), u, kFastK[2]), u * r, r);   // atan(r)
    const double a = ak.x + (pl + ak.y);                                              // atan(mn / mx) in [0, pi/4]
    return oc.hi + fma(oc.s, a, oc.lo);
}


// atan2(y, x) given rs = 1 / sqrt(x^2 + y^2) (the update has it already), with NO fp64 division: (v, u) = (mx, mn) rs is the unit
// vector (cos psi, sin psi), psi = atan(mn / mx); with the table point psi_k = atan(k / 64) nearest to it,
//   e = sin(psi - psi_k) = u cos psi_k - v sin psi_k,   |e| <= ~1 / 128,   psi - psi_k = asin(e) = e + e^3/6 + 3 e^5/40 + 15 e^7/336
// (next term < 1e-20). Worst absolute error 4.9e-16 over 4e7 cases against atan2l (rs within an ulp of the exact value).
struct AtanEntry
{
    double hi, lo, c, s;   // atan(k / 64) as hi + lo, cos and sin of it
};
static __constant__ AtanEntry kAtanUnit[65] = {
    {0.0, 0.0, 1.0, 0.0},
    {0.015623728620476831, -4.913600136566304e-19, 0.9998779520346953, 0.015623093000542114},
    {0.031239833430268277, -1.188442711587748e-18, 0.9995120760870788, 0.031234752377721213},
    {0.046840712915969654, -1.655677442254952e-19, 0.9989031743698379, 0.046823586298586156},
    {0.06241880999595735, -1.5490756308295046e-18, 0.9980525784828885, 0.06237828615518053},
    {0.0779666338315423, 5.804551873143357e-18, 0.9969621413492435, 0.07788766729290965},
    {0.09347678115858947, -6.2844725995420954e-18, 0.9956342260592881, 0.09334070869305826},
    {0.10894195698986579, 6.8267122072409585e-18, 0.9940716917543757, 0.10872659128563485},
    {0.12435499454676144, -3.1253241424539383e-18, 0.9922778767136676, 0.12403473458920845},
    {0.13970887428916365, -2.9579864247315813e-18, 0.9902565788380346, 0.1392548313990986},
    {0.15499674192394097, 9.585415594114324e-18, 0.9880120337511015, 0.1543768802736096},
    {0.1702119252854744, -3.541164079802125e-18, 0.9855488907597534, 0.16939121559933262},
    {0.18534794999569476, 4.180692268843079e-18, 0.9828721869343219, 0.18428853505018536},
    {0.2003985538258785, 3.1399542871844493e-18, 0.9799873195820534, 0.1990599242901046},
    {0.21535769969773805, 4.738160130078733e-19, 0.9769000173962616, 0.21369687880543226},
    {0.23021958727684372, 1.2313404529142703e-17, 0.973616310567801, 0.22819132278932833},
    {0.24497866312686414, 1.0698755618734451e-17, 0.9701425001453319, 0.24253562503633297},
    {0.2596296294082575, 1.9238754924615304e-17, 0.9664851269264961, 0.25672261183985057},
    {0.2741674511196588, 8.261353575163773e-18, 0.962650940153899, 0.2707455769182841},
    {0.2885873618940774, -1.428369957377257e-17, 0.9586468662780966, 0.28459828842630996},
    {0.3028848683749714, -1.1010827903001369e-17, 0.9544799780350297, 0.2982749931359468},
    {0.31705575320914703, -1.893928924292642e-17, 0.9501574640680012, 0.31177041789731286},
    {0.3310960767041321, -7.952610375793799e-18, 0.9456865993048666, 0.3250797685110479},
    {0.34500217720710513, -2.2938804755578304e-17, 0.9410747162800739, 0.33819872616315155},
    {0.35877067027057225, -2.4623815582638635e-17, 0.9363291775690445, 0.3511234415883917},
    {0.3723984466767542, 1.9612311504845653e-17, 0.9314573494796192, 0.3638505271404763},
    {0.38588266939807375, 2.378822732491941e-17, 0.9264665771223092, 0.3763770469559381},
    {0.39922076957525254, 2.246598105617042e-17, 0.921364160958329, 0.38870050540429507},
    {0.4124104415973873, -1.587652227770689e-17, 0.9161573349021892, 0.40081883401970775},
    {0.42544963737004227, 2.3315530741892885e-17, 0.9108532460343002, 0.4127303771092923},
    {0.43833655985795783, -2.494277030626541e-17, 0.9054589359588684, 0.4244338762307196},
    {0.4510696559885235, -2.2703795229420475e-17, 0.8999813238235362, 0.4359284537270253},
    {0.4636476090008061, 2.2698777452961687e-17, 0.8944271909999159, 0.4472135954999579},
    {0.4760693303227612, 1.4654487332256713e-17, 0.888803167408494, 0.4582891331950047},
    {0.48833395105640554, -1.1373236189329585e-17, 0.8831157194574105, 0.46915522596174936},
    {0.5004408131472942, -4.7181675085518756e-17, 0.8773711395523853, 0.4798123419427107},
    {0.5123894603107377, -2.5462781472855804e-17, 0.8715755371245493, 0.49026123963255896},
    {0.5241796287829132, 5.520094119641666e-18, 0.8657348311141285, 0.5005029492378555},
    {0.5358112379604637, -4.0637956834825575e-18, 0.8598547438407345, 0.5105387541554361},
    {0.5472843809874369, 4.923709671396255e-17, 0.8539407961853737, 0.520370172675462},
    {0.5585993153435624, -5.4556305485916264e-18, 0.847998304005088, 0.52999894000318},
    {0.5697564534829784, 1.2255062085054184e-17, 0.8420323756982734, 0.5394269906817064},
    {0.5807563535676704, -1.441464378193067e-17, 0.8360479108370626, 0.5486564414868224},
    {0.5915997103351114, 4.920495453686772e-17, 0.8300495997825932, 0.5576895748539298},
    {0.6022873461349642, 2.950430737228402e-17, 0.8240419241993676, 0.5665288228870652},
    {0.6128202021652414, -3.1552061848586226e-17, 0.8180291583861419, 0.575176751990256},
    {0.6231993299340659, 2.672403885140095e-17, 0.8120153713427134, 0.5836360481525753},
    {0.6334258829691446, -2.7290767436015276e-17, 0.806004429494522, 0.5919095029100396},
    {0.6435011087932844, 1.5834785051444286e-17, 0.8, 0.6},
    {0.6534263411807619, 3.5800634857340095e-17, 0.7940055545690287, 0.6079105027169125},
    {0.6632029927060933, -3.076054864429649e-17, 0.7880243737245634, 0.6156440419723151},
    {0.6728325475937632, -1.899315009714705e-17, 0.7820595514434194, 0.6232037050564748},
    {0.6823165548747481, 6.943223671560008e-18, 0.7761140001162655, 0.6305926250944658},
    {0.6916566218531999, -8.117151192285796e-18, 0.770190455771008, 0.637813971185366},
    {0.7008544078844502, -1.987626234335816e-17, 0.7642914835078908, 0.6448709392097829},
    {0.7099116184635249, -4.597166450584887e-17, 0.7584194830987478, 0.6517667432879864},
    {0.7188299996216245, -2.1478388444456983e-17, 0.7525766947068778, 0.658504607868518},
    {0.7276113326265107, 2.569325697391839e-18, 0.7467652046879308, 0.6650877604251884},
    {0.7362574289814281, 3.473937648299457e-17, 0.7409869514359827, 0.6715194247388594},
    {0.7447701257160751, 3.708315849135547e-17, 0.7352437312425926, 0.677802814739265},
    {0.7531512809621944, -2.4256934659182068e-17, 0.7295372041400852, 0.6839411288813299},
    {0.7614027698055784, 9.850030332752822e-18, 0.7238688997035583, 0.689937545029954},
    {0.7695264804056583, -3.704991905602721e-17, 0.7182402227891737, 0.695795215827012},
    {0.7775243103733478, -2.6676490951944502e-17, 0.7126524591891511, 0.7015172645143206},
    {0.7853981633974483, 3.061616997868383e-17, 0.7071067811865476, 0.7071067811865476}};

__device__ __forceinline__ double atan2_unit(double y, double x, double rs)
{
    const double ax = abs_bits(x), ay = abs_bits(y);
    const bool sw = gt_nonneg(ay, ax);
    const double mx = sw ? ay : ax, mn = sw ? ax : ay;
    const int idx = (sw ? 1 : 0) | (sign_bit(x) ? 2 : 0) | (sign_bit(y) ? 4 : 0);
    const AtanOctant oc = kAtanOct[idx];
    const float tf = __fdividef((float) mn, (float) mx);
    const int k = max(0, min(64, __float2int_rn(tf * 64.0f)));
    const AtanEntry t = kAtanUnit[k];
    const double u = mn * rs, v = mx * rs;
    const double e = fma(u, t.c, -(v * t.s));
    const double e2 = e * e;
    const double pl = fma(fma(fma(kFastK2[0], e2, kFastK2[1]), e2, kFastK2[2]), e2 * e, e);   // asin(e)
    const double a = t.hi + (pl + t.lo);
    return oc.hi + fma(oc.s, a, oc.lo);
}


// sin and cos without a slow path (no call into the device library: under -rdc such a call is an ABI call that costs the FAST kernels
// registers). Cody-Waite reduction by pi/2 in three 33-bit pieces (exact products for |a| < ~1e6; beyond that the error grows with |a|,
// a heading is normalised to [-pi, pi] after every update), then the fdlibm kernels on [-pi/4, pi/4] (|error| < 2^-58). Against the
// correctly rounded sin / cos: <= 1.7 ulp for |a| <= 1e3 (worst measured 1.63 ulp), <= 2 ulp at |a| ~ 1e6 (measured 1.94): the reduced
// argument is rounded once before the ~0.5 ulp kernels, so this is ~1 ulp of the library's results, not of the true values; far inside
// FAST mode's 1e-9. Pure fma arithmetic: the host computes the device's bits (tests/test_fastmath_tables.py checks it there).
__host__ __device__ __forceinline__ void sincos_fast(double a, double * sn, double * cs)
{
    const double k = rint(a * 6.36619772367581382433e-01);
    double r = fma(-k, 1.57079632673412561417e+00, a);
    r = fma(-k, 6.07710050630396597660e-11, r);
    r = fma(-k, 2.02226624871116645580e-21, r);
    r = fma(-k, 8.47842766036889956997e-32, r);
    const double z = r * r;
    const double ps = fma(fma(fma(fma(fma(1.58969099521155010221e-10, z, -2.50507602534068634195e-08), z, 2.75573137070700676789e-06), z,
                                  -1.98412698298579493134e-04), z, 8.33333333332248946124e-03), z, -1.66666666666666324348e-01);
    const double pc = fma(fma(fma(fma(fma(-1.13596475577881948265e-11, z, 2.08757232129817482790e-09), z, -2.75573143513906633035e-07), z,
                                  2.48015872894767294178e-05), z, -1.38888888888741095749e-03), z, 4.16666666666666019037e-02);
    const double s = fma(ps * z, r, r);
    const double c = fma(z * z, pc, fma(-0.5, z, 1.0));
    const int n = (int) (long long) k & 3;
    const double s1 = (n & 1) ? c : s, c1 = (n & 1) ? s : c;
    *sn = (n & 2) ? -s1 : s1;
    *cs = ((n + 1) & 2) ? -c1 : c1;
}

// sin and cos of a SMALL angle (|a| <= 0.25: a wheel-odometry step) straight from the Taylor series, no argument reduction; the
// truncation error is below 3e-18 and the result within 1 ulp of the correctly rounded value. Larger arguments take sincos_fast.
static __constant__ double kSinK[6] = {-1.0 / 6.0, 1.0 / 120.0, -1.0 / 5040.0, 1.0 / 362880.0, -1.0 / 39916800.0, 1.0 / 6227020800.0};
static __constant__ double kCosK[7] = {-0.5, 1.0 / 24.0, -1.0 / 720.0, 1.0 / 40320.0, -1.0 / 3628800.0, 1.0 / 479001600.0, -1.0 / 87178291200.0};
__device__ __forceinline__ void sincos_small(double a, double * sn, double * cs)
{
    if (fabs(a) > 0.25)   // warp-uniform in the EKF kernel (every lane holds the same twist)
    {
        sincos_fast(a, sn, cs);
        return;
    }
    const double u = a * a;
    const double ps = fma(fma(fma(fma(fma(kSinK[5], u, kSinK[4]), u, kSinK[3]), u, kSinK[2]), u, kSinK[1]), u, kSinK[0]);
    const double pc = fma(fma(fma(fma(fma(fma(kCosK[6], u, kCosK[5]), u, kCosK[4]), u, kCosK[3]), u, kCosK[2]), u, kCosK[1]), u, kCosK[0]);
    *sn = fma(ps * u, a, a);
    *cs = fma(pc, u, 1.0);
}

}   // namespace nuslam
