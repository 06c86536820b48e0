/* include/nuslam_b200.h -- C ABI of the B200-native batched EKF-SLAM + scan circle-detection engine.
 *
 * Drop-in boundary for the hot path of sziselman/Shermbot-Navigation. The reference has no FFI or
 * plugin layer: its seam is the C++ API of two catkin libraries, `libnuslam`
 * (nuslam/include/nuslam/slam_library.hpp:18-113, nuslam/include/nuslam/circle_fit_library.hpp:18-28)
 * and `librigid2d`. Every entry point below is the batched (B filters / S scans per call) form of one
 * of those functions and cites the interface it replaces; the B = 1 C++ facade that keeps the
 * reference's class and function names is include/nuslam_b200/slam_library.hpp (namespaces slam_library
 * and circle_fit), with forwarding headers include/nuslam_b200/compat/nuslam/{slam_library,
 * circle_fit_library}.hpp for unmodified callers. rigid2d stays the caller's own host library (it has no
 * third-party arithmetic); its functions on the path have batched entry points below.
 *
 * Conventions (all inherited from the reference):
 *   - state vector x = [theta, x, y, m1x, m1y, ...], length len = 3 + 2n   (slam_library.cpp:46-59)
 *   - landmark ids are 1-based; slot of id j is 3 + 2(j-1)                  (slam_library.cpp:152-153)
 *   - matrices are column-major (Armadillo): Sigma[b][col*len + row], Q[col*3 + row], R[col*2 + row]
 *   - a twist is (dth, dx, dy) in that order                                (rigid2d.hpp:150-155)
 *   - a measurement z is polar (range, bearing)                             (slam_library.cpp:16-22)
 *
 * Plain pointers and sizes only. Each array argument is either a host pointer or a device pointer on
 * the handle's device, as stated by the `mem` argument of the call (NUSLAM_HOST / NUSLAM_DEVICE).
 * With NUSLAM_DEVICE a call only enqueues work on the handle's stream (use nuslam_ekf_synchronize or
 * your own stream/event ordering); with NUSLAM_HOST it copies in, runs, copies results out and returns
 * after they have landed. A handle is not thread-safe; independent handles are.
 *
 * There is NO CPU fallback: every compute entry point runs hand-written sm_100a kernels and returns
 * NUSLAM_ERR_CUDA when no such device is present.
 */
#ifndef NUSLAM_B200_H
#define NUSLAM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NUSLAM_B200_VERSION 101

/* ---- return codes of every entry point ---- */
enum
{
    NUSLAM_OK = 0,
    NUSLAM_ERR_INVALID = 1,     /* bad argument (null handle, m < 0, n_landmarks < 1, ...) */
    NUSLAM_ERR_CUDA = 2,        /* CUDA runtime error or no sm_100 device; see nuslam_last_error() */
    NUSLAM_ERR_NOMEM = 3,
    NUSLAM_ERR_UNSUPPORTED = 4  /* configuration outside what the kernels cover (e.g. state too long for the batched path) */
};

enum
{
    NUSLAM_HOST = 0,
    NUSLAM_DEVICE = 1
};

/* ---- arithmetic mode ----
 * STRICT reproduces the operation order of the reference's dense expressions
 *   A*Sigma*A.t()+Q_bar (slam_library.cpp:104), Sigma*H.t()*inv(H*Sigma*H.t()+R) (:270),
 *   (I-K*H)*Sigma (:279)
 * term by term (ascending k, unfused multiply/add), skipping only structurally-zero terms, so Sigma is
 * bit-identical to the oracle given identical inputs.
 * FAST uses the algebraically identical rank-2 form Sigma -= K*(H*Sigma) with fused multiply-adds and
 * keeps Sigma in registers; it falls back to the STRICT arithmetic for any update whose landmark still
 * carries its INT_MAX prior (first touch, slam_library.cpp:28-31), where the reference's
 * (I-KH)*Sigma cancels catastrophically and only the same operation order reproduces its result.
 * The register kernel covers n_landmarks <= 12 and m <= 16; a FAST handle of any other size runs the STRICT kernels. */
enum
{
    NUSLAM_MODE_STRICT = 0,
    NUSLAM_MODE_FAST = 1,
    /* LARGE-MAP mode (BASELINE.json config 5): Sigma stays in HBM; the m updates of a step are DELAYED -- each needs only
     * rows / columns {theta, x, y, c, c+1} of the current Sigma, formed on the fly from Sigma_0 and the stored K_u, W_u -- and
     * applied in ONE rank-2m pass on the fp64 tensor pipe: one read + one write of Sigma per scan whatever m is. Selected
     * automatically when the state is too long for the on-chip kernels (n_landmarks > ~70). nuslam_ekf_step takes known or unknown correspondence
     * (associateLandmark: one thread per candidate landmark against the pass's current covariance); the single-call
     * nuslam_ekf_associate and the fused nuslam_ekf_scan_step (per-filter marker counts) work as in the other modes, and so do
     * the NUSLAM_OPT_* variants (under NUSLAM_OPT_JOSEPH the pass is a symmetric rank-4m update). */
    NUSLAM_MODE_LARGE = 2
};

/* ---- per-filter status word (bit mask, sticky); where the reference throws, the engine flags ---- */
enum
{
    NUSLAM_FILTER_OK = 0,
    NUSLAM_FILTER_MAP_FULL = 1,   /* associateLandmark with seen == n: Armadillo bounds check throws (slam_library.cpp:206).
                                     The filter is frozen from that measurement on, as the reference process would be dead. */
    NUSLAM_FILTER_SINGULAR = 2,   /* det(H Sigma H^T + R) == 0: arma::inv throws (slam_library.cpp:231,270); update skipped */
    NUSLAM_FILTER_BAD_ID = 4,     /* update/initializeLandmark with id outside 1..n: bounds check throws; call skipped */
    NUSLAM_FILTER_ASSOC_TRUNCATED = 8 /* NUSLAM_OPT_JOINT_COMPATIBILITY: a step's search hit its budget of joint tests and used the best
                                         hypothesis found so far. Informational: it never freezes a filter (nuslam_ekf_error_stats
                                         slot [6] counts such filters too, as it counts any non-zero status). */
};

/* id written by nuslam_ekf_associate / nuslam_ekf_step where the reference throws */
#define NUSLAM_ID_EXCEPTION (-1000)

typedef struct nuslam_ekf nuslam_ekf;

typedef struct
{
    int32_t n_landmarks;   /* n = mapState.n_elem / 2 (slam_library.cpp:42) */
    int32_t mode;          /* NUSLAM_MODE_* */
    double Q[9];           /* 3x3 process noise, column-major, (theta,x,y) order (slam_library.cpp:110-125) */
    double R[4];           /* 2x2 sensor noise, column-major (slam_library.cpp:215,270) */
    double assoc_min;      /* 0.01 (slam_library.cpp:193) */
    double assoc_max;      /* 60   (slam_library.cpp:194) */
    uint32_t options;      /* NUSLAM_OPT_* bit mask; 0 = the reference's behaviour (the default, and the parity contract) */
    uint32_t reserved;
    double landmark_prior; /* variance written on the landmark diagonal by nuslam_ekf_init; INT_MAX (slam_library.cpp:30) by default */
} nuslam_ekf_config;

/* Opt-in departures from the reference (SURVEY.md 8f-4), for users who want Monte-Carlo statistics that mean something; never the
 * default because parity with the reference is the contract. They run in the oracle-order kernels and in large-map mode (a FAST
 * handle with options set runs the oracle-order kernels: the register kernel implements the reference's behaviour only). */
enum
{
    NUSLAM_OPT_WRAP_INNOVATION = 1,     /* bearing innovation wrapped to (-pi, pi] in update and associateLandmark (reference: :229-231, :272 do not) */
    NUSLAM_OPT_JOSEPH = 2,              /* Sigma <- (I-KH) Sigma (I-KH)^T + K R K^T, then (Sigma + Sigma^T)/2 (reference: (I-KH) Sigma, :279) */
    NUSLAM_OPT_PRE_MOTION_JACOBIAN = 4, /* getA evaluated at theta BEFORE the motion update (reference: after it, :129) */
    /* associateLandmark by individual-compatibility nearest neighbour (reference: the FIRST candidate k = 1..seen whose distance
     * decides wins, :208-249). Every candidate is evaluated; a singular psi at any of them flags NUSLAM_FILTER_SINGULAR and returns
     * NUSLAM_ID_EXCEPTION. The smallest Mahalanobis distance d* (exact comparison, ties to the lowest id, NaN never a candidate) is a
     * match when d* < assoc_min (the gate), ambiguous (-1) when d* < assoc_max (the new-landmark threshold), and otherwise opens a
     * landmark. Only opening one on a full map (seen == n) flags NUSLAM_FILTER_MAP_FULL; a match there succeeds. A chi-square gate
     * such as 9.21 (99 %, 2 dof) with assoc_max = 60 is the intended use; combine it with NUSLAM_OPT_WRAP_INNOVATION, since an
     * unwrapped bearing innovation near +-pi defeats any distance rule. */
    NUSLAM_OPT_NEAREST_NEIGHBOUR = 8,
    /* The step's measurements associated jointly: joint compatibility branch and bound (JCBB; Neira & Tardos, IEEE T-RO 2001), in
     * the oracle-order kernels only (nuslam_ekf_create refuses it with NUSLAM_OPT_NEAREST_NEIGHBOUR or a non-finite or non-positive
     * assoc_min: NUSLAM_ERR_INVALID; on a large-map handle: NUSLAM_ERR_UNSUPPORTED). assoc_min is the individual gate, a chi-square
     * value at 2 dof (e.g. 9.21); it fixes conf = 1 - exp(-assoc_min / 2), and p pairings pass jointly when their stacked innovation
     * has D^2 = nu^T S^-1 nu < T_p = chi2_{2p}^-1(conf) (T_1 = assoc_min), S = H Sigma H^T + blockdiag(R). A step with unknown ids
     * (nuslam_ekf_step with ids == NULL, nuslam_ekf_scan_step, the step_async paths) takes at most 16 measurements
     * (NUSLAM_ERR_UNSUPPORTED above) and, after predict:
     *  1. d_ik, the nearest-neighbour distance, at the predicted state for every measurement i and candidate k = 1..seen; k is
     *     compatible with i when d_ik < assoc_min (NaN never). A singular psi anywhere flags NUSLAM_FILTER_SINGULAR: the first
     *     measurement gets NUSLAM_ID_EXCEPTION, the others 0, and no update is applied.
     *  2. Depth-first search over the measurements in order: measurement i tries its compatible candidates in ascending (d_ik, k),
     *     skipping landmarks the hypothesis already uses, then no pairing. A pairing is accepted when the joint D^2 of the hypothesis
     *     it extends (at the predicted Sigma) is < T_p; the first pairing's D^2 is its d_ik, and a child whose S is not positive
     *     definite is not accepted. A node is pruned when its pairings plus the measurements it has not decided are fewer than the
     *     best hypothesis' pairings. Better: more pairings, or as many and a strictly smaller D^2. At most 4 096 joint tests per
     *     filter and step: then the best hypothesis so far is used and NUSLAM_FILTER_ASSOC_TRUNCATED is set.
     *  3. A paired measurement gets its landmark's id; an unpaired one -1 when some d_ik < assoc_max (the new-landmark threshold),
     *     otherwise it opens a landmark (seen + 1, seen + 2, ... in measurement order; NUSLAM_FILTER_MAP_FULL and
     *     NUSLAM_ID_EXCEPTION on a full map, as under NUSLAM_OPT_NEAREST_NEIGHBOUR).
     *  4. The ids are applied as every step applies associateLandmark's, one sequential update after another.
     * With one measurement this is nearest neighbour: steps with m = 1 give the bits of a NUSLAM_OPT_NEAREST_NEIGHBOUR handle, and
     * nuslam_ekf_associate (one measurement per call) runs nearest neighbour. Association sees the predicted map only, so two
     * measurements of one unseen landmark in a scan open two landmarks. */
    NUSLAM_OPT_JOINT_COMPATIBILITY = 32
};

/* Q = 0.1 I, R = 0.001 I (nuslam/config/slam_params.yaml:2-3), thresholds 0.01 / 60, STRICT mode */
void nuslam_ekf_default_config(nuslam_ekf_config * cfg, int32_t n_landmarks);

const char * nuslam_last_error(void);
int nuslam_version(void);
/* 1: the library was built with device-side tail launches (-rdc=true): a FAST-mode step launches the oracle-order list kernel itself, and
 * only when a filter was handed over -- one kernel launch per step of a built map; 0: the host launches it after every FAST kernel.
 * (No reference counterpart: diagnostics for bench.py's launch count.) */
int nuslam_tail_launch(void);

/* Create B independent filters on `device`. `cuda_stream` is a cudaStream_t (NULL: the handle creates
 * its own non-blocking stream). State memory is owned by the handle unless nuslam_ekf_bind_state is
 * called. Replaces: ExtendedKalman::ExtendedKalman(robotState, mapState, Q, R), slam_library.cpp:39-63
 * (the state itself is set by nuslam_ekf_init). */
int nuslam_ekf_create(const nuslam_ekf_config * cfg, int64_t batch, int device, void * cuda_stream,
                      nuslam_ekf ** out);
int nuslam_ekf_destroy(nuslam_ekf * h);

/* Use caller-owned device buffers for the filter state (x: B*len f64, sigma: B*len*len f64,
 * seen: B i32, status: B i32), e.g. torch tensors that NCCL gathers at the end of a run. */
int nuslam_ekf_bind_state(nuslam_ekf * h, double * x_dev, double * sigma_dev, int32_t * seen_dev,
                          int32_t * status_dev);
int nuslam_ekf_device_pointers(nuslam_ekf * h, double ** x_dev, double ** sigma_dev, int32_t ** seen_dev,
                               int32_t ** status_dev);

/* Constructor semantics for every filter: x = [robot_state(3), map_state(2n)], Sigma = 0 with INT_MAX on
 * the landmark diagonal, seen = 0, status = OK.  robot_state: B x 3, map_state: B x 2n (NULL = zeros, as
 * slam.cpp:140-157 does).  Replaces slam_library.cpp:39-63 + initCov :24-33. */
int nuslam_ekf_init(nuslam_ekf * h, const double * robot_state, const double * map_state, int mem);

/* Checkpoint / restore / teacher forcing. NULL pointers are skipped. Replaces the getters
 * getStateVector / getCovariance / getSeenLandmarks (slam_library.cpp:284-297). */
int nuslam_ekf_set_state(nuslam_ekf * h, const double * x, const double * sigma, const int32_t * seen,
                         const int32_t * status, int mem);
int nuslam_ekf_get_state(nuslam_ekf * h, double * x, double * sigma, int32_t * seen, int32_t * status,
                         int mem);

/* ExtendedKalman::predict(tw), slam_library.cpp:65-69. twists: B x 3 (dth, dx, dy). */
int nuslam_ekf_predict(nuslam_ekf * h, const double * twists, int mem);

/* ExtendedKalman::associateLandmark(z_i), slam_library.cpp:188-253. z: B x 2; id_out: B
 * (k >= 1 existing or new landmark, -1 ambiguous, NUSLAM_ID_EXCEPTION when the map is full).
 * Mutates `seen` exactly as the reference does. */
int nuslam_ekf_associate(nuslam_ekf * h, const double * z, int32_t * id_out, int mem);

/* ExtendedKalman::initializeLandmark(z_i, id), slam_library.cpp:255-261. id: B (id <= 0: skip that filter). */
int nuslam_ekf_initialize_landmark(nuslam_ekf * h, const double * z, const int32_t * id, int mem);

/* ExtendedKalman::update(tw, z_id, id), slam_library.cpp:263-282 (tw is unused by the reference).
 * id: B (id <= 0: skip that filter). */
int nuslam_ekf_update(nuslam_ekf * h, const double * z, const int32_t * id, int mem);

/* computeTheoreticalMeasurement(j, state) :150-160 and linearizedMeasurementModel(j, state) :162-186,
 * evaluated at each filter's current state. j: B; zhat: B x 2 (may be NULL); H: B x (2 x len)
 * column-major (may be NULL). */
int nuslam_ekf_measurement_model(nuslam_ekf * h, const int32_t * j, double * zhat, double * H, int mem);

/* One iteration of the caller protocol EKFSlam::main_loop, nuslam/src/slam.cpp:262-319, fused:
 *   seen_snapshot = seen; predict(twist);
 *   for i in 0..m-1:  id = ids ? ids[i] : associateLandmark(z_i)
 *                     if id > seen_snapshot: initializeLandmark(z_i, id)
 *                     else if id < 0: continue
 *                     update(twist, z_i, id)
 * twists: B x 3; z: B x m x 2; ids: B x m (NULL = unknown data association; with known
 * correspondence id <= 0 means "no measurement in this slot" and `seen = max(seen, id)` stands in for
 * what associateLandmark would have done); ids_out: B x m or NULL. */
int nuslam_ekf_step(nuslam_ekf * h, const double * twists, const double * z, const int32_t * ids, int32_t m,
                    int32_t * ids_out, int mem);

/* Pipelined form of nuslam_ekf_step for HOST buffers (ids may be NULL: unknown correspondence): the call enqueues (1) the host->device copy of this
 * step's twists / z / ids, (2) the fused step, (3) the device->host copy of the resulting state vector into x_out (B x len f64),
 * on three streams chained by events, and returns at once; up to three steps are in flight, so the copies of steps t+1 and t-1
 * overlap the kernel of step t. All host pointers should be page-locked and must stay untouched until a later call has
 * recycled the slot (three calls later) or nuslam_ekf_wait_async has returned. Same semantics and results as the synchronous
 * call: one iteration of nuslam/src/slam.cpp:262-319 per filter, followed by getStateVector(). */
int nuslam_ekf_step_async(nuslam_ekf * h, const double * twists, const double * z, const int32_t * ids, int32_t m, double * x_out);

/* The same pipelined step with fewer, larger copies (the host-buffer path is bound by the copies, not by the kernel):
 *   nuslam_ekf_set_ids          keeps the B x m known-correspondence ids on the device (a map with fixed landmark order sends the
 *                               same ids every step); the buffer is free on return
 *   nuslam_ekf_step_async_packed  takes ONE page-locked host buffer [twists B x 3 f64][z B x m x 2 f64][ids B x m i32 if
 *                               NUSLAM_IDS_PACKED], copied by a single cudaMemcpyAsync. ids_mode: NUSLAM_IDS_NONE = unknown
 *                               correspondence (associateLandmark on the device), NUSLAM_IDS_PACKED = ids travel in the buffer,
 *                               NUSLAM_IDS_CACHED = the ids given to nuslam_ekf_set_ids (same m).
 * x_out and the pipeline semantics are those of nuslam_ekf_step_async. */
#define NUSLAM_IDS_NONE 0
#define NUSLAM_IDS_PACKED 1
#define NUSLAM_IDS_CACHED 2
int nuslam_ekf_set_ids(nuslam_ekf * h, const int32_t * ids, int32_t m, int mem);
int nuslam_ekf_step_async_packed(nuslam_ekf * h, const void * packed, int32_t m, int ids_mode, double * x_out);
int nuslam_ekf_wait_async(nuslam_ekf * h);

/* EKFSlam::broadcast_map2odom_tf, nuslam/src/slam.cpp:175-210 (the step after the path): T_mo = T_mb * T_ob.inv() with T_mb from
 * every filter's current estimate (theta, x, y) and T_ob from the odometry model's configuration.
 * odom_state7: B x 7 rows {wheelBase, wheelRad, x, y, th, thL, thR} (the array nuslam_diffdrive_step maintains);
 * out: B x 3 = (translation x, translation y, yaw = normalize_angle(asin(T_mo.getSinTh()))). */
int nuslam_ekf_map_to_odom(nuslam_ekf * h, const double * odom_state7, double * out, int mem);

/* Measurement aid for the host-buffer path: while on, nuslam_ekf_step_async performs exactly its copies (host -> device inputs,
 * device -> host state snapshot), stream hand-overs and events but launches no kernel, so that timing it gives the ceiling the
 * host side (PCIe, pinned-memory bandwidth shared by the ranks of a box) allows for that path. The filters do not advance. */
int nuslam_ekf_async_dry_run(nuslam_ekf * h, int on);
int nuslam_ekf_synchronize(nuslam_ekf * h);
/* Error statistics of the batch against a ground truth, reduced on the device (the Monte-Carlo driver's end-of-run numbers; the
 * reference has no counterpart -- its nodes only draw rviz paths, slam.cpp:161-173). All pointers are DEVICE pointers; the call
 * enqueues on the handle's stream. stats_out receives NUSLAM_STATS_COUNT doubles, SUMS over this handle's filters (so that shards
 * add up under an all-reduce):
 *   [0] squared robot position error   [1] squared heading error (wrapped)   [2] NEES e^T Sigma_rr^-1 e of the pose (3 dof)
 *   [3] filters counted in [0..2]      [4] squared landmark position error   [5] landmarks counted in [4] (the first `seen` ones)
 *   [6] filters with non-zero status   [7] entries of ids_got that differ from ids_want (both B x m, or both NULL)
 * truth_pose: B x 3 (theta, x, y) or NULL; truth_map: n x 2 landmark positions shared by all filters, or NULL. */
#define NUSLAM_STATS_COUNT 8
int nuslam_ekf_error_stats(nuslam_ekf * h, const double * truth_pose, const double * truth_map, const int32_t * ids_got,
                           const int32_t * ids_want, int32_t m, double * stats_out);

/* The cudaStream_t every NUSLAM_DEVICE call of this handle enqueues on (the one given to nuslam_ekf_create, or the handle's own
 * non-blocking stream): a caller that produces inputs / consumes outputs on another stream orders the two with events on it. */
int nuslam_ekf_get_stream(nuslam_ekf * h, void ** cuda_stream_out);

/* slam_library::cartesian2polar(x, y), slam_library.cpp:16-22, batched: xy count x 2 -> rb count x 2. */
int nuslam_cartesian2polar(const double * xy, double * rb, int64_t count, int mem, int device,
                           void * cuda_stream);

/* rigid2d::normalize_angle, rigid2d/src/rigid2d.cpp:9-13, batched. */
int nuslam_normalize_angle(const double * rad_in, double * rad_out, int64_t count, int mem, int device,
                           void * cuda_stream);

/* rigid2d::DiffDrive, batched (rigid2d/include/rigid2d/diff_drive.hpp:13-103): what nuslam/src/slam.cpp:264-265 does with the wheel
 * angles of one joint-state message -- getTwist(thL, thR) (diff_drive.cpp:80-110) then operator()(thL, thR) (:111-146) -- for
 * `count` robots. state7: count x 7 = {wheelBase, wheelRad, x, y, th, thL, thR}, updated in place; twists_out: count x 3
 * (dth, dx, dy = 0), the control input of nuslam_ekf_predict / nuslam_ekf_step. */
int nuslam_diffdrive_step(double * state7, const double * thL_new, const double * thR_new, double * twists_out, int64_t count, int mem,
                          int device, void * cuda_stream);

/* rigid2d::integrateTwist (rigid2d/src/rigid2d.cpp:294-328), batched: twists count x 3 (dth, dx, dy) -> transforms count x 4
 * (cos theta, sin theta, x, y), the Transform2D the twist reaches in unit time (T_bs * T_ss' * T_sb, pure translation for dth == 0). */
int nuslam_integrate_twist(const double * twists, double * transforms_out, int64_t count, int mem, int device, void * cuda_stream);

/* DiffDrive::convertTwist (diff_drive.cpp:66-78), batched: twists count x 3 -> wheel velocities count x 2 (uL, uR). */
int nuslam_diffdrive_convert_twist(double wheel_base, double wheel_rad, const double * twists, double * wheel_vel_out, int64_t count, int mem,
                                   int device, void * cuda_stream);

/* ------------------------------------------------------------------ simulator slice (the step before the path)
 * One iteration of TubeWorld::main_loop (nuturtlesim/src/tube_world.cpp:512-537) for `count` independent simulated robots in one
 * tube field: desired twist = cmd + twist noise (:177-189), check_collision (:371-389), wheel_vel = convertTwist, joints +=
 * wheel_vel * dt (:516-523), robot(joints + wheel_vel * slip) (:528-529, DiffDrive::operator()), simulate_lidar_scanner (:405-471).
 * The four gaussian draws of a step are INPUTS (the reference takes them from a std::mt19937 it seeds from random_device).
 *   world      : count x 9 = {wheelBase, wheelRad, x, y, th, thL, thR, jointL, jointR}, updated in place
 *   cmd        : count x 3 commanded body twist (dth, dx, dy)
 *   noise      : count x 4 = {twist dth, twist dx, slip L, slip R} or NULL (all zero)
 *   tubes      : n_tubes x 2 tube centres (at most 64)
 *   ranges_out : count x 360 f32, the sensor_msgs/LaserScan ranges (fill value max_range + 1)
 *   joints_out : 2 x count (jointL[count] then jointR[count]) or NULL -- the encoder readings, laid out as
 *                nuslam_diffdrive_step's thL_new / thR_new so that the odometry runs on them in place */
int nuslam_world_step(double * world, const double * cmd, const double * noise, double dt, const double * tubes, int32_t n_tubes,
                      double tube_rad, double robot_rad, double max_range, float * ranges_out, double * joints_out, int64_t count,
                      int mem, int device, void * cuda_stream);

/* ------------------------------------------------------------------ scan -> landmarks
 * circle_fit::clusterPoints (circle_fit_library.cpp:136-206), classifyCluster (:208-250), circleFit
 * (:15-134) and the Landmarks::main_loop protocol (nuslam/src/landmarks.cpp:84-109), batched over S
 * scans of exactly 360 float ranges.
 *   cluster_of_beam : S x 360 int16, index of the returned cluster holding the beam, -1 for none
 *   n_clusters      : S      number of clusters clusterPoints returns (after its erase loop)
 *   n_circles       : S      number of markers the landmarks node would publish; NUSLAM_SCAN_UB where the
 *                            reference indexes clusters[0] of an empty vector (undefined behaviour)
 *   circles         : S x max_circles x 4  (cx, cy, R = scale.x/2, cluster index), detection order
 */
#define NUSLAM_SCAN_UB (-2000)
#define NUSLAM_SCAN_BEAMS 360

int nuslam_scan_detect(const float * ranges, int64_t n_scans, double min_range, double max_range,
                       int16_t * cluster_of_beam, int32_t * n_clusters, int32_t * n_circles,
                       double * circles, int32_t max_circles, int mem, int device, void * cuda_stream);

/* Arithmetic of circleFit (circle_fit_library.cpp:15-134) on the batched paths (nuslam_scan_detect, nuslam_ekf_scan_step):
 *   NUSLAM_FIT_MOMENT (default): the Hyper fit from warp-shuffle moment reductions, one fused kernel per call; circles agree with
 *                                the reference to <= 1e-9 relative (measured ~1e-13), every integer output is exact; a scan whose
 *                                decisions could hinge on rounding is re-run in NUSLAM_FIT_JACOBI arithmetic
 *   NUSLAM_FIT_JACOBI:           SVD -> eig_sym -> solve in the operation order the oracle defines for Armadillo's calls
 * Process-wide; returns the previous mode (any other value only queries). The environment variable NUSLAM_SCAN_FIT=jacobi selects
 * the second at start-up. nuslam_scan_last_fallbacks: how many scans of the calling thread's last NUSLAM_FIT_MOMENT call on
 * `device` were re-run (diagnostics; synchronises the device), -1 if none was made. */
#define NUSLAM_FIT_MOMENT 0
#define NUSLAM_FIT_JACOBI 1
int nuslam_scan_set_fit(int mode);
int nuslam_scan_last_fallbacks(int device);

/* circle_fit::classifyCluster / circleFit on explicit point lists: C clusters, cluster c owns points
 * offsets[c] .. offsets[c+1]-1 of px/py. is_circle: C (0/1); fit: C x 4 (marker.id, cx, cy, R). */
int nuslam_classify_and_fit(const double * px, const double * py, const int32_t * offsets, int64_t n_clusters,
                            int32_t * is_circle, double * fit, int mem, int device, void * cuda_stream);

/* ------------------------------------------------------------------ scan -> landmarks -> EKF, fused
 * The two nodes back to back without leaving the device (SURVEY.md 8f-2): scan b belongs to filter b.
 *   markers  = Landmarks::main_loop(ranges_b)                     nuslam/src/landmarks.cpp:84-109
 *   z_i      = cartesian2polar(marker_i.pose.position.{x, y})     nuslam/src/slam.cpp:282-286
 *   one iteration of EKFSlam::main_loop with associateLandmark    nuslam/src/slam.cpp:262-319
 * The MarkerArray wire format between the nodes collapses to 16 bytes per landmark in HBM. Only the first m markers of a
 * scan are used (choose m >= the largest marker count; n_markers_out reports the full count, NUSLAM_SCAN_UB where
 * clusterPoints is undefined -- such a scan contributes no measurement).
 *   twists: B x 3; ranges: B x 360 f32; n_markers_out: B or NULL; z_out: B x m x 2 or NULL (range, bearing; zero past the
 *   filter's last marker); ids_out: B x m or NULL (association results, 0 past the last marker). */
int nuslam_ekf_scan_step(nuslam_ekf * h, const double * twists, const float * ranges, double min_range, double max_range,
                         int32_t m, int32_t * n_markers_out, double * z_out, int32_t * ids_out, int mem);

#ifdef __cplusplus
}
#endif
#endif
