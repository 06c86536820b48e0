"""Host-side mirror of the reference's ``nuslam`` library API over the C ABI (include/nuslam_b200.h).

``BatchedExtendedKalman`` keeps the member names of ``slam_library::ExtendedKalman``
(nuslam/include/nuslam/slam_library.hpp:23-113) -- ``predict``, ``associateLandmark``,
``initializeLandmark``, ``update``, ``computeTheoreticalMeasurement``, ``linearizedMeasurementModel``,
``getStateVector``, ``getCovariance``, ``getSeenLandmarks`` -- with a leading batch dimension, plus the
fused ``step`` (one iteration of nuslam/src/slam.cpp:262-319). Arguments are numpy arrays (host) or
torch CUDA tensors on the engine's device (device pointers, no copies); ids are 1-based as in the
reference; matrices are exchanged as [batch, row, col].

The CUDA library is mandatory: importing this module without ``libnuslam_b200.so`` raises, and the
library itself refuses to run without an sm_100 device. There is no CPU path.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
import os as _os
LIB_PATH = Path(_os.environ.get("NUSLAM_B200_LIB", HERE / "libnuslam_b200.so"))   # override only for kernel experiments

NUSLAM_HOST, NUSLAM_DEVICE = 0, 1
MODE_STRICT, MODE_FAST, MODE_LARGE = 0, 1, 2
FILTER_MAP_FULL, FILTER_SINGULAR, FILTER_BAD_ID = 1, 2, 4
# OPT_JOINT_COMPATIBILITY: a step's search hit its budget of joint tests (4 096) and used the best hypothesis so far; informational,
# it never freezes a filter
FILTER_ASSOC_TRUNCATED = 8
ID_EXCEPTION = -1000
SCAN_UB = -2000

EXPORTS = [
    "nuslam_last_error", "nuslam_version", "nuslam_ekf_default_config", "nuslam_ekf_create", "nuslam_ekf_destroy",
    "nuslam_ekf_bind_state", "nuslam_ekf_device_pointers", "nuslam_ekf_init", "nuslam_ekf_set_state",
    "nuslam_ekf_get_state", "nuslam_ekf_predict", "nuslam_ekf_associate", "nuslam_ekf_initialize_landmark",
    "nuslam_ekf_update", "nuslam_ekf_measurement_model", "nuslam_ekf_step", "nuslam_ekf_step_async", "nuslam_ekf_wait_async",
    "nuslam_ekf_scan_step", "nuslam_ekf_map_to_odom", "nuslam_ekf_synchronize",
    "nuslam_cartesian2polar", "nuslam_normalize_angle", "nuslam_scan_detect", "nuslam_classify_and_fit",
    "nuslam_diffdrive_step", "nuslam_diffdrive_convert_twist", "nuslam_world_step", "nuslam_integrate_twist",
    "nuslam_ekf_get_stream", "nuslam_scan_set_fit", "nuslam_scan_last_fallbacks", "nuslam_ekf_error_stats", "nuslam_ekf_async_dry_run", "nuslam_ekf_set_ids", "nuslam_ekf_step_async_packed",
    "nuslam_tail_launch",
]


OPT_WRAP_INNOVATION, OPT_JOSEPH, OPT_PRE_MOTION_JACOBIAN = 1, 2, 4   # include/nuslam_b200.h NUSLAM_OPT_*
# associateLandmark by nearest neighbour instead of the reference's first deciding candidate: the closest candidate matches when its
# Mahalanobis distance is below assoc_min (the gate, e.g. 9.21), is ambiguous (-1) below assoc_max (the new-landmark threshold, e.g.
# 60), and otherwise opens a landmark. Combine it with OPT_WRAP_INNOVATION: an unwrapped bearing innovation near +-pi defeats any
# distance rule.
OPT_NEAREST_NEIGHBOUR = 8
# a step's measurements (at most 16 with unknown ids) associated jointly by joint compatibility branch and bound: the largest set of
# pairings, each landmark used once, whose stacked innovation passes chi2_{2p}^-1(1 - exp(-assoc_min / 2)); assoc_min is the individual
# chi-square gate at 2 dof (e.g. 9.21), assoc_max the new-landmark threshold. Excludes OPT_NEAREST_NEIGHBOUR, not in large-map mode;
# include/nuslam_b200.h NUSLAM_OPT_JOINT_COMPATIBILITY has the exact rule.
OPT_JOINT_COMPATIBILITY = 32


class NuslamError(RuntimeError):
    pass


class EkfConfig(C.Structure):
    _fields_ = [("n_landmarks", C.c_int32), ("mode", C.c_int32), ("Q", C.c_double * 9), ("R", C.c_double * 4),
                ("assoc_min", C.c_double), ("assoc_max", C.c_double), ("options", C.c_uint32), ("reserved", C.c_uint32),
                ("landmark_prior", C.c_double)]


_lib = None


def lib() -> C.CDLL:
    """Load the CUDA library; fail loudly when it is missing (no fallback exists)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise NuslamError(f"{LIB_PATH} is missing: build it with __graft_entry__.build() "
                              "(python -m shermbot_navigation_b200.build). There is no CPU fallback.")
        l = C.CDLL(str(LIB_PATH))
        l.nuslam_last_error.restype = C.c_char_p
        vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int32
        l.nuslam_ekf_default_config.argtypes = [C.POINTER(EkfConfig), i32]
        l.nuslam_ekf_default_config.restype = None
        l.nuslam_ekf_create.argtypes = [C.POINTER(EkfConfig), i64, C.c_int, vp, C.POINTER(vp)]
        l.nuslam_ekf_destroy.argtypes = [vp]
        l.nuslam_ekf_bind_state.argtypes = [vp, vp, vp, vp, vp]
        l.nuslam_ekf_device_pointers.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
        l.nuslam_ekf_init.argtypes = [vp, vp, vp, C.c_int]
        l.nuslam_ekf_set_state.argtypes = [vp, vp, vp, vp, vp, C.c_int]
        l.nuslam_ekf_get_state.argtypes = [vp, vp, vp, vp, vp, C.c_int]
        l.nuslam_ekf_predict.argtypes = [vp, vp, C.c_int]
        l.nuslam_ekf_associate.argtypes = [vp, vp, vp, C.c_int]
        l.nuslam_ekf_initialize_landmark.argtypes = [vp, vp, vp, C.c_int]
        l.nuslam_ekf_update.argtypes = [vp, vp, vp, C.c_int]
        l.nuslam_ekf_measurement_model.argtypes = [vp, vp, vp, vp, C.c_int]
        l.nuslam_ekf_step.argtypes = [vp, vp, vp, vp, i32, vp, C.c_int]
        l.nuslam_ekf_map_to_odom.argtypes = [vp, vp, vp, C.c_int]
        l.nuslam_world_step.argtypes = [vp, vp, vp, C.c_double, vp, i32, C.c_double, C.c_double, C.c_double, vp, vp, i64, C.c_int, C.c_int, vp]
        l.nuslam_ekf_scan_step.argtypes = [vp, vp, vp, C.c_double, C.c_double, i32, vp, vp, vp, C.c_int]
        l.nuslam_ekf_step_async.argtypes = [vp, vp, vp, vp, i32, vp]
        l.nuslam_scan_set_fit.argtypes = [C.c_int]
        l.nuslam_ekf_get_stream.argtypes = [vp, C.POINTER(vp)]
        l.nuslam_ekf_async_dry_run.argtypes = [vp, C.c_int]
        l.nuslam_ekf_set_ids.argtypes = [vp, vp, i32, C.c_int]
        l.nuslam_ekf_step_async_packed.argtypes = [vp, vp, i32, C.c_int, vp]
        l.nuslam_ekf_error_stats.argtypes = [vp, vp, vp, vp, vp, i32, vp]
        l.nuslam_scan_last_fallbacks.argtypes = [C.c_int]
        l.nuslam_ekf_wait_async.argtypes = [vp]
        l.nuslam_ekf_synchronize.argtypes = [vp]
        l.nuslam_cartesian2polar.argtypes = [vp, vp, i64, C.c_int, C.c_int, vp]
        l.nuslam_normalize_angle.argtypes = [vp, vp, i64, C.c_int, C.c_int, vp]
        l.nuslam_scan_detect.argtypes = [vp, i64, C.c_double, C.c_double, vp, vp, vp, vp, i32, C.c_int, C.c_int, vp]
        l.nuslam_classify_and_fit.argtypes = [vp, vp, vp, i64, vp, vp, C.c_int, C.c_int, vp]
        l.nuslam_diffdrive_step.argtypes = [vp, vp, vp, vp, i64, C.c_int, C.c_int, vp]
        l.nuslam_integrate_twist.argtypes = [vp, vp, i64, C.c_int, C.c_int, vp]
        l.nuslam_diffdrive_convert_twist.argtypes = [C.c_double, C.c_double, vp, vp, i64, C.c_int, C.c_int, vp]
        _lib = l
    return _lib


def _check(rc: int, what: str):
    if rc != 0:
        raise NuslamError(f"{what} failed (code {rc}): {lib().nuslam_last_error().decode()}")


def _is_torch(a) -> bool:
    return a is not None and type(a).__module__.startswith("torch")


def _ptr(a, dtype, mem_expected=None):
    """(pointer, keepalive, mem) for a numpy array / torch tensor / None."""
    if a is None:
        return None, None, mem_expected
    if _is_torch(a):
        import torch
        want = {np.float64: torch.float64, np.int32: torch.int32, np.float32: torch.float32, np.int16: torch.int16}[dtype]
        if a.dtype != want or not a.is_contiguous():
            raise NuslamError(f"tensor must be contiguous {want}")
        return a.data_ptr(), a, (NUSLAM_DEVICE if a.is_cuda else NUSLAM_HOST)
    arr = np.ascontiguousarray(a, dtype=dtype)
    return arr.ctypes.data, arr, NUSLAM_HOST


def _mem_of(*ptrs):
    mems = {p[2] for p in ptrs if p[0] is not None}
    if len(mems) > 1:
        raise NuslamError("all arrays of one call must live on the same side (all numpy or all CUDA tensors)")
    return mems.pop() if mems else NUSLAM_HOST


class BatchedExtendedKalman:
    """B independent ``slam_library::ExtendedKalman`` filters on one B200.

    ``assoc_min`` / ``assoc_max`` are associateLandmark's thresholds (0.01 / 60 in the reference). Under ``options`` with
    OPT_NEAREST_NEIGHBOUR, ``assoc_min`` is the gate of the nearest candidate and ``assoc_max`` the new-landmark threshold. Under
    OPT_JOINT_COMPATIBILITY, ``assoc_min`` is the individual chi-square gate (2 dof) that also fixes the joint thresholds, and
    ``assoc_max`` the new-landmark threshold; steps with unknown ids then take at most 16 measurements."""

    def __init__(self, robotState, mapState=None, Q=None, R=None, n_landmarks=None, mode="strict", device=0,
                 stream=None, assoc_min=0.01, assoc_max=60.0, options=0, landmark_prior=None):
        l = lib()
        robot = np.atleast_2d(np.asarray(robotState, dtype=np.float64))
        self.batch = robot.shape[0]
        if mapState is not None:
            mp = np.atleast_2d(np.asarray(mapState, dtype=np.float64))
            n_landmarks = mp.shape[1] // 2
            mp = np.ascontiguousarray(np.broadcast_to(mp, (self.batch, 2 * n_landmarks)))
        else:
            mp = None
        if n_landmarks is None:
            raise NuslamError("give mapState or n_landmarks")
        self.n = int(n_landmarks)
        self.len = 3 + 2 * self.n
        self.device = int(device)
        cfg = EkfConfig()
        l.nuslam_ekf_default_config(C.byref(cfg), self.n)
        cfg.mode = {"strict": MODE_STRICT, "fast": MODE_FAST, "large": MODE_LARGE}[mode]
        if Q is not None:
            cfg.Q[:] = list(np.asarray(Q, dtype=np.float64).reshape(3, 3).T.ravel())
        if R is not None:
            cfg.R[:] = list(np.asarray(R, dtype=np.float64).reshape(2, 2).T.ravel())
        cfg.assoc_min, cfg.assoc_max = float(assoc_min), float(assoc_max)
        cfg.options = int(options)   # OPT_* bit mask: opt-in departures from the reference, 0 = reference behaviour
        if landmark_prior is not None:
            cfg.landmark_prior = float(landmark_prior)
        self.mode = mode
        h = C.c_void_p()
        _check(l.nuslam_ekf_create(C.byref(cfg), self.batch, self.device, stream, C.byref(h)), "nuslam_ekf_create")
        self._h = h
        self._keep = None
        self.stream_ptr = stream   # the cudaStream_t the handle launches on when the caller supplied one (None: the handle's own stream)
        hs = C.c_void_p()
        _check(l.nuslam_ekf_get_stream(self._h, C.byref(hs)), "nuslam_ekf_get_stream")
        self._stream = hs.value or 0   # the stream every DEVICE call enqueues on
        robot = np.ascontiguousarray(robot)
        _check(l.nuslam_ekf_init(self._h, robot.ctypes.data, mp.ctypes.data if mp is not None else None, NUSLAM_HOST),
               "nuslam_ekf_init")

    # ---- stream ordering for CUDA-tensor arguments ----
    # A DEVICE call only enqueues work on the handle's stream. When that is not torch's current stream, the wrapper orders the two
    # with events: the handle's stream first waits for everything queued on torch's current stream (the producers of the argument
    # tensors), and torch's current stream afterwards waits for the call's kernels, so that tensors returned by the call (and the
    # state tensors of bind_state) can be used by ordinary torch code without a manual synchronize. No host synchronisation.
    def _order_begin(self, *args):
        tens = [a for a in args if _is_torch(a) and a.is_cuda]
        if not tens:
            return None
        import torch
        dev = tens[0].device
        cur = torch.cuda.current_stream(dev)
        if cur.cuda_stream == self._stream:
            return None   # same stream: program order
        hs = torch.cuda.ExternalStream(self._stream, device=dev)
        hs.wait_stream(cur)
        return cur, hs

    @staticmethod
    def _order_end(tok):
        if tok is not None:
            tok[0].wait_stream(tok[1])

    def close(self):
        if getattr(self, "_h", None):
            lib().nuslam_ekf_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- state ----
    def bind_state(self, x, sigma, seen, status):
        """Run on caller-owned CUDA tensors (x [B,len] f64, sigma [B,len,len] f64 holding column-major
        matrices, seen [B] i32, status [B] i32)."""
        _check(lib().nuslam_ekf_bind_state(self._h, x.data_ptr(), sigma.data_ptr(), seen.data_ptr(), status.data_ptr()),
               "nuslam_ekf_bind_state")
        self._keep = (x, sigma, seen, status)

    def set_state(self, x=None, sigma=None, seen=None, status=None):
        """sigma is [B,row,col]; transposed to the column-major wire format here."""
        if sigma is not None and not _is_torch(sigma):
            sigma = np.ascontiguousarray(np.transpose(np.asarray(sigma, dtype=np.float64).reshape(self.batch, self.len, self.len), (0, 2, 1)))
        px, ps = _ptr(x, np.float64), _ptr(sigma, np.float64)
        pn, pt = _ptr(seen, np.int32), _ptr(status, np.int32)
        tok = self._order_begin(x, sigma, seen, status)
        _check(lib().nuslam_ekf_set_state(self._h, px[0], ps[0], pn[0], pt[0], _mem_of(px, ps, pn, pt)), "nuslam_ekf_set_state")
        self._order_end(tok)

    def get_state(self):
        x = np.empty((self.batch, self.len))
        s = np.empty((self.batch, self.len, self.len))
        seen = np.empty(self.batch, dtype=np.int32)
        status = np.empty(self.batch, dtype=np.int32)
        _check(lib().nuslam_ekf_get_state(self._h, x.ctypes.data, s.ctypes.data, seen.ctypes.data, status.ctypes.data, NUSLAM_HOST),
               "nuslam_ekf_get_state")
        return x, np.transpose(s, (0, 2, 1)).copy(), seen, status

    def getStateVector(self, out=None):
        """Only x travels (B x len f64); pass a pinned numpy buffer as ``out`` to avoid an allocation per call."""
        x = out if out is not None else np.empty((self.batch, self.len))
        _check(lib().nuslam_ekf_get_state(self._h, x.ctypes.data, None, None, None, NUSLAM_HOST), "nuslam_ekf_get_state")
        return x

    def getCovariance(self):
        return self.get_state()[1]

    def getSeenLandmarks(self):
        seen = np.empty(self.batch, dtype=np.int32)
        _check(lib().nuslam_ekf_get_state(self._h, None, None, seen.ctypes.data, None, NUSLAM_HOST), "nuslam_ekf_get_state")
        return seen

    def getStatus(self):
        status = np.empty(self.batch, dtype=np.int32)
        _check(lib().nuslam_ekf_get_state(self._h, None, None, None, status.ctypes.data, NUSLAM_HOST), "nuslam_ekf_get_state")
        return status

    # ---- ExtendedKalman members, batched ----
    def predict(self, twists):
        p = _ptr(twists, np.float64)
        tok = self._order_begin(twists)
        _check(lib().nuslam_ekf_predict(self._h, p[0], p[2]), "nuslam_ekf_predict")
        self._order_end(tok)

    def associateLandmark(self, z):
        pz = _ptr(z, np.float64)
        if pz[2] == NUSLAM_DEVICE:
            import torch
            out = torch.empty(self.batch, dtype=torch.int32, device=z.device)
            tok = self._order_begin(z, out)
            _check(lib().nuslam_ekf_associate(self._h, pz[0], out.data_ptr(), NUSLAM_DEVICE), "nuslam_ekf_associate")
            self._order_end(tok)
            return out
        out = np.empty(self.batch, dtype=np.int32)
        _check(lib().nuslam_ekf_associate(self._h, pz[0], out.ctypes.data, NUSLAM_HOST), "nuslam_ekf_associate")
        return out

    def initializeLandmark(self, z, ids):
        pz, pi = _ptr(z, np.float64), _ptr(ids, np.int32)
        tok = self._order_begin(z, ids)
        _check(lib().nuslam_ekf_initialize_landmark(self._h, pz[0], pi[0], _mem_of(pz, pi)), "nuslam_ekf_initialize_landmark")
        self._order_end(tok)

    def update(self, z, ids, twists=None):
        """``twists`` is accepted for signature parity with update(tw, z, id) and ignored, as in the reference."""
        pz, pi = _ptr(z, np.float64), _ptr(ids, np.int32)
        tok = self._order_begin(z, ids)
        _check(lib().nuslam_ekf_update(self._h, pz[0], pi[0], _mem_of(pz, pi)), "nuslam_ekf_update")
        self._order_end(tok)

    def computeTheoreticalMeasurement(self, j):
        j = np.ascontiguousarray(np.broadcast_to(np.asarray(j, dtype=np.int32), (self.batch,)))
        out = np.zeros((self.batch, 2))
        _check(lib().nuslam_ekf_measurement_model(self._h, j.ctypes.data, out.ctypes.data, None, NUSLAM_HOST), "nuslam_ekf_measurement_model")
        return out

    def linearizedMeasurementModel(self, j):
        j = np.ascontiguousarray(np.broadcast_to(np.asarray(j, dtype=np.int32), (self.batch,)))
        out = np.zeros((self.batch, self.len, 2))
        _check(lib().nuslam_ekf_measurement_model(self._h, j.ctypes.data, None, out.ctypes.data, NUSLAM_HOST), "nuslam_ekf_measurement_model")
        return np.transpose(out, (0, 2, 1)).copy()

    def step(self, twists, z, ids=None, return_ids=False):
        """One iteration of EKFSlam::main_loop (slam.cpp:262-319). z: [B,m,2]; ids: [B,m] or None."""
        pt, pz, pi = _ptr(twists, np.float64), _ptr(z, np.float64), _ptr(ids, np.int32)
        mem = _mem_of(pt, pz, pi)
        m = int(z.shape[1]) if z is not None else 0
        out = None
        optr = None
        if return_ids:
            if mem == NUSLAM_DEVICE:
                import torch
                out = torch.empty((self.batch, m), dtype=torch.int32, device=z.device)
                optr = out.data_ptr()
            else:
                out = np.empty((self.batch, m), dtype=np.int32)
                optr = out.ctypes.data
        tok = self._order_begin(twists, z, ids, out)
        _check(lib().nuslam_ekf_step(self._h, pt[0], pz[0], pi[0], m, optr, mem), "nuslam_ekf_step")
        self._order_end(tok)
        return out

    def scan_step(self, twists, ranges, min_range, max_range, m, return_all=False):
        """Landmarks::main_loop (landmarks.cpp:84-109) -> cartesian2polar (slam.cpp:282-286) -> one EKFSlam::main_loop iteration with
        associateLandmark (slam.cpp:262-319), fused on the device: scan b feeds filter b. twists [B,3] f64, ranges [B,360] f32.
        With return_all: (n_markers [B], z [B,m,2], ids [B,m])."""
        pt, pr = _ptr(twists, np.float64), _ptr(ranges, np.float32)
        mem = _mem_of(pt, pr)
        outs, ptrs = (None, None, None), (None, None, None)
        if return_all:
            if mem == NUSLAM_DEVICE:
                import torch
                dev = ranges.device
                outs = (torch.empty((self.batch,), dtype=torch.int32, device=dev), torch.empty((self.batch, m, 2), dtype=torch.float64, device=dev),
                        torch.empty((self.batch, m), dtype=torch.int32, device=dev))
                ptrs = tuple(o.data_ptr() for o in outs)
            else:
                outs = (np.empty((self.batch,), np.int32), np.empty((self.batch, m, 2), np.float64), np.empty((self.batch, m), np.int32))
                ptrs = tuple(o.ctypes.data for o in outs)
        tok = self._order_begin(twists, ranges, *outs)
        _check(lib().nuslam_ekf_scan_step(self._h, pt[0], pr[0], float(min_range), float(max_range), int(m), ptrs[0], ptrs[1], ptrs[2], mem),
               "nuslam_ekf_scan_step")
        self._order_end(tok)
        return outs if return_all else None

    def map_to_odom(self, odom_state7):
        """EKFSlam::broadcast_map2odom_tf (slam.cpp:175-210) for every filter: [B,3] = (tx, ty, yaw) of map -> odom, from the filter's
        estimate and the odometry model's state rows {wheelBase, wheelRad, x, y, th, thL, thR}."""
        po = _ptr(odom_state7, np.float64)
        if po[2] == NUSLAM_DEVICE:
            import torch
            out = torch.empty((self.batch, 3), dtype=torch.float64, device=odom_state7.device)
            optr = out.data_ptr()
        else:
            out = np.empty((self.batch, 3))
            optr = out.ctypes.data
        tok = self._order_begin(odom_state7, out)
        _check(lib().nuslam_ekf_map_to_odom(self._h, po[0], optr, po[2]), "nuslam_ekf_map_to_odom")
        self._order_end(tok)
        return out

    STATS = ("sq_position_error", "sq_heading_error", "nees", "filters", "sq_landmark_error", "landmarks", "bad_status", "id_mismatches")

    def error_stats(self, truth_pose=None, truth_map=None, ids_got=None, ids_want=None):
        """K6: error statistics of this shard against a ground truth, reduced on the device (nuslam_ekf_error_stats): a CUDA tensor
        of 8 SUMS (see ``STATS``) that the ranks add up with one NCCL all-reduce. All arguments are CUDA tensors (or None)."""
        import torch
        dev = torch.device("cuda", self.device)
        out = torch.zeros(8, dtype=torch.float64, device=dev)
        m = int(ids_got.shape[1]) if ids_got is not None else 0
        ptr = lambda t: t.data_ptr() if t is not None else None
        for t, dt in ((truth_pose, torch.float64), (truth_map, torch.float64), (ids_got, torch.int32), (ids_want, torch.int32)):
            if t is not None and (t.dtype != dt or not t.is_cuda or not t.is_contiguous()):
                raise NuslamError(f"error_stats takes contiguous CUDA tensors ({dt})")
        tok = self._order_begin(out, truth_pose, truth_map, ids_got, ids_want)
        _check(lib().nuslam_ekf_error_stats(self._h, ptr(truth_pose), ptr(truth_map), ptr(ids_got), ptr(ids_want), m, out.data_ptr()),
               "nuslam_ekf_error_stats")
        self._order_end(tok)
        return out

    def step_async(self, twists, z, ids, x_out):
        """Pipelined host-buffer step (nuslam_ekf_step_async): numpy views of page-locked buffers; ``x_out`` [B,len] receives the state
        vector once the step has left the pipeline (three calls later, or after ``wait_async``)."""
        for a, dt in ((twists, np.float64), (z, np.float64), (ids, np.int32), (x_out, np.float64)):
            if a is None and dt == np.int32:
                continue   # unknown correspondence: associateLandmark on the device
            if not (isinstance(a, np.ndarray) and a.dtype == dt and a.flags["C_CONTIGUOUS"]):
                raise NuslamError("step_async takes contiguous numpy arrays of the exact dtype (no hidden copies in a pipelined call)")
        _check(lib().nuslam_ekf_step_async(self._h, twists.ctypes.data, z.ctypes.data, ids.ctypes.data if ids is not None else None, int(z.shape[1]),
                                           x_out.ctypes.data),
               "nuslam_ekf_step_async")

    IDS_NONE, IDS_PACKED, IDS_CACHED = 0, 1, 2   # NUSLAM_IDS_* of include/nuslam_b200.h

    def set_ids(self, ids):
        """Keep the [B,m] known-correspondence ids on the device for ``step_async_packed(..., ids_mode=IDS_CACHED)``."""
        p = _ptr(ids, np.int32)
        tok = self._order_begin(ids)
        _check(lib().nuslam_ekf_set_ids(self._h, p[0], int(ids.shape[1]), p[2]), "nuslam_ekf_set_ids")
        self._order_end(tok)

    def packed_layout(self, m, with_ids):
        """(total bytes, offset of z, offset of ids) of the packed host buffer of ``step_async_packed``: [twists B x 3 f64][z B x m x 2 f64]
        [ids B x m i32 when with_ids]."""
        b_tw, b_z = 8 * 3 * self.batch, 8 * 2 * self.batch * m
        return b_tw + b_z + (4 * self.batch * m if with_ids else 0), b_tw, b_tw + b_z

    def step_async_packed(self, packed, m, ids_mode, x_out):
        """Pipelined host-buffer step from ONE page-locked buffer (a uint8 numpy view laid out by ``packed_layout``), one host -> device
        copy per step (nuslam_ekf_step_async_packed)."""
        if not (isinstance(packed, np.ndarray) and packed.dtype == np.uint8 and packed.flags["C_CONTIGUOUS"]):
            raise NuslamError("step_async_packed takes a contiguous uint8 numpy view of the packed buffer")
        need = self.packed_layout(m, ids_mode == self.IDS_PACKED)[0]
        if packed.size < need:
            raise NuslamError(f"packed buffer holds {packed.size} bytes, the step needs {need}")
        _check(lib().nuslam_ekf_step_async_packed(self._h, packed.ctypes.data, int(m), int(ids_mode), x_out.ctypes.data), "nuslam_ekf_step_async_packed")

    def async_dry_run(self, on: bool):
        """Measurement aid: while on, step_async performs its copies and stream hand-overs without launching kernels (copy ceiling)."""
        _check(lib().nuslam_ekf_async_dry_run(self._h, 1 if on else 0), "nuslam_ekf_async_dry_run")

    def wait_async(self):
        _check(lib().nuslam_ekf_wait_async(self._h), "nuslam_ekf_wait_async")

    def synchronize(self):
        _check(lib().nuslam_ekf_synchronize(self._h), "nuslam_ekf_synchronize")


def cartesian2polar(xy, device=0):
    """slam_library::cartesian2polar (slam_library.cpp:16-22), batched: [N,2] -> [N,2]."""
    if _is_torch(xy) and xy.is_cuda:
        import torch
        out = torch.empty_like(xy)
        _check(lib().nuslam_cartesian2polar(xy.data_ptr(), out.data_ptr(), xy.shape[0], NUSLAM_DEVICE, xy.device.index, None), "nuslam_cartesian2polar")
        torch.cuda.synchronize(xy.device)
        return out
    a = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1, 2)
    out = np.empty_like(a)
    _check(lib().nuslam_cartesian2polar(a.ctypes.data, out.ctypes.data, a.shape[0], NUSLAM_HOST, device, None), "nuslam_cartesian2polar")
    return out


def normalize_angle(rad, device=0):
    """rigid2d::normalize_angle (rigid2d.cpp:9-13), batched."""
    a = np.ascontiguousarray(rad, dtype=np.float64).ravel()
    out = np.empty_like(a)
    _check(lib().nuslam_normalize_angle(a.ctypes.data, out.ctypes.data, a.shape[0], NUSLAM_HOST, device, None), "nuslam_normalize_angle")
    return out.reshape(np.shape(rad))
