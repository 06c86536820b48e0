"""oracle -- TEST INFRASTRUCTURE ONLY.

CPU checker for the CUDA EKF-SLAM / circle-fit path. Two interchangeable libraries implement
``oracle/oracle_api.h``:

* ``load("ref")``  -> ``oracle/_ref/libnuslam_ref.so``: the UNMODIFIED reference sources
  (``nuslam/src/{slam_library,circle_fit_library}.cpp`` and ``rigid2d/src/{rigid2d,diff_drive}.cpp``
  of a checkout of sziselman/Shermbot-Navigation) compiled where they lie against
  ``oracle/shim/`` (Armadillo + ROS message stand-ins).  Built only where such a checkout is found
  (``reference_dir()``: ``$NUSLAM_REFERENCE``, else oracle/Makefile's default ``REF``); the reference is
  not part of this repository.
* ``load("port")`` -> ``oracle/libnuslam_oracle.so``: the plain-C restatement (``nuslam_oracle.c``).

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this package.  Nothing under ``shermbot-navigation_b200/`` does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ORC_EXC = -1000
ORC_UB = -2000

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_fp = C.POINTER(C.c_float)
_sp = C.POINTER(C.c_short)


def reference_dir() -> Path | None:
    """The checkout of the reference project that oracle/Makefile builds oracle/_ref from (its REF: $NUSLAM_REFERENCE, else the
    Makefile's default), if it exists and can be read (os.path.isdir is False, not an error, for a path the user may not stat)."""
    out = subprocess.run(["make", "-s", "--no-print-directory", "-C", str(HERE), "print-ref"], capture_output=True, text=True)
    d = out.stdout.strip()
    return Path(d) if out.returncode == 0 and d and os.path.isdir(d) else None


def build(verbose: bool = False) -> None:
    """Compile the C restatement and, when reference_dir() is set, oracle/_ref."""
    out = subprocess.run(["make", "-C", str(HERE), "all"], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout, out.stderr)
    if out.returncode != 0:
        raise RuntimeError("oracle build failed")
    # the reference's own circle-fit test against the B200 facade (needs reference_dir() and the built CUDA library; a no-op otherwise)
    out = subprocess.run(["make", "-C", str(HERE), "facade_tests"], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout, out.stderr)
    if out.returncode != 0:
        raise RuntimeError("facade_tests build failed")


def lib_path(kind: str) -> Path:
    return {"ref": HERE / "_ref" / "libnuslam_ref.so", "port": HERE / "libnuslam_oracle.so", "ref_blas": HERE / "_ref" / "libnuslam_ref_blas.so",
            "ref_det": HERE / "_ref" / "libnuslam_ref_det.so", "port_det": HERE / "libnuslam_oracle_det.so"}[kind]


def available(kind: str) -> bool:
    return lib_path(kind).exists()


def _d(a):
    return a.ctypes.data_as(_dp)


def _i(a):
    return a.ctypes.data_as(_ip)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class Ekf:
    """One reference filter (slam_library::ExtendedKalman). Matrices are column-major on the C side;
    ``sigma`` is returned as a (len, len) numpy array indexed [row, col]."""

    def __init__(self, lib, n, robot, mapstate, Q, R):
        self._l = lib
        self.n = int(n)
        self.len = 3 + 2 * self.n
        robot = _f64(robot)
        mapstate = _f64(mapstate)
        Qc = _f64(np.asarray(Q, dtype=np.float64).reshape(3, 3).T)  # column-major bytes
        Rc = _f64(np.asarray(R, dtype=np.float64).reshape(2, 2).T)
        self._h = lib._c.orc_ekf_new(self.n, _d(robot), _d(mapstate), _d(Qc), _d(Rc))

    def __del__(self):
        if getattr(self, "_h", None):
            self._l._c.orc_ekf_free(self._h)
            self._h = None

    def predict(self, dth, dx, dy=0.0):
        self._l._c.orc_ekf_predict(self._h, float(dth), float(dx), float(dy))

    def associate(self, z):
        z = _f64(z)
        return int(self._l._c.orc_ekf_associate(self._h, _d(z)))

    def init_landmark(self, z, idx):
        z = _f64(z)
        self._l._c.orc_ekf_init_landmark(self._h, _d(z), int(idx))

    def update(self, z, idx):
        z = _f64(z)
        return int(self._l._c.orc_ekf_update(self._h, _d(z), int(idx)))

    def get(self):
        x = np.empty(self.len)
        s = np.empty((self.len, self.len))
        seen = C.c_int(0)
        self._l._c.orc_ekf_get(self._h, _d(x), _d(s), C.byref(seen))
        return x, s.T.copy(), seen.value  # column-major bytes -> [row, col]

    def set(self, x, sigma, seen):
        x = _f64(x)
        s = _f64(np.asarray(sigma, dtype=np.float64).T)
        self._l._c.orc_ekf_set(self._h, _d(x), _d(s), int(seen))

    def zhat(self, j):
        out = np.empty(2)
        self._l._c.orc_ekf_zhat(self._h, int(j), _d(out))
        return out

    def H(self, j):
        out = np.empty((self.len, 2))
        self._l._c.orc_ekf_H(self._h, int(j), _d(out))
        return out.T.copy()


class OracleLib:
    def __init__(self, kind: str):
        p = lib_path(kind)
        if not p.exists():
            raise FileNotFoundError(f"oracle library {p} missing: run oracle.build()")
        self.kind = kind
        self._c = c = C.CDLL(str(p))
        c.orc_flavour.restype = C.c_char_p
        c.orc_eig_sym_full_sweeps.argtypes = [C.c_int]
        c.orc_eig_sym_full_sweeps.restype = C.c_int
        c.orc_ekf_new.restype = C.c_void_p
        c.orc_ekf_new.argtypes = [C.c_int, _dp, _dp, _dp, _dp]
        c.orc_ekf_free.argtypes = [C.c_void_p]
        c.orc_ekf_predict.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double]
        c.orc_ekf_associate.argtypes = [C.c_void_p, _dp]
        c.orc_ekf_init_landmark.argtypes = [C.c_void_p, _dp, C.c_int]
        c.orc_ekf_update.argtypes = [C.c_void_p, _dp, C.c_int]
        c.orc_ekf_get.argtypes = [C.c_void_p, _dp, _dp, _ip]
        c.orc_ekf_set.argtypes = [C.c_void_p, _dp, _dp, C.c_int]
        c.orc_ekf_zhat.argtypes = [C.c_void_p, C.c_int, _dp]
        c.orc_ekf_H.argtypes = [C.c_void_p, C.c_int, _dp]
        c.orc_cartesian2polar.argtypes = [C.c_double, C.c_double, _dp]
        c.orc_normalize_angle.restype = C.c_double
        c.orc_normalize_angle.argtypes = [C.c_double]
        c.orc_diffdrive_convert_twist.argtypes = [C.c_double] * 4 + [_dp]
        c.orc_diffdrive_step.argtypes = [_dp, C.c_double, C.c_double, _dp]
        c.orc_integrate_twist.argtypes = [C.c_double] * 3 + [_dp]
        c.orc_ekf_run.argtypes = [C.c_int, C.c_long, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, _ip,
                                  _dp, _dp, _ip, _ip, _ip, _dp, C.c_int, C.c_int]
        c.orc_cluster_points.argtypes = [_fp, C.c_double, C.c_double, _ip, _ip, _dp, _dp]
        c.orc_classify_cluster.argtypes = [_dp, _dp, C.c_int]
        c.orc_circle_fit.argtypes = [_dp, _dp, C.c_int, _dp]
        c.orc_scan_detect.argtypes = [_fp, C.c_double, C.c_double, _ip, _ip, _dp, C.c_int]
        c.orc_scan_detect_batch.argtypes = [C.c_long, _fp, C.c_double, C.c_double, _sp, _ip, _ip, _dp, C.c_int, C.c_int]
        c.orc_map_to_odom.restype = None
        c.orc_map_to_odom.argtypes = [_dp, _dp, _dp]
        c.orc_world_step_batch.restype = None
        c.orc_world_step_batch.argtypes = [C.c_long, _dp, _dp, _dp, C.c_double, _dp, C.c_int, C.c_double, C.c_double, C.c_double, _fp]

    @property
    def flavour(self) -> str:
        return self._c.orc_flavour().decode()

    def eig_sym_full_sweeps(self, on: bool) -> bool:
        """Test hook of the "ref" flavour: True = the shim's eig_sym runs to its criterion / 100-sweep cap instead of stopping at the fixed
        point of its outputs (bit-identical results, tests/test_oracle.py). Returns the previous setting."""
        return bool(self._c.orc_eig_sym_full_sweeps(1 if on else 0))

    # ---- EKF ----
    def ekf(self, n, robot, mapstate, Q, R) -> Ekf:
        return Ekf(self, n, robot, mapstate, Q, R)

    def cartesian2polar(self, x, y):
        out = np.empty(2)
        self._c.orc_cartesian2polar(float(x), float(y), _d(out))
        return out

    def normalize_angle(self, r):
        return float(self._c.orc_normalize_angle(float(r)))

    def convert_twist(self, base, rad, dth, dx):
        out = np.empty(2)
        self._c.orc_diffdrive_convert_twist(base, rad, dth, dx, _d(out))
        return out

    def diffdrive_step(self, state7, thL, thR):
        s = _f64(state7).copy()
        tw = np.empty(3)
        self._c.orc_diffdrive_step(_d(s), float(thL), float(thR), _d(tw))
        return s, tw

    def integrate_twist(self, dth, dx, dy):
        out = np.empty(4)
        self._c.orc_integrate_twist(float(dth), float(dx), float(dy), _d(out))
        return out

    def ekf_run(self, n, robot0, map0, Q, R, twists, z, ids=None, init=None, trace=False, nthreads=1):
        """Batch driver (slam.cpp:262-319). twists (T,B,3); z (T,B,m,2); ids (T,B,m) int32 or None.
        init = (x (B,len), sigma (B,len,len)[row,col], seen (B,)) to start from a given state.
        Returns dict(x, sigma[row,col], seen, status, ids_out, trace)."""
        twists = _f64(twists)
        z = _f64(z)
        T, B, m = z.shape[0], z.shape[1], z.shape[2]
        ln = 3 + 2 * n
        robot0 = _f64(np.broadcast_to(robot0, (B, 3)))
        map0 = _f64(np.broadcast_to(map0, (B, 2 * n)))
        Qc = _f64(np.asarray(Q, dtype=np.float64).reshape(3, 3).T)
        Rc = _f64(np.asarray(R, dtype=np.float64).reshape(2, 2).T)
        x = np.zeros((B, ln))
        s = np.zeros((B, ln, ln))
        seen = np.zeros(B, dtype=np.int32)
        if init is not None:
            x[:] = init[0]
            s[:] = np.transpose(np.asarray(init[1]), (0, 2, 1))
            seen[:] = init[2]
        status = np.zeros(B, dtype=np.int32)
        ids_out = np.zeros((T, B, m), dtype=np.int32)
        tr = np.zeros((T, B, ln)) if trace else None
        idp = None
        if ids is not None:
            ids = np.ascontiguousarray(ids, dtype=np.int32)
            idp = _i(ids)
        self._c.orc_ekf_run(n, B, T, m, _d(robot0), _d(map0), _d(Qc), _d(Rc), _d(twists), _d(z), idp,
                            _d(x), _d(s), _i(seen), _i(status), _i(ids_out),
                            _d(tr) if trace else None, 1 if init is not None else 0, int(nthreads))
        return dict(x=x, sigma=np.transpose(s, (0, 2, 1)).copy(), seen=seen, status=status, ids_out=ids_out, trace=tr)

    def ekf_stepper(self, n, robot0, map0, Q, R, nthreads=1):
        """A persistent batch of B reference filters advanced one slam.cpp:262-319 iteration per call, state kept in the library's own
        layout between calls (no per-step copies or transposes on the Python side): what bench.py's reference arm times."""
        return _Stepper(self, n, robot0, map0, Q, R, nthreads)

    def map_to_odom(self, odom3, est3):
        """EKFSlam::broadcast_map2odom_tf (slam.cpp:175-210): (tx, ty, yaw) of the map -> odom transform."""
        o, e, out = _f64(odom3), _f64(est3), np.empty(3)
        self._c.orc_map_to_odom(_d(o), _d(e), _d(out))
        return out

    # ---- simulator slice ----
    def world_step(self, world, cmd, noise, dt, tubes, tube_rad, robot_rad, max_range):
        """One TubeWorld::main_loop iteration per robot (tube_world.cpp:512-537). world (B,9) is updated IN PLACE;
        returns the scans (B,360) float32."""
        assert world.dtype == np.float64 and world.flags["C_CONTIGUOUS"]
        B = world.shape[0]
        cmd = _f64(np.broadcast_to(cmd, (B, 3)))
        tubes = _f64(tubes)
        nz = None if noise is None else _f64(np.broadcast_to(noise, (B, 4)))
        ranges = np.empty((B, 360), dtype=np.float32)
        self._c.orc_world_step_batch(B, _d(world), _d(cmd), _d(nz) if nz is not None else None, float(dt), _d(tubes),
                                     int(tubes.shape[0]), float(tube_rad), float(robot_rad), float(max_range),
                                     ranges.ctypes.data_as(_fp))
        return ranges

    # ---- circle path ----
    def cluster_points(self, ranges, min_range, max_range):
        """Returns list of (beams int array, points (N,2)) or ORC_UB."""
        r = np.ascontiguousarray(ranges, dtype=np.float32)
        assert r.shape == (360,)
        off = np.zeros(362, dtype=np.int32)
        beams = np.zeros(362, dtype=np.int32)
        px = np.zeros(362)
        py = np.zeros(362)
        nc = self._c.orc_cluster_points(r.ctypes.data_as(_fp), float(min_range), float(max_range), _i(off), _i(beams), _d(px), _d(py))
        if nc < 0:
            return nc
        out = []
        for c in range(nc):
            a, b = off[c], off[c + 1]
            out.append((beams[a:b].copy(), np.stack([px[a:b], py[a:b]], axis=1)))
        return out

    def classify_cluster(self, pts):
        pts = _f64(pts)
        px = _f64(pts[:, 0])
        py = _f64(pts[:, 1])
        return bool(self._c.orc_classify_cluster(_d(px), _d(py), len(px)))

    def circle_fit(self, pts):
        """Returns (marker.id, cx, cy, R) with R = scale.x / 2."""
        pts = _f64(pts)
        px = _f64(pts[:, 0])
        py = _f64(pts[:, 1])
        out = np.zeros(3)
        mid = self._c.orc_circle_fit(_d(px), _d(py), len(px), _d(out))
        return mid, out[0], out[1], out[2]

    def scan_detect_batch(self, ranges, min_range, max_range, kmax=16, nthreads=1):
        r = np.ascontiguousarray(ranges, dtype=np.float32).reshape(-1, 360)
        S = r.shape[0]
        cob = np.zeros((S, 360), dtype=np.int16)
        ncl = np.zeros(S, dtype=np.int32)
        nci = np.zeros(S, dtype=np.int32)
        circ = np.zeros((S, kmax, 4))
        self._c.orc_scan_detect_batch(S, r.ctypes.data_as(_fp), float(min_range), float(max_range),
                                      cob.ctypes.data_as(_sp), _i(ncl), _i(nci), _d(circ), kmax, int(nthreads))
        return dict(cluster_of_beam=cob, n_clusters=ncl, n_circles=nci, circles=circ)


class _Stepper:
    def __init__(self, lib, n, robot0, map0, Q, R, nthreads):
        self.lib, self.n, self.nthreads = lib, int(n), int(nthreads)
        self.robot0 = _f64(np.atleast_2d(robot0))
        self.B = self.robot0.shape[0]
        ln = 3 + 2 * self.n
        self.map0 = _f64(np.broadcast_to(map0, (self.B, 2 * self.n)))
        self.Qc = _f64(np.asarray(Q, dtype=np.float64).reshape(3, 3).T)
        self.Rc = _f64(np.asarray(R, dtype=np.float64).reshape(2, 2).T)
        self.x = np.zeros((self.B, ln))
        self.s = np.zeros((self.B, ln, ln))   # the library's layout (column-major per filter)
        self.seen = np.zeros(self.B, dtype=np.int32)
        self.status = np.zeros(self.B, dtype=np.int32)
        self.started = False

    def step(self, twists, z, ids):
        """twists (B,3) f64, z (B,m,2) f64, ids (B,m) int32: all C-contiguous."""
        assert twists.flags["C_CONTIGUOUS"] and z.flags["C_CONTIGUOUS"] and ids.flags["C_CONTIGUOUS"] and ids.dtype == np.int32
        m = z.shape[1]
        self.lib._c.orc_ekf_run(self.n, self.B, 1, m, _d(self.robot0), _d(self.map0), _d(self.Qc), _d(self.Rc), _d(twists), _d(z), _i(ids),
                                _d(self.x), _d(self.s), _i(self.seen), _i(self.status), None, None, 1 if self.started else 0, self.nthreads)
        self.started = True


class TubeWorldRef:
    """oracle/_ref/libtube_world_ref.so: the UNMODIFIED simulator node nuturtlesim/src/tube_world.cpp, compiled against the roscpp
    stand-ins of oracle/shim_ros and driven by oracle/tube_world_driver.cpp. Pins oracle/world_oracle.h (tests/test_oracle.py)."""

    PATH = HERE / "_ref" / "libtube_world_ref.so"

    def __init__(self):
        if not self.PATH.exists():
            raise FileNotFoundError(f"{self.PATH} missing: run oracle.build() where reference_dir() finds the reference")
        self._c = c = C.CDLL(str(self.PATH))
        c.twref_flavour.restype = C.c_char_p
        c.twref_lidar.argtypes = [C.c_double, C.c_double, C.c_double, _dp, C.c_double, C.c_double, _fp]
        c.twref_run.argtypes = [C.c_int, _dp, C.c_double, C.c_double, C.c_double, _dp, C.c_double, C.c_double, C.c_double, _dp, _dp, _fp, _dp]

    @staticmethod
    def available() -> bool:
        return TubeWorldRef.PATH.exists()

    def lidar(self, x, y, th, tubes6, tube_rad, max_scan_range):
        """TubeWorld::simulate_lidar_scanner (tube_world.cpp:405-471) at robot configuration (x, y, th): 360 float ranges."""
        tubes = _f64(tubes6)
        assert tubes.shape == (6, 2)
        out = np.empty(360, dtype=np.float32)
        rc = self._c.twref_lidar(float(x), float(y), float(th), _d(tubes), float(tube_rad), float(max_scan_range), out.ctypes.data_as(_fp))
        assert rc == 0
        return out

    def run(self, cmd, wheel_base, wheel_rad, slip, tubes6, tube_rad, robot_rad, max_scan_range):
        """TubeWorld::main_loop (tube_world.cpp:473-544) for the T commanded twists `cmd` (T,3) from the origin, noise-free (the node's
        generator is seeded from random_device): returns poses (T,3) = (x, y, th), joints (T,2), scans (T,360), dt."""
        cmd = _f64(cmd)
        tubes = _f64(tubes6)
        T = cmd.shape[0]
        poses, joints, scans, dt = np.empty((T, 3)), np.empty((T, 2)), np.empty((T, 360), dtype=np.float32), np.zeros(1)
        rc = self._c.twref_run(T, _d(cmd), float(wheel_base), float(wheel_rad), float(slip), _d(tubes), float(tube_rad), float(robot_rad),
                               float(max_scan_range), _d(poses), _d(joints), scans.ctypes.data_as(_fp), _d(dt))
        assert rc == 0
        return poses, joints, scans, float(dt[0])


_cache: dict[str, OracleLib] = {}


def load(kind: str = "port") -> OracleLib:
    if kind not in _cache:
        _cache[kind] = OracleLib(kind)
    return _cache[kind]


def best() -> OracleLib:
    """The compiled reference when it exists (pins parity), else the restatement."""
    return load("ref") if available("ref") else load("port")
