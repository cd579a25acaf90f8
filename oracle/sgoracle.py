"""ctypes binding of the CPU oracle (oracle/libsgoracle.so) -- TEST INFRASTRUCTURE ONLY.

Only tests/, ``__graft_entry__.smoke()`` and bench.py's ``cpu_baseline`` / ``--impl reference`` legs may
import this module; the product package never does (see oracle/sg_oracle.c header).  PARITY UNPINNED:
the reference ships no golden vectors for this path and MuJoCo is not installable here.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

ST_DIVERGED, ST_CON_FULL, ST_EFC_FULL, ST_UNSUPPORTED = 1, 2, 4, 8


def build(force=False):
    so = os.path.join(_HERE, "libsgoracle.so")
    src = os.path.join(_HERE, "sg_oracle.c")
    if force or not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-B", "libsgoracle.so"], stdout=subprocess.DEVNULL)
    return so


def build_native(out_dir):
    """-O3 -march=native build for the CPU arm of bench.py, compiled on the box it runs on into `out_dir` (the source tree
    may be read-only), falling back to the portable build when the compiler is missing; same arithmetic, same results.
    Returns the library's path.  The parent process builds it once before it starts its workers; the workers only load it."""
    so = os.path.join(os.path.abspath(out_dir), "libsgoracle_native.so")
    try:
        subprocess.check_call(["make", "-C", _HERE, "-B", "NATIVE=" + so, so], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        return so
    except Exception:
        return build()


def use_native(path):
    """Switch this process to the library at `path`, as returned by build_native (call before the first lib())."""
    global _NATIVE
    if _LIB is None:
        _NATIVE = path


_NATIVE = None


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(_NATIVE or build())
        P, D, I = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int)
        L.sgo_model_load.restype = P
        L.sgo_model_load.argtypes = [C.c_char_p, C.c_size_t]
        L.sgo_model_free.argtypes = [P]
        L.sgo_model_int.argtypes = [P, C.c_char_p]
        L.sgo_world_create.restype = P
        L.sgo_world_create.argtypes = [P]
        L.sgo_world_free.argtypes = [P]
        for f in ("sgo_set_jnt_stiffness", "sgo_set_tendon_stiffness", "sgo_set_dof_damping", "sgo_set_tendon_damping"):
            getattr(L, f).argtypes = [P, C.c_int, C.c_double]
        L.sgo_set_body_pos.argtypes = [P, C.c_int, D]
        L.sgo_set_ctrl.argtypes = [P, D]
        L.sgo_set_dense_solver.argtypes = [P, C.c_int]
        L.sgo_set_capsule_box_single.argtypes = [P, C.c_int]
        L.sgo_set_implicit_tendon_damping.argtypes = [P, C.c_int]
        L.sgo_set_geom_mask.argtypes = [P, I]
        L.sgo_reset.argtypes = [P]
        L.sgo_forward.argtypes = [P]
        L.sgo_step.argtypes = [P]
        L.sgo_status.argtypes = [P]
        L.sgo_get_state.argtypes = [P, D, D, D, D]
        L.sgo_set_state.argtypes = [P, D, D, D, D]
        L.sgo_get_sensordata.argtypes = [P, D]
        L.sgo_get_touch_mask.argtypes = [P]
        L.sgo_get_int.argtypes = [P, C.c_char_p]
        L.sgo_get_array.argtypes = [P, C.c_char_p, D, C.c_int]
        L.sgo_episode.argtypes = [P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, D, I]
        L.sgo_last_step_flops.restype = C.c_double
        L.sgo_last_step_flops.argtypes = [P]
        L.sgo_flops_get.argtypes = [P, D]
        L.sgo_flops_reset.argtypes = [P]
        L.sgo_test_capsule_box.argtypes = [D, D, D, D, D, D, D]
        L.sgo_test_sphere_box.argtypes = [D, C.c_double, D, D, D, D]
        L.sgo_test_qcqp2.argtypes = [D, D, D, C.c_double, D]
        L.sgo_test_impedance.restype = C.c_double
        L.sgo_test_impedance.argtypes = [D, C.c_double, C.c_double]
        L.sgo_test_box_box.argtypes = [D, D, D, D, D, D]
        L.sgo_test_make_frame.argtypes = [D]
        _LIB = L
    return _LIB


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


class OracleModel:
    def __init__(self, blob: bytes):
        self._L = lib()
        self._blob = bytes(blob)
        self.h = self._L.sgo_model_load(self._blob, len(self._blob))
        if not self.h:
            raise ValueError("oracle could not parse the model blob")
        for k in ("nv", "nbody", "ngeom", "neq", "nu", "nsensordata", "ntendon", "njnt", "npair", "nsite", "nM"):
            setattr(self, k, self._L.sgo_model_int(self.h, k.encode()))

    def __del__(self):
        if getattr(self, "h", None):
            self._L.sgo_model_free(self.h)
            self.h = None


class OracleWorld:
    """One fp64 world (the mjData of a single ManEnv)."""

    def __init__(self, model: OracleModel):
        self.m = model
        self._L = lib()
        self.h = self._L.sgo_world_create(model.h)

    def __del__(self):
        if getattr(self, "h", None):
            self._L.sgo_world_free(self.h)
            self.h = None

    # parameters ------------------------------------------------------------------------
    def set_stiffness(self, k, joint_ids=range(11, 64), tendon_ids=(0,)):
        """ManEnv.set_new_stiffness (ref: environment/manenv.py:103-109)."""
        for j in joint_ids:
            self._L.sgo_set_jnt_stiffness(self.h, int(j), float(k))
        for t in tendon_ids:
            self._L.sgo_set_tendon_stiffness(self.h, int(t), float(k))

    def set_jnt_stiffness(self, j, k): self._L.sgo_set_jnt_stiffness(self.h, int(j), float(k))
    def set_tendon_stiffness(self, t, k): self._L.sgo_set_tendon_stiffness(self.h, int(t), float(k))
    def set_dof_damping(self, i, v): self._L.sgo_set_dof_damping(self.h, int(i), float(v))
    def set_tendon_damping(self, t, v): self._L.sgo_set_tendon_damping(self.h, int(t), float(v))

    def set_body_pos(self, b, xyz):
        a = np.ascontiguousarray(xyz, dtype=np.float64)
        self._L.sgo_set_body_pos(self.h, int(b), _dp(a))

    def set_ctrl(self, ctrl):
        a = np.ascontiguousarray(ctrl, dtype=np.float64)
        assert a.shape[0] == self.m.nu
        self._L.sgo_set_ctrl(self.h, _dp(a))

    def set_dense_solver(self, on): self._L.sgo_set_dense_solver(self.h, int(on))
    def set_capsule_box_single(self, on): self._L.sgo_set_capsule_box_single(self.h, int(on))
    def set_implicit_tendon_damping(self, on): self._L.sgo_set_implicit_tendon_damping(self.h, int(on))

    def set_geom_mask(self, mask):
        a = np.ascontiguousarray(mask, dtype=np.int32)
        assert a.shape[0] == self.m.ngeom
        self._L.sgo_set_geom_mask(self.h, a.ctypes.data_as(C.POINTER(C.c_int)))

    # stepping ---------------------------------------------------------------------------
    def reset(self): self._L.sgo_reset(self.h)
    def forward(self): self._L.sgo_forward(self.h)
    def step(self): return self._L.sgo_step(self.h)
    def status(self): return self._L.sgo_status(self.h)

    def get_state(self):
        nv, nu = self.m.nv, self.m.nu
        q, v, a, w = np.zeros(nv), np.zeros(nv), np.zeros(nu), np.zeros(nv)
        self._L.sgo_get_state(self.h, _dp(q), _dp(v), _dp(a), _dp(w))
        return q, v, a, w

    def set_state(self, qpos=None, qvel=None, act=None, warm=None):
        arrs = [None if x is None else np.ascontiguousarray(x, dtype=np.float64) for x in (qpos, qvel, act, warm)]
        self._L.sgo_set_state(self.h, *[_dp(x) for x in arrs])

    def sensordata(self):
        out = np.zeros(self.m.nsensordata)
        self._L.sgo_get_sensordata(self.h, _dp(out))
        return out

    def touch_mask(self): return self._L.sgo_get_touch_mask(self.h)
    def get_int(self, key): return self._L.sgo_get_int(self.h, key.encode())

    def get(self, key):
        n = self._L.sgo_get_array(self.h, key.encode(), None, 0)
        if n < 0:
            raise KeyError(key)
        out = np.zeros(max(n, 1))
        self._L.sgo_get_array(self.h, key.encode(), _dp(out), n)
        return out[:n]

    def last_step_flops(self): return self._L.sgo_last_step_flops(self.h)

    def flops(self, reset=False):
        """(forwards, PGS flops, all-stage flops) accumulated since the last reset."""
        out = np.zeros(3)
        self._L.sgo_flops_get(self.h, _dp(out))
        if reset:
            self._L.sgo_flops_reset(self.h)
        return out

    def episode(self, sim_start=1, sim_step=7, n_settle=40, n_iter=160, open_close_div=80, ctrl_mag=0.2):
        """create_dataset.log_into_file's episode (ref: create_dataset.py:33-60) -> (rows[T,12], touch[T], status)."""
        T = n_settle + n_iter
        out = np.zeros((T, self.m.nsensordata))
        touch = np.zeros(T, dtype=np.int32)
        st = self._L.sgo_episode(self.h, sim_start, sim_step, n_settle, n_iter, open_close_div, float(ctrl_mag),
                                 _dp(out), touch.ctypes.data_as(C.POINTER(C.c_int)))
        return out, touch, st


# ---- hooks for known-answer tests of the oracle's static helpers -----------------------------------
def _arr(x):
    return np.ascontiguousarray(x, dtype=np.float64)


def capsule_box(cpos, cmat, csize, bpos, bmat, bsize):
    """-> list of (dist, pos[3], normal[3]) from the oracle's capsule-box narrowphase."""
    out = np.zeros(14)
    a = [_arr(v) for v in (cpos, np.asarray(cmat).reshape(9), csize, bpos, np.asarray(bmat).reshape(9), bsize)]
    n = lib().sgo_test_capsule_box(*[_dp(v) for v in a], _dp(out))
    return [(out[7 * i], out[7 * i + 1:7 * i + 4].copy(), out[7 * i + 4:7 * i + 7].copy()) for i in range(n)]


def sphere_box(spos, radius, bpos, bmat, bsize):
    out = np.zeros(7)
    a = [_arr(v) for v in (spos, bpos, np.asarray(bmat).reshape(9), bsize)]
    n = lib().sgo_test_sphere_box(_dp(a[0]), float(radius), _dp(a[1]), _dp(a[2]), _dp(a[3]), _dp(out))
    return (out[0], out[1:4].copy(), out[4:7].copy()) if n else None


def qcqp2(A, b, d, r):
    res = np.zeros(2)
    a = [_arr(np.asarray(A).reshape(4)), _arr(b), _arr(d)]
    active = lib().sgo_test_qcqp2(_dp(a[0]), _dp(a[1]), _dp(a[2]), float(r), _dp(res))
    return res, bool(active)


def impedance(solimp, pos, margin=0.0):
    a = _arr(solimp)
    return lib().sgo_test_impedance(_dp(a), float(pos), float(margin))


def box_box_overlap(p1, R1, s1, p2, R2, s2):
    a = [_arr(np.asarray(v).reshape(-1)) for v in (p1, R1, s1, p2, R2, s2)]
    return bool(lib().sgo_test_box_box(*[_dp(v) for v in a]))


def make_frame(frame):
    a = _arr(np.asarray(frame).reshape(9)).copy()
    lib().sgo_test_make_frame(_dp(a))
    return a.reshape(3, 3)
