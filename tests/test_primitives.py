"""The step kernel's small device primitives, one by one, against the oracle's own primitives or a high-precision
restatement, at inputs chosen for their edges.

tests/prim/sg_prim.cu applies each primitive of sg_math.cuh / sg_kernels2.cuh element by element.  It is built two ways
into a temporary directory: under the SIMT emulator (g++, the `-m "not gpu"` tests) and with nvcc for sm_100a with the
product's flags (the `-m gpu` tests), where the fp32 entry points run the MUFU approximations (rcp / sqrt / rsqrt.approx,
-use_fast_math) that the emulator build replaces by exact arithmetic.

Bars: fp64 equals the oracle to 1e-12 of the geometry scale.  fp32 gets the inputs rounded to fp32 on both sides and is
held to about ten times the error measured on a B200 (profiles/primitives_measured.txt); where an fp64 reference moves by
more than AMP x its input perturbation inside a ball of relative radius BAND (a discrete threshold: contact count, branch,
tie, the 0.5 switch of make_frame) the fp32 result only has to be finite and show a count seen inside that ball.
friction_fast is held to an fp64 bisection of the same secular equation on the domain the step kernel produces
(profiles/fric_domain.json, scripts/dev_fric_domain.py)."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import ROOT

CSRC = os.path.join(ROOT, "soft-grip_b200", "csrc")
SIMT = os.path.join(ROOT, "tests", "simt")
PRIM = os.path.join(ROOT, "tests", "prim", "sg_prim.cu")

BAND, AMP, KPERT = 1e-6, 30.0, 16          # fp32 threshold band (relative to the scale), amplification that marks one, probes
BAND64 = 1e-9                              # the same for fp64 on the device
FP64_TOL = 1e-12
# fp32 bars, about ten times the worst error measured on a B200 at 1000 W (profiles/primitives_measured.txt)
FP32_GEOM_TOL = 3e-6                       # dist / pos over the geometry scale, normals absolute (measured 3.4e-7)
FP32_CAPSULE_TOL = 1e-4                    # capsule-box (4.0e-5): the closest segment point interpolates a piecewise-linear derivative
FP32_FRAME_TOL = 2e-5                      # make_frame, absolute (2.2e-6)
FP32_IMP_TOL = 3e-6                        # impedance, absolute, values in (0, 1) (2.6e-7)
FRIC_ACTIVE_TOL = 3e-6                     # DESIGN.md section 3: the same root to 3e-6 relative, from a cold start (8.0e-7)
FRIC_WARM_TOL = 1e-5                       # from a warm start anywhere in 1e-5 .. 1e5 x the root (1.0e-6; 2.9e-6 in the emulator)
FRIC_CONE_TOL = 2e-6                       # active: | |f| / (frc f0) - 1 | (2.0e-7)
FRIC_INACTIVE_K = 8.0                      # inactive: error <= K x condition x fp32 epsilon, the 2x2 solve's det cancels (0.78)
EPS32 = float(np.finfo(np.float32).eps)
# the domain of friction_fast's arguments in the fp32 step kernel, measured under the emulator over the twelve golden softbox
# snapshots and five emulated squeeze episodes (profiles/fric_domain.json): f0 1.9e-6 .. 12.9, |bc| kb / f0 6.6e-4 .. 2.0e4,
# condition of the normalised block 1.14 .. 54.8, warm start over root 6.3e-5 .. 1.5e4.  The bars below hold on a margin
# around it.  Outside it, |bc| kb / f0 >= 1e12 drops the friction force (|w|^2 or w' adj w overflows fp32 at the multiplier that
# puts the force on the cone, rsqrt(inf) = 0): eight decades beyond anything the kernel produces, stated here, not asserted.
DOMAIN = {"f0": (1e-6, 1e2), "q": (1e-4, 1e5), "cond": 100.0, "warm": (1e-5, 1e5)}


def _make_var(d, name):
    return subprocess.check_output(["make", "-s", "-C", d, "--eval", "print-%: ; @echo $($*)", "print-" + name], text=True).split()


def device_commands(out):
    """nvcc command lines of the device build: NVCCFLAGS of soft-grip_b200/csrc/Makefile, plus FASTFLAGS for fp32 (as its
    fp32 step-kernel instances)."""
    nvcc, flags, fast, arch = _make_var(CSRC, "NVCC")[0], _make_var(CSRC, "NVCCFLAGS"), _make_var(CSRC, "FASTFLAGS"), _make_var(CSRC, "ARCH")
    o32, o64, so = (os.path.join(out, x) for x in ("prim32.o", "prim64.o", "libsgprim.so"))
    return [[nvcc] + flags + fast + ["-I", CSRC, "-DSGP_PREC=32", "-c", "-o", o32, PRIM],
            [nvcc] + flags + ["-I", CSRC, "-DSGP_PREC=64", "-c", "-o", o64, PRIM],
            [nvcc] + arch + ["-shared", "-o", so, o32, o64]], so


def emulator_commands(out):
    cxx, flags = _make_var(SIMT, "CXX")[0], _make_var(SIMT, "CXXFLAGS")
    o32, o64, so = (os.path.join(out, x) for x in ("prim32.o", "prim64.o", "libsgprim_emu.so"))
    return [[cxx] + flags + ["-x", "c++", "-DSGP_PREC=32", "-c", "-o", o32, PRIM],
            [cxx] + flags + ["-x", "c++", "-DSGP_PREC=64", "-c", "-o", o64, PRIM],
            [cxx, "-shared", "-o", so, o32, o64]], so


class Prim:
    def __init__(self, so, where):
        self.L, self.where = C.CDLL(so), where

    def __call__(self, name, prec, x, no, extra=None):
        dt = np.float32 if prec == 32 else np.float64
        x = np.ascontiguousarray(x, dtype=dt)
        out = np.empty((x.shape[0], no), dtype=dt)
        f = getattr(self.L, "sgp_%s_f%d" % (name, prec))
        args = ([extra.ctypes.data_as(C.c_void_p)] if extra is not None else []) + [x.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), C.c_int(x.shape[0])]
        rc = f(*args)
        assert rc == 0, "%s %s: CUDA error %d" % (self.where, name, -rc)
        return out.astype(np.float64)


@pytest.fixture(scope="module", params=["emu", pytest.param("dev", marks=pytest.mark.gpu)])
def prim(request):
    out = tempfile.mkdtemp(prefix="sg_prim_")
    try:
        if request.param == "dev":
            cmds, so = device_commands(out)
            if shutil.which(cmds[0][0]) is None:
                pytest.fail("nvcc not found (%s): the device build of the primitives needs it" % cmds[0][0])
            for c in cmds:
                subprocess.check_call(c, cwd=CSRC, stdout=subprocess.DEVNULL)
        else:
            cmds, so = emulator_commands(out)
            for c in cmds:
                subprocess.check_call(c, cwd=SIMT)
        yield Prim(so, request.param)
    finally:
        shutil.rmtree(out, ignore_errors=True)


@pytest.fixture(scope="module")
def so(oracle):
    return oracle


def report(prim, what, prec, measured, bound):
    print("MEASURED %-4s %-28s fp%d  worst %.3e  bound %.1e" % (prim.where, what, prec, measured, bound))


def rng_for(name):
    return np.random.default_rng([ord(c) for c in name])


def rotations(rng, n):
    Q, R = np.linalg.qr(rng.standard_normal((n, 3, 3)))
    Q = Q * np.sign(np.diagonal(R, axis1=1, axis2=2))[:, None, :]
    Q[np.linalg.det(Q) < 0, :, 0] *= -1
    return Q


def exact_rotations():
    """the 24 proper rotations of the cube: signed permutation matrices, exact in any precision"""
    out = []
    for p in ((0, 1, 2), (1, 2, 0), (2, 0, 1), (0, 2, 1), (2, 1, 0), (1, 0, 2)):
        for s in np.array(np.meshgrid([1, -1], [1, -1], [1, -1])).T.reshape(-1, 3):
            M = np.zeros((3, 3))
            M[[0, 1, 2], p] = s
            if np.linalg.det(M) > 0:
                out.append(M)
    return np.array(out)


def rounded(x, prec):
    return np.asarray(x, dtype=np.float32).astype(np.float64) if prec == 32 else np.asarray(x, dtype=np.float64)


def check_geometry(prim, what, prec, got, X, ref_fn, scale, pert_cols, unit_cols, rng, max_flagged=None, unit_in=(), tol=None):
    """got: kernel outputs (column 0 the contact count); X: the inputs as the kernel saw them; ref_fn: fp64 reference on
    an input array; pert_cols: inputs probed for thresholds, by band x scale (unit_in: by band, directions and rotations).
    fp64 under the emulator (the oracle's own arithmetic, no fused multiply-adds): equal counts and values to FP64_TOL
    everywhere.  fp64 on the device, which contracts to FMAs, and fp32: the same away from a threshold, a count seen
    within the band at one (module docstring); the band is BAND64 resp. BAND."""
    ref = ref_fn(X)
    assert got.shape == ref.shape
    colscale = np.where(np.isin(np.arange(ref.shape[1]), unit_cols), 1.0, scale[:, None])
    err = np.abs(got - ref) / colscale
    if prec == 64 and prim.where == "emu":
        bad = np.flatnonzero(got[:, 0] != ref[:, 0])
        assert bad.size == 0, (what, "count differs from the oracle", bad[:5], X[bad[:1]])
        worst = float(err.max())
        report(prim, what, prec, worst, FP64_TOL)
        assert worst <= FP64_TOL, (what, np.unravel_index(err.argmax(), err.shape), X[err.max(axis=1).argmax()])
        return
    band = BAND if prec == 32 else BAND64
    tol = (tol or FP32_GEOM_TOL) if prec == 32 else FP64_TOL
    assert np.isfinite(got).all(), (what, "non-finite output", X[~np.isfinite(got).all(axis=1)][:1])
    flagged = np.zeros(len(X), bool)
    counts = [ref[:, 0]]
    for _ in range(KPERT):
        Xp = X.copy()
        Xp[:, pert_cols] += band * scale[:, None] * rng.uniform(-1, 1, (len(X), len(pert_cols)))
        Xp[:, list(unit_in)] += band * rng.uniform(-1, 1, (len(X), len(unit_in)))
        rp = ref_fn(Xp)
        counts.append(rp[:, 0])
        flagged |= (rp[:, 0] != ref[:, 0]) | (np.abs(rp - ref) / colscale > AMP * band).any(axis=1)
    counts = np.stack(counts, 1)
    ok_count = (counts == got[:, :1]).any(axis=1)
    assert ok_count.all(), (what, "count outside those seen within the band", X[~ok_count][:1], got[~ok_count][:1], ref[~ok_count][:1])
    keep = ~flagged
    assert (got[keep, 0] == ref[keep, 0]).all(), (what, "count flips away from a threshold")
    worst = float(err[keep].max()) if keep.any() else 0.0
    report(prim, what + " (%d/%d near a threshold)" % (int(flagged.sum()), len(X)), prec, worst, tol)
    if max_flagged is not None:
        assert flagged.mean() <= max_flagged, (what, "too many inputs near a threshold to test", flagged.mean())
    assert worst <= tol, (what, X[keep][err[keep].max(axis=1).argmax()], got[keep][err[keep].max(axis=1).argmax()], ref[keep][err[keep].max(axis=1).argmax()])


# ---------------------------------------------------------------------------------------------------------------------
# sphere-box
# ---------------------------------------------------------------------------------------------------------------------
def sphere_box_inputs(rng, n=3000):
    bsize = rng.uniform(0.01, 0.08, (n, 3))
    bpos = rng.uniform(-0.2, 0.2, (n, 3))
    R = rotations(rng, n)
    radius = rng.uniform(0.005, 0.05, n)
    local = rng.uniform(-1, 1, (n, 3)) * (bsize + 1.2 * radius[:, None])
    spos = bpos + np.einsum("nij,nj->ni", R, local)
    X = [np.concatenate([spos, radius[:, None], bpos, R.reshape(n, 9), bsize], 1)]
    # constructed, in exact arithmetic: the centre inside with ties between faces, exactly on a face, an edge, a corner
    s = 0.0625
    locs = [(0, 0, 0), (s / 2, s / 2, 0), (s / 2, -s / 2, s / 2), (s, 0.01, 0.02), (-s, 0.01, 0.02), (0.01, s, -0.02), (s, s, 0.01),
            (s, -s, 0.01), (s, s, s), (-s, -s, -s), (s + 0.0078125, 0, 0), (s + 0.0078125, s + 0.0078125, 0), (0.03125, 0.0078125, 0)]
    rows = []
    for M in exact_rotations():
        for size in ((s, s, s), (s, s / 2, 2 * s)):
            for loc in locs:
                bp = np.array([0.125, -0.25, 0.5])
                sp = bp + M @ (np.array(loc) * np.array(size) / s)
                rows.append(np.concatenate([sp, [0.015625], bp, M.reshape(9), size]))
    X.append(np.array(rows))
    return np.concatenate(X)


def sphere_box_ref(so):
    def f(X):
        out = np.zeros((len(X), 8))
        for i, x in enumerate(X):
            r = so.sphere_box(x[0:3], x[3], x[4:7], x[7:16].reshape(3, 3), x[16:19])
            if r is not None:
                out[i] = [1, r[0], *r[1], *r[2]]
        return out
    return f


def geom_scale(*cols):
    return np.maximum.reduce([np.abs(c).max(axis=1) if c.ndim == 2 else np.abs(c) for c in cols])


@pytest.mark.parametrize("prec", [64, 32])
def test_sphere_box_matches_oracle(prim, so, prec):
    X = rounded(sphere_box_inputs(rng_for("sphere_box")), prec)
    got = prim("sphere_box", prec, X, 8)
    scale = geom_scale(X[:, 0:3], X[:, 3], X[:, 4:7], X[:, 16:19])
    check_geometry(prim, "sphere_box", prec, got, X, sphere_box_ref(so), scale, [0, 1, 2, 3, 4, 5, 6, 16, 17, 18], [5, 6, 7],
                   rng_for("sphere_box/pert"))
    assert got[:, 0].sum() > len(X) // 3


# ---------------------------------------------------------------------------------------------------------------------
# capsule-box (seg_box_grad, the in-box branches)
# ---------------------------------------------------------------------------------------------------------------------
def capsule_box_inputs(rng, n=3000):
    bsize = rng.uniform(0.01, 0.08, (n, 3))
    bpos = rng.uniform(-0.2, 0.2, (n, 3))
    R = rotations(rng, n)
    radius = rng.uniform(0.005, 0.03, n)
    hl = rng.uniform(0.01, 0.08, n)
    axis = rng.standard_normal((n, 3))
    axis /= np.linalg.norm(axis, axis=1, keepdims=True)
    local = rng.uniform(-1, 1, (n, 3)) * (bsize + radius[:, None] + 0.5 * hl[:, None])
    cpos = bpos + np.einsum("nij,nj->ni", R, local)
    X = [np.concatenate([cpos, axis, radius[:, None], hl[:, None], bpos, R.reshape(n, 9), bsize], 1)]
    # constructed, exact: axis parallel to a face (h[k] = 0), a segment through the box, one end inside (in0 / in1), both
    # inside (the deeper end), an end exactly on a face plane, a segment along a face
    s, e = 0.0625, 0.0078125
    cases = [((0, 0, s + e), (1, 0, 0), 0.03125), ((0, 0.01, 0.02), (1, 0, 0), 0.125), ((s, 0, 0), (1, 0, 0), 0.03125),
             ((-s, 0, 0), (1, 0, 0), 0.03125), ((0.01, 0, 0), (1, 0, 0), 0.03125), ((-0.01, 0.02, 0), (0, 1, 0), 0.015625),
             ((0.03125, 0, 0), (1, 0, 0), 0.03125), ((0, s, 0), (1, 0, 0), 0.03125), ((0, s, s), (1, 0, 0), 0.03125),
             ((s + 2 * e, 0, 0), (0, 0, 1), 0.03125), ((s + 0.03125, 0, 0), (1, 0, 0), 0.03125), ((0.6 * s, 0.8 * s, 0), (0.6, 0.8, 0), 0.125)]
    rows = []
    bp = np.array([0.125, -0.25, 0.5])
    for M in exact_rotations():
        for c, a, h in cases:
            rows.append(np.concatenate([bp + M @ np.array(c), M @ np.array(a, float), [0.015625, h], bp, M.reshape(9), [s, s, s]]))
    X.append(np.array(rows))
    return np.concatenate(X)


def capsule_box_ref(so):
    def f(X):
        out = np.zeros((len(X), 15))
        for i, x in enumerate(X):
            cmat = np.zeros(9)
            cmat[[2, 5, 8]] = x[3:6]
            cons = so.capsule_box(x[0:3], cmat, [x[6], x[7]], x[8:11], x[11:20].reshape(3, 3), x[20:23])
            out[i, 0] = len(cons)
            for j, (d, p, nrm) in enumerate(cons):
                out[i, 1 + 7 * j:8 + 7 * j] = [d, *p, *nrm]
        return out
    return f


@pytest.mark.parametrize("prec", [64, 32])
def test_capsule_box_matches_oracle(prim, so, prec):
    X = rounded(capsule_box_inputs(rng_for("capsule_box")), prec)
    got = prim("capsule_box", prec, X, 15)
    scale = geom_scale(X[:, 0:3], X[:, 6], X[:, 7], X[:, 8:11], X[:, 20:23])
    check_geometry(prim, "capsule_box", prec, got, X, capsule_box_ref(so), scale, [0, 1, 2, 6, 7, 8, 9, 10, 20, 21, 22],
                   [5, 6, 7, 12, 13, 14], rng_for("capsule_box/pert"), unit_in=range(3, 6),
                   tol=FP32_CAPSULE_TOL)
    assert (got[:, 0] == 2).sum() > 100 and (got[:, 0] == 1).sum() > 100


# ---------------------------------------------------------------------------------------------------------------------
# plane-capsule: the oracle does not export it, so a numpy restatement of mjc_PlaneCapsule
# ---------------------------------------------------------------------------------------------------------------------
def plane_capsule_ref(X):
    ppos, nrm, cpos, axis, r, hl = X[:, 0:3], X[:, 3:12].reshape(-1, 3, 3)[:, :, 2], X[:, 12:15], X[:, 15:18], X[:, 18], X[:, 19]
    out = np.zeros((len(X), 21))
    for side in (1, -1):
        sp = cpos + side * axis * hl[:, None]
        dist = ((sp - ppos) * nrm).sum(1) - r
        hit = dist <= 0
        j = out[:, 0].astype(int)
        for i in np.flatnonzero(hit):
            o = 1 + 10 * j[i]
            out[i, o] = dist[i]
            out[i, o + 1:o + 4] = sp[i] - nrm[i] * (r[i] + 0.5 * dist[i])
            out[i, o + 4:o + 7] = nrm[i]
            out[i, o + 7:o + 10] = axis[i]
        out[hit, 0] += 1
    return out


def plane_capsule_inputs(rng, n=3000):
    R = rotations(rng, n)
    ppos = rng.uniform(-0.2, 0.2, (n, 3))
    radius, hl = rng.uniform(0.005, 0.03, n), rng.uniform(0.01, 0.08, n)
    axis = rng.standard_normal((n, 3))
    axis /= np.linalg.norm(axis, axis=1, keepdims=True)
    height = rng.uniform(-1, 1, n) * (radius + hl)
    cpos = ppos + R[:, :, 2] * height[:, None] + np.einsum("nij,nj->ni", R[:, :, :2], rng.uniform(-0.1, 0.1, (n, 2)))
    X = [np.concatenate([ppos, R.reshape(n, 9), cpos, axis, radius[:, None], hl[:, None]], 1)]
    rows = []   # exact: capsule parallel to the plane touching it (dist = 0 at both ends), one end exactly touching
    for M in exact_rotations():
        p = np.array([0.125, -0.25, 0.5])
        for c, a in (((0, 0, 0.015625), (1, 0, 0)), ((0, 0, 0.046875), (0, 0, 1)), ((0.25, 0, 0.015625 + 2 ** -20), (0, 1, 0))):
            rows.append(np.concatenate([p, M.reshape(9), p + M @ np.array(c), M @ np.array(a, float), [0.015625, 0.03125]]))
    X.append(np.array(rows))
    return np.concatenate(X)


@pytest.mark.parametrize("prec", [64, 32])
def test_plane_capsule_matches_restatement(prim, prec):
    X = rounded(plane_capsule_inputs(rng_for("plane_capsule")), prec)
    got = prim("plane_capsule", prec, X, 21)
    scale = geom_scale(X[:, 0:3], X[:, 12:15], X[:, 18], X[:, 19])
    unit = [5, 6, 7, 8, 9, 10, 15, 16, 17, 18, 19, 20]
    check_geometry(prim, "plane_capsule", prec, got, X, plane_capsule_ref, scale, [0, 1, 2, 12, 13, 14, 18, 19], unit,
                   rng_for("plane_capsule/pert"))
    assert (got[:, 0] == 2).sum() > 100 and (got[:, 0] == 1).sum() > 100


# ---------------------------------------------------------------------------------------------------------------------
# box-box overlap (separating axes with a 1e-12 slack)
# ---------------------------------------------------------------------------------------------------------------------
def test_box_box_overlap_matches_oracle_and_its_slack(prim, so):
    rng = rng_for("box_box")
    n = 3000
    s1, s2 = rng.uniform(0.01, 0.08, (n, 3)), rng.uniform(0.01, 0.08, (n, 3))
    R1, R2 = rotations(rng, n), rotations(rng, n)
    p1 = rng.uniform(-0.2, 0.2, (n, 3))
    p2 = p1 + np.einsum("nij,nj->ni", R1, rng.uniform(-1, 1, (n, 3)) * (s1 + 1.2 * s2))
    X = np.concatenate([p1, R1.reshape(n, 9), s1, p2, R2.reshape(n, 9), s2], 1)
    ref = lambda A: np.array([[so.box_box_overlap(x[0:3], x[3:12], x[12:15], x[15:18], x[18:27], x[27:30])] for x in A], float)  # noqa: E731
    # touching cubes face to face: the gap at which they separate is 1e-12 x (sum of the half sizes) plus the largest
    # edge-axis slack; a gap of half the smallest slack still overlaps, a gap of twice the largest does not
    s, I = 0.0625, np.eye(3)
    p = np.array([0.125, -0.25, 0.5])
    touch, want = [], []
    for M in exact_rotations():
        d = M @ np.array([2 * s, 0, 0])
        for gap, ov in ((0.0, 1), (0.5 * 1e-12 * 3 * s, 1), (2 * 1e-12 * 4 * s, 0), (1e-5 * s, 0)):
            touch.append(np.concatenate([p, I.reshape(9), [s, s, s], p + d * (1 + gap / (2 * s)), M.reshape(9), [s, s, s]]))
            want.append(ov)
    touch, want = np.array(touch), np.array(want, float)
    for prec in (64, 32):
        Xp = rounded(X, prec)
        got = prim("box_box_overlap", prec, Xp, 1)
        assert set(np.unique(got[:, 0])) <= {0.0, 1.0}
        if prec == 64:
            np.testing.assert_array_equal(got, ref(Xp))
            gt = prim("box_box_overlap", 64, touch, 1)
            np.testing.assert_array_equal(ref(touch)[:, 0], want)
            np.testing.assert_array_equal(gt[:, 0], want)
            report(prim, "box_box_overlap", 64, 0.0, 0.0)
        else:
            scale = geom_scale(Xp[:, 0:3], Xp[:, 12:15], Xp[:, 15:18], Xp[:, 27:30])
            check_geometry(prim, "box_box_overlap", 32, got, Xp, ref, scale, [0, 1, 2, 12, 13, 14, 15, 16, 17, 27, 28, 29], [],
                           rng_for("box_box/pert"), max_flagged=0.02)
            # the 1e-12 slack is below fp32 resolution: touching overlaps, a gap of 1e-5 of the size separates
            gt = prim("box_box_overlap", 32, rounded(touch, 32), 1)
            np.testing.assert_array_equal(gt[0::4, 0], 1.0)
            np.testing.assert_array_equal(gt[3::4, 0], 0.0)
    assert 0.2 < got[:, 0].mean() < 0.9


# ---------------------------------------------------------------------------------------------------------------------
# make_frame
# ---------------------------------------------------------------------------------------------------------------------
def test_make_frame_matches_oracle(prim, so):
    rng = rng_for("make_frame")
    n = 4000
    nrm = rng.standard_normal((n, 3)) * rng.uniform(0.1, 3, (n, 1))
    hint = rng.standard_normal((n, 3))
    hint *= (rng.uniform(0, 1.5, n) / np.linalg.norm(hint, axis=1))[:, None]
    X = [np.concatenate([nrm, hint], 1)]
    # normals near +-y (the 0.5 switch of the default tangent), hints just below / at / above length 0.5
    rows = []
    for y in (0.5, -0.5):
        for dy in (-1e-3, -1e-6, 0.0, 1e-6, 1e-3):
            yy = y + dy
            rows.append([np.sqrt(1 - yy * yy), yy, 0, 0.1, 0, 0.2])
            rows.append([0, yy, np.sqrt(1 - yy * yy), 0, 0, 0])
    for hl in (0.49, 0.5, 0.51):
        rows += [[0, 0, 1, hl, 0, 0], [0, 1, 0, 0, 0, hl], [1, 0, 0, 0, hl, 0]]
    rows += [[0, 1, 0, 0, 0, 0], [0, -1, 0, 0, 0, 0], [1e-3, 1, 0, 0, 0, 0], [0, 0, 1, 0.3, 0.3, 0.3]]
    X.append(np.array(rows, float))
    X = np.concatenate(X)
    ref = lambda A: np.array([so.make_frame(np.concatenate([x, np.zeros(3)])).reshape(9) for x in A])  # noqa: E731
    for prec in (64, 32):
        Xp = rounded(X, prec)
        got = prim("make_frame", prec, Xp, 9)
        if prec == 64:
            err = float(np.abs(got - ref(Xp)).max())
            report(prim, "make_frame", 64, err, FP64_TOL)
            assert err <= FP64_TOL
        else:
            # a zero count column in front so that check_geometry can be reused
            pad = lambda A: np.concatenate([np.zeros((len(A), 1)), A], 1)  # noqa: E731
            check_geometry(prim, "make_frame", 32, pad(got), Xp, lambda A: pad(ref(A)), np.ones(len(Xp)), list(range(6)),
                           list(range(1, 10)), rng_for("make_frame/pert"), max_flagged=0.02, tol=FP32_FRAME_TOL)


# ---------------------------------------------------------------------------------------------------------------------
# impedance2 on fill_si constants
# ---------------------------------------------------------------------------------------------------------------------
def test_impedance2_matches_oracle(prim, so):
    rng = rng_for("impedance")
    n = 4000
    si = np.stack([rng.uniform(1e-4, 0.9999, n), rng.uniform(1e-4, 0.9999, n), rng.uniform(1e-4, 0.1, n), rng.uniform(0.01, 0.99, n),
                   np.where(rng.uniform(size=n) < 0.2, 1.0, rng.uniform(1, 6, n))], 1)
    si[rng.uniform(size=n) < 0.2, 4] = 2.0
    pos = rng.uniform(-1.5, 1.5, n) * si[:, 2]
    # edges: pos = 0, |pos| = width, x = mid, power 1, d0 = d1, width 0 and below MINVAL (exact values)
    edge_si, edge_pos = [], []
    base = [0.5, 0.875, 0.25, 0.5, 2.0]
    for sv, p in ((base, 0.0), (base, 0.25), (base, -0.25), (base, 0.125), (base, -0.125), ([0.5, 0.875, 0.25, 0.5, 1.0], 0.0625),
                  ([0.625, 0.625, 0.25, 0.5, 2.0], 0.0625), ([0.5, 0.875, 0.0, 0.5, 2.0], 0.0625), ([0.5, 0.875, 1e-16, 0.5, 2.0], 0.0),
                  ([0.9, 0.95, 0.001, 0.5, 2.0], 0.0005), ([0.9, 0.95, 0.001, 0.25, 3.0], 0.00075), (base, 0.5)):
        edge_si.append(sv); edge_pos.append(p)
    si = np.concatenate([si, edge_si]); pos = np.concatenate([pos, edge_pos])
    for prec in (64, 32):
        p = rounded(pos, prec)
        got = prim("impedance2", prec, p[:, None], 1, extra=np.ascontiguousarray(si))[:, 0]
        want = np.array([so.impedance(s, x) for s, x in zip(si, p)])
        assert np.isfinite(got).all()
        err = float(np.abs(got - want).max())
        report(prim, "impedance2", prec, err, FP64_TOL if prec == 64 else FP32_IMP_TOL)
        assert err <= (FP64_TOL if prec == 64 else FP32_IMP_TOL), (si[np.abs(got - want).argmax()], p[np.abs(got - want).argmax()])
        k = len(pos) - len(edge_pos)       # the edges hit their branch values exactly
        assert got[k] == rounded(0.5, prec) and got[k + 1] == rounded(0.875, prec) and got[k + 2] == rounded(0.875, prec)
        assert got[k + 6] == rounded(0.625, prec) and got[k + 7] == rounded(0.6875, prec) and got[k + 8] == rounded(0.6875, prec)


# ---------------------------------------------------------------------------------------------------------------------
# friction: qcqp2_fast<double> + the rescaling of friction() against the oracle; friction_fast against a bisection
# ---------------------------------------------------------------------------------------------------------------------
def spd_blocks(rng, n, cond_hi):
    """2x2 SPD blocks of trace 1, condition log-uniform in [1, cond_hi], random orientation -> a11, a12 (a22 = 1 - a11)"""
    cond = np.exp(rng.uniform(0, np.log(cond_hi), n))
    lmin = 1 / (1 + cond)
    lmax = 1 - lmin
    th = rng.uniform(0, np.pi, n)
    c, s = np.cos(th), np.sin(th)
    return lmax * c * c + lmin * s * s, (lmax - lmin) * c * s


def test_qcqp2_and_friction_fp64_match_oracle(prim, so):
    rng = rng_for("qcqp2")
    n = 3000
    a11, a12 = spd_blocks(rng, n, 1e4)
    tr = np.exp(rng.uniform(np.log(1e-3), np.log(1e3), n))
    A11, A12, A22 = a11 * tr, a12 * tr, (1 - a11) * tr
    frc = np.exp(rng.uniform(np.log(1e-2), np.log(3), n))
    f0 = np.exp(rng.uniform(np.log(1e-6), np.log(1e2), n))
    ang = rng.uniform(0, 2 * np.pi, n)
    bmag = f0 * tr * np.exp(rng.uniform(np.log(1e-3), np.log(1e4), n)) / frc
    bc = np.stack([bmag * np.cos(ang), bmag * np.sin(ang)], 1)
    d2 = np.where(rng.uniform(size=n) < 0.3, frc * rng.uniform(0.5, 2, n), frc)
    got = prim("qcqp2", 64, np.stack([A11, A12, A22, bc[:, 0], bc[:, 1], frc, d2, f0], 1), 3)
    want = np.array([np.r_[r, a] for r, a in (so.qcqp2([[A11[i], A12[i]], [A12[i], A22[i]]], bc[i], [frc[i], d2[i]], f0[i]) for i in range(n))])
    np.testing.assert_array_equal(got[:, 2], want[:, 2])
    sc = np.maximum(np.abs(want[:, :2]).max(1), f0 * np.maximum(frc, d2))
    err = float((np.abs(got[:, :2] - want[:, :2]) / sc[:, None]).max())
    report(prim, "qcqp2_fast<double>", 64, err, FP64_TOL)
    assert err <= FP64_TOL
    # friction(): the same with d = (frc, frc), then onto the cone (mj_solPGS)
    got = prim("friction", 64, np.stack([A11, A12, A22, bc[:, 0], bc[:, 1], frc, f0], 1), 2)
    want = np.zeros((n, 2))
    for i in range(n):
        vv, active = so.qcqp2([[A11[i], A12[i]], [A12[i], A22[i]]], bc[i], [frc[i], frc[i]], f0[i])
        if active:
            s = np.sqrt(f0[i] ** 2 / max(1e-15, (vv[0] ** 2 + vv[1] ** 2) / frc[i] ** 2))
            vv = vv * s
        want[i] = vv
    err = float((np.abs(got - want) / (frc * f0)[:, None]).max())
    report(prim, "friction() fp64 (rescaled)", 64, err, FP64_TOL)
    assert err <= FP64_TOL
    # (no cone bar here: MuJoCo's iteration stops at |v|^2 - r^2 < 1e-10 absolute, which leaves a small f0 outside its cone)


def secular_ref(a11, a12, kb, bc, f0):
    """fp64 / long double solution of min 0.5 v'Av + b'v, |v| <= f0 with A = [[a11, a12], [a12, 1 - a11]], b = kb bc: the
    free minimiser when it lies in the cone, otherwise v(la) = -(A + la)^-1 b with |v(la)| = f0 by bisection.
    Returns v (n x 2), la (0 when inactive), active."""
    L = np.longdouble
    a11, a12, kb, f0 = (np.asarray(x, dtype=L) for x in (a11, a12, kb, f0))
    a22 = L(1) - a11
    b1, b2 = np.asarray(bc[:, 0], L) * kb, np.asarray(bc[:, 1], L) * kb

    def v(la):
        c11, c22 = a11 + la, a22 + la
        det = c11 * c22 - a12 * a12
        return -(c22 * b1 - a12 * b2) / det, -(c11 * b2 - a12 * b1) / det

    v1, v2 = v(L(0))
    active = np.hypot(v1, v2) > f0
    lo = np.zeros_like(f0)
    hi = np.hypot(b1, b2) / f0
    for _ in range(200):
        mid = L(0.5) * (lo + hi)
        x1, x2 = v(mid)
        big = np.hypot(x1, x2) > f0
        lo = np.where(big, mid, lo)
        hi = np.where(big, hi, mid)
    la = np.where(active, L(0.5) * (lo + hi), L(0))
    x1, x2 = v(la)
    return np.stack([x1, x2], 1).astype(np.float64), la.astype(np.float64), active


def fric_problems(rng, n, cond_hi, f0_rng, q_rng, warm=None):
    a11, a12 = spd_blocks(rng, n, cond_hi)
    kb = np.exp(rng.uniform(np.log(1e-3), np.log(1e3), n))
    frc = np.exp(rng.uniform(np.log(1e-2), np.log(3), n))
    f0 = np.exp(rng.uniform(np.log(f0_rng[0]), np.log(f0_rng[1]), n))
    q = np.exp(rng.uniform(np.log(q_rng[0]), np.log(q_rng[1]), n))
    ang = rng.uniform(0, 2 * np.pi, n)
    bc = (q * f0 / kb)[:, None] * np.stack([np.cos(ang), np.sin(ang)], 1)
    la = np.zeros(n) if warm is None else warm
    X = np.stack([a11, a12, kb, bc[:, 0], bc[:, 1], frc, f0, la], 1).astype(np.float32).astype(np.float64)
    X[:, 0] = np.clip(X[:, 0], 2 ** -24, 1 - 2 ** -24)
    return X


def fric_solve(prim, X):
    got = prim("friction_fast", 32, X, 3)
    v, la, active = secular_ref(X[:, 0], X[:, 1], X[:, 2], X[:, 3:5], X[:, 6])
    frc, f0 = X[:, 5], X[:, 6]
    want = v * frc[:, None]
    err = np.abs(got[:, :2] - want).max(1) / np.maximum(frc * f0, np.abs(want).max(1))
    a11, a12 = X[:, 0], X[:, 1]
    det = a11 * (1 - a11) - a12 * a12
    disc = np.sqrt(np.maximum(0, 0.25 - det))
    cond = (0.5 + disc) / (det / (0.5 + disc))
    return got, want, la, active, err, cond


def check_friction(prim, what, X, got, want, active, err, cond, active_tol=FRIC_ACTIVE_TOL):
    frc, f0 = X[:, 5], X[:, 6]
    assert np.isfinite(got).all(), (what, X[~np.isfinite(got).all(1)][:1])
    fn = np.hypot(got[:, 0], got[:, 1])
    inside = fn <= frc * f0 * (1 + 1e-5)
    assert inside.all(), (what, "outside the cone", X[~inside][:1], fn[~inside][:1] / (frc * f0)[~inside][:1])
    on = np.abs(fn[active] / (frc * f0)[active] - 1)
    worst_on = float(on.max()) if on.size else 0.0
    worst_act = float(err[active].max()) if active.any() else 0.0
    ratio = err[~active] / (cond[~active] * EPS32)
    worst_in = float(ratio.max()) if ratio.size else 0.0
    report(prim, what + " on cone", 32, worst_on, FRIC_CONE_TOL)
    report(prim, what + " active", 32, worst_act, active_tol)
    report(prim, what + " inactive/(cond eps)", 32, worst_in, FRIC_INACTIVE_K)
    assert worst_on <= FRIC_CONE_TOL, (what, X[active][on.argmax()])
    assert worst_act <= active_tol, (what, X[active][err[active].argmax()], got[active][err[active].argmax()], want[active][err[active].argmax()])
    assert worst_in <= FRIC_INACTIVE_K, (what, X[~active][ratio.argmax()])


def test_friction_fast_on_the_kernel_domain(prim):
    rng = rng_for("friction_fast")
    n = 20000
    X = fric_problems(rng, n, DOMAIN["cond"], DOMAIN["f0"], DOMAIN["q"])
    got, want, la, active, err, cond = fric_solve(prim, X)
    assert 0.2 < active.mean() < 0.9
    check_friction(prim, "friction_fast cold", X, got, want, active, err, cond)


def test_friction_fast_warm_starts_settle_within_the_cap(prim):
    rng = rng_for("friction_fast/warm")
    n = 12000
    X = fric_problems(rng, n, DOMAIN["cond"], DOMAIN["f0"], DOMAIN["q"])
    _, _, root, active, _, _ = fric_solve(prim, X)
    # left of the root, right of the root (up to the measured 1.5e4 x), and an inactive problem after an active warm start
    side = rng.integers(0, 2, n)
    rel = np.where(side == 0, np.exp(rng.uniform(np.log(DOMAIN["warm"][0]), np.log(0.999), n)), np.exp(rng.uniform(np.log(1.001), np.log(DOMAIN["warm"][1]), n)))
    warm = np.where(active, root * rel, np.exp(rng.uniform(np.log(1e-3), np.log(1e4), n)))
    X[:, 7] = warm.astype(np.float32)
    got, want, la, active2, err, cond = fric_solve(prim, X)
    assert (active2 == active).all()
    assert (got[~active, 2] == 0).all(), "an inactive problem keeps a multiplier after a warm start"
    check_friction(prim, "friction_fast warm", X, got, want, active, err, cond, active_tol=FRIC_WARM_TOL)
    r = np.abs(got[active, 2] / la[active] - 1)
    report(prim, "friction_fast warm root", 32, float(r.max()), 1e-3)
    assert float(r.max()) <= 1e-3          # the multiplier it leaves for the next sweep is the root


def test_friction_fast_outside_the_domain_stays_finite_and_in_the_cone(prim):
    """Ranges wider than what the kernel produces: condition to 1e6, f0 from 1e-12, |bc| kb / f0 from 1e-3 to 1e15.  Finite
    and inside the cone except where fp32 underflows (below).  The errors are reported, not asserted: with a condition far
    beyond the kernel's 55 and |bc| kb / f0 >= 1e12 (friction force dropped) they reach the size of the force."""
    rng = rng_for("friction_fast/wide")
    n = 20000
    warm = np.where(rng.uniform(size=n) < 0.5, 0.0, np.exp(rng.uniform(np.log(1e-3), np.log(1e6), n)))
    X = fric_problems(rng, n, 1e6, (1e-12, 1e2), (1e-3, 1e15), warm=warm)
    got, want, la, active, err, cond = fric_solve(prim, X)
    b = np.hypot(X[:, 3], X[:, 4]) * X[:, 2]
    # Where |b|^2 f0 falls below ~1e-30 (f0 below 1e-8 and |bc| kb below 1e-11: far outside the kernel's domain, where f0 >=
    # 1.9e-6 and |bc| kb >= 1e-9), the Newton step's Q f0 underflows fp32, 1 / (Q f0) is inf and the result NaN.  Stated, not fixed.
    tiny = b * b * X[:, 6] < 1e-30
    report(prim, "friction_fast wide: non-finite where |b|^2 f0 < 1e-30", 32, float((~np.isfinite(got[tiny])).any(1).mean()) if tiny.any() else 0.0, float("nan"))
    assert np.isfinite(got[~tiny]).all(), X[~tiny][~np.isfinite(got[~tiny]).all(1)][:3]
    fn = np.hypot(got[:, 0], got[:, 1])[~tiny]
    assert (fn <= (X[:, 5] * X[:, 6])[~tiny] * (1 + 1e-5)).all()
    q = b / X[:, 6]
    active &= ~tiny
    sel = active & (q >= 1) & (q < 1e12)
    report(prim, "friction_fast wide active q<1e12", 32, float(err[sel].max()), float("nan"))
    report(prim, "friction_fast wide q>=1e12", 32, float(err[q >= 1e12].max()), float("nan"))


def test_device_build_uses_the_product_flags():
    """The device build of the primitives compiles with exactly what soft-grip_b200/csrc/Makefile gives its step-kernel
    instances: NVCCFLAGS, and FASTFLAGS for fp32 only (make -n of one instance of each precision)."""
    cmds, _ = device_commands(tempfile.gettempdir())

    def inst_flags(inst):
        line = subprocess.check_output(["make", "-n", "-B", "-C", CSRC, "build/%s.o" % inst], text=True).splitlines()
        line = [x for x in line if "sg_inst.cu" in x and " -c " in x][0].split(" 2> ")[0].split()
        drop = {"-Xptxas", "-v", "-c", "sg_inst.cu"}
        return [t for i, t in enumerate(line) if t not in drop and not t.startswith("-DSG_INST_") and line[i - 1] != "-o"]

    def prim_flags(cmd):
        return [t for i, t in enumerate(cmd) if t not in {"-c", PRIM, "-I", CSRC} and not t.startswith("-DSGP_") and cmd[i - 1] != "-o"]

    assert prim_flags(cmds[0]) == inst_flags("inst_float_8")
    assert prim_flags(cmds[1]) == inst_flags("inst_double_8")
    assert "-use_fast_math" in cmds[0] and "-use_fast_math" not in cmds[1]
    assert "arch=compute_100a,code=sm_100a" in cmds[0]
