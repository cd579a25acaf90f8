"""Kernel-source parity WITHOUT a GPU: soft-grip_b200/csrc (device code + C-ABI host logic) is compiled for the CPU
under the SIMT emulator of tests/simt (test infrastructure; never part of the product) and compared with the oracle
and the golden vectors.  Warp collectives are emulated exactly (the emulator aborts on divergent collectives), so
these tests pin the warp-synchronous logic: sub-warp worlds, ballot compaction, contact scheduling, level sweeps.
The `-m gpu` tests repeat the same comparisons on the real device through libsoftgrip.so."""
import importlib
import os
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, blob_path

sys.path.insert(0, os.path.join(ROOT, "tests", "simt"))

# about ten times what is measured on a B200 for softbox (profiles/r02x_test_gpu_measured.txt: q 1.1e-6, v 3.6e-5, qacc 1.6e-5,
# sens 1.0e-4 over the twelve golden snapshots); the larger models, in contact from the first step, get their own bound below
FP32_TOL = {"q": 1e-5, "v": 3e-4, "qacc": 2e-4, "sens": 1e-3}
FP32_TOL_OTHER = {"q": 5e-5, "v": 3e-3, "qacc": 3e-3, "sens": 1e-2}


def rel(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / max(1e-12, np.abs(b).max()))


@pytest.fixture(scope="module")
def emu():
    import emu as _emu
    _emu.build()
    return _emu


@pytest.fixture(scope="module")
def states():
    return np.load(os.path.join(GOLDEN, "softbox_states.npz"))


@pytest.mark.parametrize("prec,lpw", [(64, 8), (64, 4), (64, 32), (64, 16), (32, 8)])
def test_emulated_single_step_parity_against_golden_states(emu, states, prec, lpw):
    W = 32 // lpw + 1                      # one full warp of worlds plus a ragged tail
    env = emu.EmuBatch(blob_path("softbox"), W, prec=prec, lpw=lpw)
    env.set_params(stiffness=np.full(W, 700.0))
    env.set_debug_world(W - 1)
    idx = range(len(states["step"])) if (prec, lpw) == (64, 8) else range(0, len(states["step"]), 3)
    for i in idx:
        env.set_state(states["q"][i], states["v"][i], states["act"][i], states["warm"][i])
        env.set_ctrl([states["ctrl"][i]] * 2)
        sens, touch = env.step(1)
        q1, v1, a1, qacc = env.get_state()
        assert int(env.debug("ncon")[0]) == states["ncon1"][i]
        assert int(env.debug("nefc")[0]) == states["nefc1"][i]
        assert (touch == states["touch1"][i]).all()
        err = {"q": rel(q1[-1], states["q1"][i]), "v": rel(v1[-1], states["v1"][i]), "qacc": rel(qacc[-1], states["qacc1"][i]),
               "sens": rel(sens[-1], states["sens1"][i])}
        for k, e in err.items():
            assert e <= (1e-10 if prec == 64 else FP32_TOL[k]), (int(states["step"][i]), k, e)
        if prec == 64:
            assert int(env.debug("solver_iter")[0]) == states["iter1"][i]
        for w in range(W - 1):             # every group of the warp computes the same bits
            np.testing.assert_array_equal(q1[w], q1[-1])
            np.testing.assert_array_equal(qacc[w], qacc[-1])
        assert (env.status() == 0).all()
    env.close()


@pytest.mark.parametrize("lpw,nw", [(8, 4), (4, 2), (16, 8)])
def test_emulated_multi_warp_cta_parity(emu, states, lpw, nw):
    """Multi-warp CTAs (per-step CTA barrier, CTA-shared tables, ragged last warp) on contact-rich golden states: same
    parity bar as the single-warp case."""
    W = 19                                  # 16 worlds + a ragged tail
    env = emu.EmuBatch(blob_path("softbox"), W, prec=64, lpw=lpw, nw=nw)
    env.set_params(stiffness=np.full(W, 700.0))
    env.set_debug_world(17)
    for i in (4, 6, 7, 9, 11):
        env.set_state(states["q"][i], states["v"][i], states["act"][i], states["warm"][i])
        env.set_ctrl([states["ctrl"][i]] * 2)
        sens, touch = env.step(1)
        q1, v1, a1, qacc = env.get_state()
        assert int(env.debug("ncon")[0]) == states["ncon1"][i] and int(env.debug("solver_iter")[0]) == states["iter1"][i]
        for w in (0, 5, 15, 16, 18):
            assert rel(q1[w], states["q1"][i]) < 1e-9 and rel(v1[w], states["v1"][i]) < 1e-9 and rel(qacc[w], states["qacc1"][i]) < 1e-9
            assert rel(sens[w], states["sens1"][i]) < 1e-9
        assert (env.status() == 0).all()
    env.close()


def test_emulated_stage_diagnostics_match_oracle(emu, states, make_world):
    i = list(states["step"]).index(850)
    env = emu.EmuBatch(blob_path("softbox"), 2, prec=64, lpw=8)
    env.set_params(stiffness=np.full(2, 700.0))
    env.set_debug_world(1)
    env.set_state(states["q"][i], states["v"][i], states["act"][i], states["warm"][i]); env.set_ctrl([states["ctrl"][i]] * 2)
    env.step(1)
    w = make_world("softbox")
    w.set_state(states["q"][i], states["v"][i], states["act"][i], states["warm"][i]); w.set_ctrl([states["ctrl"][i]] * 2)
    w.step()
    for key, tol in (("con_dist", 1e-12), ("con_pos", 1e-12), ("con_frame", 1e-10), ("efc_aref", 1e-9), ("efc_R", 1e-11), ("efc_force", 1e-9)):
        a, b = env.debug(key), w.get(key)
        assert a.shape == b.shape, key
        np.testing.assert_allclose(a, b, atol=tol * max(1.0, np.abs(b).max()), err_msg=key)
    env.close()


def test_emulated_rollout_matches_oracle_episode_and_step_api(emu, batched, make_world):
    """Short squeeze episode on-chip (rollout mode) == oracle episode == the same episode through the step API."""
    sched = batched.default_schedule(2, n_settle=2, n_iter=8, open_close_div=4)
    W = 5
    ks = np.array([500.0, 900.0, 500.0, 1300.0, 900.0])
    env = emu.EmuBatch(blob_path("softbox"), W, prec=64, lpw=8)
    env.set_params(stiffness=ks)
    traj, touch, st = env.rollout(sched)
    assert (st == 0).all()
    np.testing.assert_array_equal(traj[0], traj[2])
    np.testing.assert_array_equal(traj[1], traj[4])
    for wi in (0, 3):
        ow = make_world("softbox", k=float(ks[wi]))
        rows, otouch, ost = ow.episode(n_settle=2, n_iter=8, open_close_div=4)
        scale = np.abs(rows).max(axis=0) + 1e-9
        assert (np.abs(traj[wi] - rows) / scale).max() < 1e-8
        np.testing.assert_array_equal(touch[wi], otouch)
    env2 = emu.EmuBatch(blob_path("softbox"), W, prec=64, lpw=8)
    env2.set_params(stiffness=ks)
    env2.reset(); env2.forward(); env2.step(1)
    ev, val = sched
    rows = []
    for t in range(ev.shape[0]):
        if ev[t]:
            env2.set_ctrl(val[t])
        s, _ = env2.step(7)
        rows.append(s)
    np.testing.assert_array_equal(np.stack(rows, 1), traj)
    env.close(); env2.close()


def test_emulated_multi_warp_cta_and_persistent_batches(emu, batched):
    """Several warps per CTA (shared step tables, one __syncthreads per step) and CTAs that walk more than one batch
    of worlds give the same bits as one-warp CTAs."""
    sched = batched.default_schedule(2, n_settle=1, n_iter=3, open_close_div=2)
    W = 21
    ks = 300.0 + 50.0 * np.arange(W)
    out = []
    for nw, lpw in ((1, 8), (4, 8), (2, 16), (8, 8)):
        env = emu.EmuBatch(blob_path("softbox"), W, prec=32, lpw=lpw, nw=nw)
        env.set_params(stiffness=ks)
        traj, touch, st = env.rollout(sched, want_touch=False)
        assert (st == 0).all() and np.isfinite(traj).all()
        out.append(traj)
        env.close()
    np.testing.assert_array_equal(out[0], out[1])
    np.testing.assert_array_equal(out[0], out[3])
    assert np.abs(out[0] - out[2]).max() / np.abs(out[0]).max() < 1e-4      # other lane count: other summation order


@pytest.mark.parametrize("prec,lpw,nw", [(32, 8, 2), (64, 8, 5), (32, 32, 1), (32, 4, 2), (64, 16, 3)])
def test_emulated_tensor_memory_rows_and_record_ring_are_bit_identical(emu, states, monkeypatch, prec, lpw, nw):
    """The equality rows in tensor memory (tcgen05.ld / st, one TMEM lane per thread) and the contact records read through
    the per-lane shared-memory ring compute the same bits as the rows in shared memory and the records read from the
    scratch: same arithmetic, other storage.  The emulator aborts on a tensor-memory address that is not uniform over
    the warp, outside the warp's lane quarter or outside the 512 columns; several warps per CTA exercise the column
    blocks of warps 4.. (nw = 5) and the quarters of warps 1..3."""
    W = (32 // lpw) * nw + 1
    out = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("SOFTGRIP_TMEM", mode)
        env = emu.EmuBatch(blob_path("softbox"), W, prec=prec, lpw=lpw, nw=nw)
        tm = env.debug("tensor_memory")
        esz, nrow = prec // 8, int(env.debug("sweep_schedule")[3])
        ring_fits = lpw * (2 * 32 * esz + 16) <= 2 * nrow * esz      # two 32-word records + skew per lane in the (aref, R) region
        assert (tm[0] > 0) == (mode == "1") and (tm[2] > 0) == (mode == "1" and ring_fits)
        assert ring_fits == (lpw <= 8)
        if mode == "1":
            words = 2 if prec == 32 else 4
            assert tm[1] == (env.debug("sweep_schedule")[0] + 1) * words and tm[0] >= tm[1] * ((nw + 3) // 4) and tm[0] <= 512
        env.set_params(stiffness=np.linspace(400.0, 1000.0, W))
        env.set_debug_world(W - 1)
        res = []
        for i in (len(states["step"]) - 1, int(np.argmax(states["ncon1"]))):     # late squeeze and the contact-richest snapshot
            env.set_state(states["q"][i], states["v"][i], states["act"][i], states["warm"][i])
            env.set_ctrl([states["ctrl"][i]] * 2)
            sens, touch = env.step(2)
            res.append((sens.copy(), touch.copy(), [x.copy() for x in env.get_state()], env.debug("efc_force").copy(), env.debug("solver_iter").copy()))
        assert (env.status() == 0).all()
        out[mode] = res
        env.close()
    for (s0, t0, g0, f0, it0), (s1, t1, g1, f1, it1) in zip(out["0"], out["1"]):
        np.testing.assert_array_equal(s0, s1)
        np.testing.assert_array_equal(t0, t1)
        for x, y in zip(g0, g1):
            np.testing.assert_array_equal(x, y)
        np.testing.assert_array_equal(f0, f1)
        np.testing.assert_array_equal(it0, it1)


@pytest.mark.parametrize("name,prec,lpw", [("softball", 32, 8), ("softcylinder", 64, 8), ("softbox_refined", 32, 32)])
def test_emulated_tensor_memory_rows_on_the_other_models(emu, batched, monkeypatch, name, prec, lpw):
    """The other shells (other row counts and sweep schedules; the refined composite at 32 lanes per world, where the
    window is 2 columns x (steps + 1) of a single column block and the record ring does not fit) through a short episode
    with the rows in tensor memory and in shared memory: same bits."""
    sched = batched.default_schedule(2, n_settle=1, n_iter=1, open_close_div=1)
    W = 32 // lpw + 1
    out = []
    for mode in ("0", "1"):
        monkeypatch.setenv("SOFTGRIP_TMEM", mode)
        env = emu.EmuBatch(blob_path(name), W, prec=prec, lpw=lpw)
        tm = env.debug("tensor_memory")
        assert (tm[0] > 0) == (mode == "1") and tm[0] <= 512
        env.set_params(stiffness=np.linspace(500.0, 900.0, W))
        traj, touch, st = env.rollout(sched)
        assert np.isfinite(traj).all() and np.abs(traj).max() > 0
        out.append((traj.copy(), [x.copy() for x in env.get_state()]))
        env.close()
    np.testing.assert_array_equal(out[0][0], out[1][0])
    for x, y in zip(out[0][1], out[1][1]):
        np.testing.assert_array_equal(x, y)


def test_emulated_dynamic_batch_hand_out_equals_fixed_shares(emu, states, monkeypatch):
    """More worlds than resident CTA slots: the persistent CTAs take their batches of worlds from a counter (default) or in
    fixed shares (SOFTGRIP_DYNAMIC=0).  Which CTA simulates a world does not enter its arithmetic: the two orders give
    the same bits, every world is simulated exactly once, and identical inputs give identical outputs in every batch.
    (The emulator's device has two SMs; one-warp CTAs of four worlds leave 18 resident slots.)"""
    W = 4 * 18 * 2 + 3
    i = int(np.argmax(states["ncon1"]))
    out = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("SOFTGRIP_DYNAMIC", mode)
        monkeypatch.setenv("SOFTGRIP_TMEM", "1")
        env = emu.EmuBatch(blob_path("softbox"), W, prec=32, lpw=8, nw=1)
        k = np.full(W, 700.0); k[5] = 450.0; k[W - 2] = 1200.0
        env.set_params(stiffness=k)
        env.set_state(states["q"][i], states["v"][i], states["act"][i], states["warm"][i])
        env.set_ctrl([states["ctrl"][i]] * 2)
        sens, touch = env.step(2)
        out[mode] = (sens.copy(), [x.copy() for x in env.get_state()])
        assert (env.status() == 0).all()
        env.close()
    np.testing.assert_array_equal(out["0"][0], out["1"][0])
    for x, y in zip(out["0"][1], out["1"][1]):
        np.testing.assert_array_equal(x, y)
    s = out["1"][0]
    same = [w for w in range(W) if w not in (5, W - 2)]
    assert (s[same] == s[0]).all() and not (s[5] == s[0]).all() and not (s[W - 2] == s[0]).all()


@pytest.mark.parametrize("W,nw", [(4, None), (18, 4)])
def test_emulated_divergence_is_contained_in_its_group(emu, W, nw):
    """A diverging world is reset and flagged; the other worlds of the same warp / CTA are bit-identical to a
    clean run (the re-run of mj_forward after the reset is taken by the whole CTA)."""
    env = emu.EmuBatch(blob_path("softbox"), W, prec=32, lpw=8, nw=nw)
    q = np.zeros((W, 118)); q[1, 30] = 1e11
    z = np.zeros((W, 118))
    env.set_state(q, z, np.zeros((W, 2)), z)
    env.step(2)
    st = env.status(clear=True)
    assert st[1] & 1 and st[0] == 0 and st[2] == 0 and st[3] == 0
    g = env.get_state()
    assert np.abs(g[0][1]).max() < 1e-3
    ref = emu.EmuBatch(blob_path("softbox"), W, prec=32, lpw=8, nw=nw)
    ref.set_state(z, z, np.zeros((W, 2)), z)
    ref.step(2)
    r = ref.get_state()
    for w in (0, 2, 3, W - 1):
        np.testing.assert_array_equal(g[0][w], r[0][w])
        np.testing.assert_array_equal(g[3][w], r[3][w])
    # acceleration blow-up inside the step (huge velocity): the reset + re-run path
    v = np.zeros((W, 118)); v[2, 40] = 1e9
    env.set_state(z, v, np.zeros((W, 2)), z)
    env.step(1)
    st = env.status(clear=True)
    g = env.get_state()
    assert st[2] & 1 and st[0] == 0 and st[1] == 0
    ref.set_state(z, z, np.zeros((W, 2)), z)
    ref.step(1)
    r = ref.get_state()
    for w in (0, 1, 3, W - 1):
        np.testing.assert_array_equal(g[0][w], r[0][w])
        np.testing.assert_array_equal(g[3][w], r[3][w])
    env.close(); ref.close()


@pytest.mark.parametrize("name", ["softball", "softcylinder"])
def test_emulated_other_models_first_steps(emu, make_world, name):
    env = emu.EmuBatch(blob_path(name), 1, prec=64, lpw=8)
    env.set_params(stiffness=np.full(1, 700.0))
    env.set_debug_world(0)
    w = make_world(name)
    w.reset()
    for step in range(8):
        q, v, a, ws = w.get_state()
        if w.step():
            break
        env.set_state(q, v, a, ws); env.set_ctrl([0, 0])
        env.step(1)
        q1, v1, a1, qacc = env.get_state()
        oq, ov, _, oacc = w.get_state()
        assert int(env.debug("ncon")[0]) == w.get_int("ncon")
        assert rel(q1[0], oq) < 1e-8 and rel(v1[0], ov) < 1e-8 and rel(qacc[0], oacc) < 1e-8, step
    assert step >= 5
    env.close()


def _decode_schedule(env):
    """-> nstep, lanes, bytes per real, nrow, modelled wavefronts, rows per slot, slots [nstep+1][lanes][2*rps], perm."""
    t = env.debug("sweep_schedule")
    nstep, lpw, esize, nrow = (int(x) for x in t[:4])
    rps = int(t[4] // 1e9)
    wavefronts = int(t[4] - 1e9 * rps)
    n = 2 * rps * (nstep + 1) * lpw
    sd = t[5:5 + n].astype(np.uint64).reshape(nstep + 1, lpw, 2 * rps)
    perm = t[5 + n:].astype(int)
    return nstep, lpw, esize, nrow, wavefronts, rps, sd, perm


@pytest.mark.parametrize("model,lpw,prec", [("softbox", 8, 32), ("softbox", 4, 32), ("softbox", 16, 64), ("softball", 8, 32), ("softcylinder", 8, 64),
                                            ("softbox_refined", 32, 32)])
def test_equality_sweep_schedule_is_a_valid_gauss_seidel_order(emu, model, lpw, prec):
    """Host logic of the equality sweep (sg_plan.hpp build_step_tables): one row per slot; every row is swept exactly
    once; within a step different lanes share no slider; rows that share a slider keep MuJoCo's order (an earlier step);
    the storage positions are a permutation; and the conflict-aware schedule costs no more modelled shared-memory
    wavefronts than the plain list schedule."""
    import importlib
    mjcf = importlib.import_module("soft-grip_b200.mjcf")
    A = mjcf.load_blob(blob_path(model)).arrays
    env = emu.EmuBatch(blob_path(model), 2, prec=prec, lpw=lpw)
    nstep, lpw_, esize, nrow, wavefronts, rps, sd, perm = _decode_schedule(env)
    assert rps == 1
    assert lpw_ == lpw and esize == prec // 8 and nrow == len(A["eq_obj1id"]) - 1
    assert sorted(perm.tolist()) == list(range(nrow))
    nfd = int((A["jnt_type"] == 3).sum())                      # hinge joints of the fingers come first
    key_to_eq = {}
    for r in range(nrow):
        d1, d2 = int(A["eq_obj1id"][r]) - nfd, int(A["eq_obj2id"][r])
        key_to_eq[(d1, d2 - nfd if d2 >= 0 else -1)] = r
    assert len(key_to_eq) == nrow
    when, seen_pos = {}, set()                                 # row -> step
    for s in range(nstep):
        owner = {}                                             # slider -> lane that touches it in this step
        for k in range(lpw):
            x, y = int(sd[s, k, 0]), int(sd[s, k, 1])
            if not (y >> 30) & 1:
                continue
            d1 = (x & 0xffff) // esize
            d2 = (x >> 16) // esize if (x >> 16) != 0xffff else -1
            pos = (y & 0x3fffffff) // (2 * esize)
            assert pos not in seen_pos and 0 <= pos < nrow
            seen_pos.add(pos)
            for d in (d1, d2):
                if d >= 0:
                    assert owner.setdefault(d, k) == k         # different lanes of a step touch disjoint sliders
            r = key_to_eq[(d1, d2)]
            assert r not in when
            when[r] = s
    assert len(when) == nrow
    assert all(not (int(sd[nstep, k, 1]) >> 30) & 1 for k in range(lpw))   # padding step
    last = {}
    for r in range(nrow):                                      # MuJoCo's sequential order
        for d in (int(A["eq_obj1id"][r]) - nfd, int(A["eq_obj2id"][r]) - nfd if A["eq_obj2id"][r] >= 0 else None):
            if d is None:
                continue
            if d in last:
                assert when[last[d]] < when[r]
            last[d] = r
    os.environ["SOFTGRIP_NO_BANK_SCHEDULE"] = "1"
    try:
        plain = emu.EmuBatch(blob_path(model), 2, prec=prec, lpw=lpw)
        nstep0, _, _, _, wavefronts0, _, _, perm0 = _decode_schedule(plain)
    finally:
        del os.environ["SOFTGRIP_NO_BANK_SCHEDULE"]
    assert perm0.tolist() == list(range(nrow))
    assert wavefronts + 6 * nstep <= wavefronts0 + 6 * nstep0


def test_removed_placement_options_fail_loudly(emu):
    """The shared-memory placement of the once-per-step data is gone from the step kernel: asking for it is an error, not
    a silent fallback."""
    with pytest.raises(RuntimeError, match="removed"):
        emu.EmuBatch(blob_path("softbox"), 2, prec=32, lpw=8, aux_smem=1)
    with pytest.raises(RuntimeError, match="removed"):
        emu.EmuBatch(blob_path("softbox"), 2, prec=32, lpw=8, qv_smem=1)
    with pytest.raises(RuntimeError, match="removed"):
        emu.EmuBatch(blob_path("softbox"), 2, prec=32, lpw=8, nw=4, team=1)


@pytest.mark.parametrize("model", ["softbox", "softball", "softcylinder"])
def test_broadphase_runs_reproduce_the_pair_list(emu, model):
    """Host logic of the collision tables (sg_plan.hpp): the run-length blocks the device broadphase walks expand to
    exactly the candidate pair list, in MuJoCo's contact order (b-major, collider-minor inside a block)."""
    env = emu.EmuBatch(blob_path(model), 2, prec=32, lpw=8)
    t = env.debug("pair_runs").astype(int)
    npair, nrun = int(t[0]), int(t[1])
    pairs = t[2:2 + 3 * npair].reshape(npair, 3)
    runs = t[2 + 3 * npair:].reshape(nrun, 4)
    out = []
    for pt, a, b0, nb in runs:
        a0, na = a & 255, a >> 8
        assert na >= 1 and nb >= 1
        for j in range(na * nb):
            out.append((pt, a0 + j % na, b0 + j // na))
    assert len(out) == npair and nrun < npair // 8          # the point of the encoding: long runs
    np.testing.assert_array_equal(np.array(out), pairs)
    env.close()


def test_emulated_contact_capacity_overflow_keeps_the_first_contacts(emu, states, mjcf, oracle, batched, tmp_path):
    """More contacts than the capacity (MuJoCo: nconmax warning): the first `maxcon` contacts in MuJoCo's order are kept,
    the rest dropped, status bit SG_ST_CON_FULL set -- same step as the oracle with the same nconmax."""
    cap = 16
    model = mjcf.load_blob(blob_path("softbox"))
    model.opt["nconmax"] = cap
    blob = mjcf.model_to_blob(model)
    p = tmp_path / "softbox_cap.sgm"
    p.write_bytes(blob)
    om = oracle.OracleModel(blob)
    ow = oracle.OracleWorld(om)
    ow.set_geom_mask(batched.geom_name_mask(model.names["geom"], "OBJ", ("g12", "g2")))
    ow.set_stiffness(700.0)
    os.environ["SOFTGRIP_MAXCON"] = str(cap)
    try:
        env = emu.EmuBatch(str(p), 5, prec=64, lpw=8)
    finally:
        os.environ.pop("SOFTGRIP_MAXCON", None)
    env.set_params(stiffness=np.full(5, 700.0))
    env.set_debug_world(4)
    for i in (4, 6, 7):                               # 8 (fits), 35 and 58 contacts
        env.set_state(states["q"][i], states["v"][i], states["act"][i], states["warm"][i])
        env.set_ctrl([states["ctrl"][i]] * 2)
        env.status(clear=True)
        env.step(1)
        q1, v1, a1, qacc = env.get_state()
        ow.set_state(states["q"][i], states["v"][i], states["act"][i], states["warm"][i])
        ow.set_ctrl([states["ctrl"][i]] * 2)
        ost = ow.step()
        oq, ov, oa, owarm = ow.get_state()
        full = states["ncon1"][i] > cap
        # "ncon" counts every detected contact, "ncon_rows" the ones that were given constraint rows (the capped list)
        assert int(env.debug("ncon")[0]) == int(states["ncon1"][i])
        assert int(env.debug("ncon_rows")[0]) == min(cap, int(states["ncon1"][i])) == ow.get_int("ncon")
        assert bool(ost & 2) == full and all(bool(s & 2) == full for s in env.status())
        assert rel(q1[-1], oq) < 1e-9 and rel(v1[-1], ov) < 1e-9 and rel(qacc[-1], owarm) < 1e-9
    env.close()


# SURVEY App. E: under the restated semantics the volume mode is stable iff (1 + n d_t / d_j) / 65.7 < 2, i.e. n d_t < ~130 d_j:
# ball / cylinder (n = 218 / 192) need a volume-tendon damper d_t <= ~70, the refined softbox of BASELINE configs[4]
# (7x9x13 grid, n = 434) d_t <= ~30; the committed files have d_t = d_j = 100.  These are the stated stable values.
STABLE_TENDON_DAMPING = {"softball": 50.0, "softcylinder": 50.0, "softbox_refined": 20.0}


def _protocol_ctrl(step):
    """ctrl of create_dataset's episode at physics step `step` (ref: create_dataset.py:33-60 with sim_start 1, sim_step 7)."""
    return 0.0 if step < 281 else (-0.2 if step < 841 else 0.2)


@pytest.mark.parametrize("prec", [64, 32])
@pytest.mark.parametrize("name", ["softball", "softcylinder", "softbox_refined"])
def test_emulated_other_models_along_a_stabilised_episode(emu, make_world, name, prec):
    """SURVEY 8d cfg 3: softball / softcylinder run away under the restated semantics at the committed tendon damper; with
    the damper at a stable value (stated above) the whole squeeze episode runs clean in the oracle, and the kernel source
    agrees with it step for step from snapshots taken all along that episode (settle, closing, peak contact, release)."""
    w = make_world(name)
    w.set_tendon_damping(0, STABLE_TENDON_DAMPING[name])
    w.reset()
    snaps, want = {}, (0, 150, 285, 500, 838, 1000, 1395)
    for step in range(1401):
        w.set_ctrl([_protocol_ctrl(step)] * 2)
        if step in want:
            snaps[step] = w.get_state()
        assert w.step() == 0, step                       # no divergence, no capacity / unsupported-pair flags
        if step in want:
            snaps[step] = (snaps[step], w.get_state(), w.get_int("ncon"))
    q_end = w.get_state()[0]
    assert np.isfinite(q_end).all() and np.abs(q_end).max() < 1.0
    env = emu.EmuBatch(blob_path(name), 2, prec=prec, lpw=8)
    env.set_params(stiffness=np.full(2, 700.0), tdamping=np.full(2, STABLE_TENDON_DAMPING[name]))
    env.set_debug_world(1)
    ncons = []
    for step in want:
        (q, v, a, ws), (oq, ov, oa, oacc), ncon = snaps[step]
        env.set_state(q, v, a, ws); env.set_ctrl([_protocol_ctrl(step)] * 2)
        env.step(1)
        q1, v1, a1, qacc = env.get_state()
        assert int(env.debug("ncon")[0]) == ncon
        err = {"q": rel(q1[1], oq), "v": rel(v1[1], ov), "qacc": rel(qacc[1], oacc)}
        for key, e in err.items():
            assert e < (1e-8 if prec == 64 else FP32_TOL_OTHER[key]), (step, key, e)
        assert rel(a1[1], oa) < (1e-12 if prec == 64 else 1e-6), step
        ncons.append(ncon)
    assert (env.status() == 0).all() and max(ncons) > min(ncons)
    env.close()


def test_c_abi_rejects_empty_and_malformed_requests(emu):
    """Empty / malformed inputs at the boundary are error returns with a message, never a launch: zero sub-steps, an empty
    or negative schedule, null buffers, zero worlds, unknown precision, a device that does not exist."""
    import ctypes as C
    lib_ = importlib.import_module("soft-grip_b200._lib")
    env = emu.EmuBatch(blob_path("softbox"), 1, prec=32, lpw=8)
    env.reset()
    L = env.L
    err = lambda: L.sg_last_error().decode()
    for nsub in (0, -1):
        assert L.sg_batch_step(env.b, nsub, None, None, None) < 0 and "nsub" in err()
    traj = np.zeros((1, 3, 12), dtype=np.float32)
    ev, val = np.zeros(3, dtype=np.int32), np.zeros((3, 2))
    pe, pv = ev.ctypes.data_as(C.POINTER(C.c_int)), val.ctypes.data_as(C.POINTER(C.c_double))
    for T, sim_step, sim_start, ok in ((0, 7, 1, False), (3, 0, 1, False), (3, -1, 1, False), (3, 7, -1, False), (3, 7, 0, True), (3, 7, 1, True)):
        sc = lib_.SgSchedule(sim_start, sim_step, T, pe, pv)
        rc = L.sg_batch_rollout(env.b, C.byref(sc), traj.ctypes.data_as(C.c_void_p), None, None)
        assert (rc == 0) == ok, (T, sim_step, sim_start, err())
        if not ok:
            assert "schedule" in err()
    assert np.isfinite(traj).all()
    sc = lib_.SgSchedule(1, 7, 3, None, None)
    assert L.sg_batch_rollout(env.b, C.byref(sc), traj.ctypes.data_as(C.c_void_p), None, None) < 0 and "schedule" in err()
    sc = lib_.SgSchedule(1, 7, 3, pe, pv)
    assert L.sg_batch_rollout(env.b, C.byref(sc), None, None, None) < 0 and "null" in err()
    b = C.c_void_p()
    assert L.sg_batch_create(env.m, 0, 0, 32, C.byref(b)) < 0 and "nworlds" in err()
    assert L.sg_batch_create(env.m, 1, 0, 16, C.byref(b)) < 0 and "precision" in err()
    assert L.sg_batch_create(env.m, 1, 5, 32, C.byref(b)) < 0 and "device" in err()
    assert L.sg_batch_set_debug_world(env.b, 7) < 0 and "range" in err()
    env.close()


@pytest.mark.parametrize("name,lpw", [("softbox_refined", 16), ("softbox_refined", 32), ("softball", 16)])
def test_emulated_larger_models_at_more_lanes_per_world(emu, make_world, name, lpw):
    """The lane counts DESIGN.md section 7 proposes for the larger models (shorter equality sweeps): same step parity at
    peak contact as the default 8 lanes, and the sweep really is shorter."""
    w = make_world(name)
    w.set_tendon_damping(0, STABLE_TENDON_DAMPING[name])
    w.reset()
    for step in range(839):
        w.set_ctrl([_protocol_ctrl(step)] * 2)
        before = w.get_state()
        assert w.step() == 0
    oq, ov, oa, oacc = w.get_state()
    steps = {}
    for lanes in (8, lpw):
        env = emu.EmuBatch(blob_path(name), 32 // lanes + 1, prec=64, lpw=lanes)
        W = 32 // lanes + 1
        env.set_params(stiffness=np.full(W, 700.0), tdamping=np.full(W, STABLE_TENDON_DAMPING[name]))
        env.set_debug_world(W - 1)
        env.set_state(*before); env.set_ctrl([_protocol_ctrl(838)] * 2)
        env.step(1)
        q1, v1, a1, qacc = env.get_state()
        assert int(env.debug("ncon")[0]) == w.get_int("ncon") > 20
        assert rel(q1[-1], oq) < 1e-8 and rel(v1[-1], ov) < 1e-8 and rel(qacc[-1], oacc) < 1e-8
        steps[lanes] = int(env.debug("sweep_schedule")[0])
        env.close()
    assert steps[lpw] < 0.8 * steps[8], steps


def test_emulated_step_kernel_is_clean_under_asan(tmp_path):
    """The kernel source and the C-ABI host logic built with -fsanitize=address (emulator build) and driven through steps and
    rollouts over precisions, lanes per world, multi-warp CTAs and the larger models (tests/simt/asan_drive.py): no heap
    out-of-bounds access anywhere on the path."""
    import shutil
    import subprocess
    if os.environ.get("SOFTGRIP_ASAN") != "1":
        pytest.skip("opt-in (SOFTGRIP_ASAN=1): the sanitizer run of the whole step kernel takes 5-20 minutes; last run clean, see DESIGN.md")
    libasan = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(libasan) or not os.path.exists(libasan):
        pytest.skip("no libasan")
    simt = os.path.join(ROOT, "tests", "simt")
    for f in ("Makefile", "simt.h", "cuda_shim.h"):
        shutil.copy(os.path.join(simt, f), str(tmp_path))
    csrc = os.path.join(ROOT, "soft-grip_b200", "csrc")
    flags = "-O1 -g -std=c++17 -fPIC -DSG_SIMT_EMU -I. -I%s -fsanitize=address -fno-omit-frame-pointer -Wno-unknown-pragmas" % csrc
    subprocess.check_call(["make", "-s", "-j8", "-C", str(tmp_path), "CSRC=" + csrc, "CXXFLAGS=" + flags], stdout=subprocess.DEVNULL)
    env = dict(os.environ, LD_PRELOAD=libasan, ASAN_OPTIONS="detect_leaks=0:detect_stack_use_after_return=0:halt_on_error=1")
    out = subprocess.run([sys.executable, os.path.join(simt, "asan_drive.py"), ROOT, str(tmp_path / "libsoftgrip_simt.so")],
                         capture_output=True, text=True, env=env, timeout=3000)
    assert out.returncode == 0 and "ASAN DRIVE DONE" in out.stdout, (out.stdout[-500:], out.stderr[-3000:])
    assert "ERROR: AddressSanitizer" not in out.stderr


def test_launch_geometry_fills_every_sm_in_one_pass(emu):
    """sg_batch_create picks the CTA size from the batch size (DESIGN.md section 3): the emulated device has 2 SMs, so
    112 softbox worlds run as 2 CTAs of 56 worlds (14 warps) in one pass rather than as 64 + 48, a batch that needs
    several passes takes the largest CTA, a handful of worlds takes one small CTA -- and the bits do not depend on it."""
    import ctypes as C

    def geometry(W, nw=None):
        env = emu.EmuBatch(blob_path("softbox"), W, prec=32, lpw=8, nw=nw)
        out = (C.c_int * 8)()
        assert env.L.sg_batch_config(env.b, out) == 0
        return env, {"warps_per_cta": out[1], "worlds_per_cta": out[2]}

    env, g = geometry(112)
    assert g == {"warps_per_cta": 14, "worlds_per_cta": 56}
    env.close()
    env, g = geometry(1000)
    assert g["warps_per_cta"] == 16
    env.close()
    env, g = geometry(3)
    assert g["warps_per_cta"] == 1
    env.close()
    env, g = geometry(112, nw=16)                       # the development override still wins
    assert g["warps_per_cta"] == 16
    env.close()
