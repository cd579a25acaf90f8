"""Host-side logic: episode schedule, per-world RNG, dataset format, driver CLI, sharding (gloo, world_size 2)."""
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, blob_path, pkg


def test_default_schedule_is_the_reference_protocol(batched):
    """ctrl = 0 for 40 rows, close_hand at row 40, toggle (-> +0.2) at row 120 only (ref: create_dataset.py:41-60)."""
    ev, val = batched.default_schedule(2)
    assert ev.shape == (200,) and val.shape == (200, 2)
    assert list(np.nonzero(ev)[0]) == [40, 120]
    np.testing.assert_array_equal(val[40], [-0.2, -0.2]); np.testing.assert_array_equal(val[120], [0.2, 0.2])
    ev2, val2 = batched.default_schedule(2, n_settle=5, n_iter=50, open_close_div=20)
    assert list(np.nonzero(ev2)[0]) == [5, 25, 45] and val2[25, 0] == 0.2 and val2[45, 0] == -0.2


def test_world_uniform_is_sharding_invariant(batched):
    full = batched.world_uniform(7, np.arange(1000), 300, 1400, stream=3)
    parts = np.concatenate([batched.world_uniform(7, np.arange(a, b), 300, 1400, stream=3) for a, b in ((0, 250), (250, 600), (600, 1000))])
    np.testing.assert_array_equal(full, parts)
    assert full.min() >= 300 and full.max() <= 1400 and abs(full.mean() - 850) < 30
    assert not np.array_equal(full, batched.world_uniform(8, np.arange(1000), 300, 1400, stream=3))
    assert not np.array_equal(full, batched.world_uniform(7, np.arange(1000), 300, 1400, stream=4))


def test_geom_name_mask(batched):
    names = ["ground", None, "g121", "g122", "g21", "g23", "OBJGcenter", "OBJG2_1_0"]
    m = batched.geom_name_mask(names, "OBJ", ("g12", "g2"))
    assert list(m) == [0, 0, 2, 2, 4, 4, 1, 1]          # 'g2' must not match g122, 'G2' (upper case) must not match


def test_dataset_pickle_layout(tmp_path):
    ds = pkg("dataset")
    traj = np.random.default_rng(0).normal(size=(5, 200, 12)).astype(np.float32)
    k = np.linspace(300, 1400, 5)
    p = tmp_path / "d" / "x.pickle"
    ds.write_pickle(str(p), traj, k)
    raw = pickle.load(open(p, "rb"))
    assert sorted(raw) == ["data", "stiffness"] and len(raw["data"]) == 5
    assert raw["data"][0].shape == (200, 12) and raw["data"][0].dtype == np.float64 and isinstance(raw["stiffness"][0], float)
    x, y = ds.read_pickle(str(p))                      # what functions/utils.create_tf_generators does
    assert x.shape == (5, 200, 12) and y.shape == (5,)
    np.testing.assert_allclose(x, traj.astype(np.float64))
    masked = ds.mask_contact(traj, np.zeros((5, 200), dtype=bool))
    assert not masked.any()
    edges, stats = ds.feature_stats(x, y, nbins=2)
    assert stats[0]["n"] + stats[1]["n"] == 5 and stats[0]["mean"].shape == (4,)


def test_create_dataset_cli_flags():
    sys.path.insert(0, os.path.join(ROOT, "soft-grip_b200"))
    cd = pkg("create_dataset")
    args, _ = cd.build_parser().parse_known_args(["--mujoco-model-paths", "a.xml", "b.xml", "--vis", "False"])
    assert args.sim_step == 7 and args.sim_start == 1 and args.mujoco_model_paths == ["a.xml", "b.xml"]
    assert args.vis is True                  # type=bool quirk kept (SURVEY App. C item 7)
    assert args.data_name == "dataset_all_shapes" and args.mask_contact is False
    assert (cd.NUM_EPISODES, cd.MAX_ITER_PER_EP, cd.OPEN_CLOSE_DIV, cd.START_STEP) == (1, 160, 80, 40)


def test_episode_rows_protocol():
    """episode_rows drives the ManEnv verbs in the reference order (fake env, no GPU)."""
    cd = pkg("create_dataset")

    class Fake:
        def __init__(self): self.log = []; self.n = 0
        def step(self): self.n += 1; self.log.append("s"); return np.full(12, float(self.n)), self.n % 2 == 0
        def close_hand(self): self.log.append("close")
        def toggle_grip(self): self.log.append("toggle")
        def render(self): pass

    env = Fake()
    rows = list(cd.episode_rows(env, mask_contact=True))
    assert len(rows) == 200
    assert env.log.index("close") == 40 and env.log.count("toggle") == 1
    assert env.log.index("toggle") == 40 + 1 + 80          # before the 81st squeeze step
    assert rows[0].sum() == 0 and rows[1].sum() == 24       # odd steps masked (no contact), even kept


def test_manenv_surface_matches_reference():
    sys.path.insert(0, os.path.join(ROOT, "soft-grip_b200"))
    from environment import ManEnv
    from environment.interface import Env
    assert issubclass(ManEnv, Env)
    assert ManEnv.joint_ids == list(range(11, 64)) and ManEnv.tendon_ids == [0]
    assert ManEnv.obj_name == "OBJ" and list(ManEnv._finger_names0) == ["g12", "g2"]
    for name in ("step", "reset", "get_sensor_sensordata", "toggle_grip", "close_hand", "loose_hand", "set_new_stiffness",
                 "get_env", "render", "load_env", "get_std_spec"):
        assert callable(getattr(ManEnv, name))

    class A: sim_start = 1; sim_step = 7; mujoco_model_paths = ["x.xml"]; vis = False
    assert ManEnv.get_std_spec(A) == {"sim_start": 1, "sim_step": 7, "env_paths": ["x.xml"], "is_vis": False}
    with pytest.raises(NotImplementedError):
        Env(1, 7).step()


def test_bench_shard_plan():
    sys.path.insert(0, ROOT)
    import bench
    for n in (1, 2, 4, 8):
        shards = [bench.shard_range(1000, r, n) for r in range(n)]
        assert shards[0][0] == 0 and shards[-1][1] == 1000
        assert all(shards[i][1] == shards[i + 1][0] for i in range(n - 1))
    assert bench.shard_range(10, 3, 4) == (9, 10)


WORKER = r'''
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
import bench
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
lo, hi = bench.shard_range(64, rank, world)
import importlib
batched = importlib.import_module("soft-grip_b200.batched")
k = batched.world_uniform(0, np.arange(lo, hi), 300, 1400)
ms = 10.0 + rank
tmax = bench.max_over_ranks(ms, torch.device("cpu"))
total = bench.sum_over_ranks(float(hi - lo), torch.device("cpu"))
gathered = [None] * world
dist.all_gather_object(gathered, k)
if rank == 0:
    full = batched.world_uniform(0, np.arange(64), 300, 1400)
    assert np.array_equal(np.concatenate(gathered), full)
    assert tmax == 10.0 + world - 1 and total == 64.0
    print("OK")
dist.destroy_process_group()
'''


def test_two_rank_sharding_with_gloo(tmp_path):
    """N>1 host path on CPU: contiguous world shards, max-over-ranks timing, shard gather == unsharded draw."""
    pytest.importorskip("torch")
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29617")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                          "127.0.0.1", "--master-port", "29617", str(script), ROOT], capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "OK" in out.stdout


def test_regenerate_plans_the_reference_file_tree_with_disjoint_samples(tmp_path):
    """BASELINE configs[3]: the simulated files run_experiments.sh consumes (ref: run_experiments.sh:2-7), each in the
    pickle layout of create_dataset.py:75-78, no sample shared between files; driven by a stub rollout (no GPU)."""
    rg = pkg("regenerate")
    ds = pkg("dataset")
    batched = pkg("batched")
    plan = rg.plan_files(10, 4, 3)
    stems = [s for s, _ in plan]
    assert stems == ["sim_box/train", "sim_box/val", "sim_all/train", "sim_all/softball_testing", "sim_all/softbox_testing",
                     "sim_all/softcylinder_testing"]
    used = {}
    for stem, parts in plan:
        for shape, first, count in parts:
            ids = set(range(first, first + count))
            assert not (ids & used.setdefault(shape, set()))
            used[shape] |= ids
    assert sum(c for _, _, c in dict(plan)["sim_all/train"]) == 10 and [c for _, _, c in dict(plan)["sim_all/train"]] == [4, 3, 3]
    assert rg.plan_files(6, 2, 2, shapes=("softbox",))[2] == ("sim_all/train", [("softbox", 8, 6)])

    calls = []

    def rollouts(shape, first, count):
        calls.append((shape, first, count))
        for a in range(0, count, 4):                      # chunks of 4 worlds per "launch"
            n = min(4, count - a)
            ids = np.arange(first + a, first + a + n)
            k = batched.world_uniform(0, ids, 300.0, 1400.0)
            traj = np.broadcast_to(k[:, None, None], (n, 200, 12)).astype(np.float32) + SHAPE_TAG[shape]
            st = np.where(ids % 7 == 5, 1, 0)              # some worlds "diverged"
            yield traj, k, st

    SHAPE_TAG = {"softball": 0.0, "softbox": 10000.0, "softcylinder": 20000.0}
    out = rg.regenerate(str(tmp_path), 10, 4, 3, rollouts, stats_fn=lambda t: (np.mean(t, axis=(0, 1)), np.std(t, axis=(0, 1))),
                        npz=True, log=lambda *_: None)
    assert [o["file"] for o in out] == [str(tmp_path / (s + ".pickle")) for s in stems]
    seen = {}
    for o, (stem, parts) in zip(out, plan):
        x, y = ds.read_pickle(o["file"])                   # what functions/utils.create_tf_generators does
        want_n = sum(c for _, _, c in parts) - o["diverged"]
        assert x.shape == (want_n, 200, 12) and y.shape == (want_n,) and o["samples"] == want_n
        assert ((y >= 300) & (y <= 1400)).all()
        st = np.load(str(tmp_path / (stem + ".stats.npz")))
        assert int(st["n"]) == want_n and np.allclose(st["mean"], x.mean(axis=(0, 1))) and st["std"].shape == (12,)
        z = np.load(str(tmp_path / (stem + ".npz")))
        assert z["data"].dtype == np.float32 and z["data"].shape == x.shape
        for xi, yi in zip(x, y):                           # (shape tag, stiffness) identifies a sample: no file shares one
            key = (round(float(xi[0, 0] - yi), -3), float(yi))
            assert key not in seen, (stem, seen.get(key))
            seen[key] = stem
    assert sum(o["diverged"] for o in out) > 0
    kept = rg.regenerate(str(tmp_path / "all"), 10, 4, 3, rollouts, drop_diverged=False, log=lambda *_: None)
    assert [o["samples"] for o in kept] == [10, 4, 10, 3, 3, 3]
    # noise_seed is handed to the rollouts of the */train files only
    calls.clear()
    noisy = []

    def rollouts_n(shape, first, count, noise_seed=None):
        noisy.append((shape, first, noise_seed))
        return rollouts(shape, first, count)

    rg.regenerate(str(tmp_path / "noise"), 10, 4, 3, rollouts_n, log=lambda *_: None, noise_seed=5)
    assert [n for _, _, n in noisy] == [5, None, 5, 5, 5, None, None, None]


def test_bench_traj_kernel_probe_never_raises():
    """bench.py's informational `traj_kernels` key: without a device the probe reports the error instead of raising, so it
    can never take the headline JSON line down with it."""
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    sys.path.insert(0, ROOT)
    import bench
    out = bench.measure_traj_kernels(torch, torch.zeros(4, 200, 12), torch.zeros(16, dtype=torch.uint8), 6546.2)
    assert list(out) == ["error"] and out["error"]


@pytest.mark.parametrize("world", [2, 3, 8])
def test_regenerate_shards_merge_to_the_single_gpu_tree(tmp_path, world):
    """SURVEY section 8e: worlds shard over ranks with no collective; the only exchange is the final gather of dataset
    shards, and the merged files equal the single-GPU files sample for sample (stub rollouts, no GPU)."""
    rg, ds, batched = pkg("regenerate"), pkg("dataset"), pkg("batched")
    tag = {"softball": 0.0, "softbox": 10000.0, "softcylinder": 20000.0}

    def rollouts(shape, first, count):
        for a in range(0, count, 5):
            n = min(5, count - a)
            ids = np.arange(first + a, first + a + n)
            k = batched.world_uniform(3, ids, 300.0, 1400.0)
            yield np.broadcast_to(k[:, None, None], (n, 200, 12)) + tag[shape], k, np.where(ids % 6 == 1, 1, 0)

    single = rg.regenerate(str(tmp_path / "one"), 11, 5, 4, rollouts, log=lambda *_: None)
    stems = None
    for r in range(world):
        stems = rg.regenerate_shard(str(tmp_path / "many"), 11, 5, 4, rollouts, r, world)
    merged = rg.merge_shards(str(tmp_path / "many"), stems, world, ds)
    assert [m["samples"] for m in merged] == [s["samples"] for s in single]
    for m, s1 in zip(merged, single):
        xa, ya = ds.read_pickle(s1["file"])
        xb, yb = ds.read_pickle(m["file"])
        assert (xa == xb).all() and (ya == yb).all()
    assert not [f for f in os.listdir(str(tmp_path / "many" / "sim_all")) if ".rank" in f]       # shard files removed
    # every world id of a part lands on exactly one rank
    for _, parts in rg.plan_files(11, 5, 4):
        for part in parts:
            got = sorted(i for r in range(world) for (_, f, c) in rg.shard_parts([part], r, world) for i in range(f, f + c))
            assert got == list(range(part[1], part[1] + part[2]))


REGEN_WORKER = r'''
import importlib, os, sys, numpy as np
sys.path.insert(0, sys.argv[1])
rg = importlib.import_module("soft-grip_b200.regenerate")
batched = importlib.import_module("soft-grip_b200.batched")
def rollouts(shape, first, count):
    ids = np.arange(first, first + count)
    k = batched.world_uniform(1, ids, 300.0, 1400.0)
    yield np.broadcast_to(k[:, None, None], (count, 200, 12)) + len(shape), k, np.zeros(count, dtype=np.int32)
out = rg.regenerate_distributed(sys.argv[2], 9, 3, 2, rollouts, backend="gloo")
if int(os.environ["RANK"]) == 0:
    one = rg.regenerate(sys.argv[2] + "_one", 9, 3, 2, rollouts, log=lambda *_: None)
    ds = importlib.import_module("soft-grip_b200.dataset")
    for a, b in zip(out, one):
        xa, ya = ds.read_pickle(a["file"]); xb, yb = ds.read_pickle(b["file"])
        assert a["samples"] == b["samples"] and (xa == xb).all() and (ya == yb).all()
    print("OK")
else:
    assert out is None
'''


def test_two_rank_dataset_regeneration_with_gloo(tmp_path):
    """The N>1 dataset path end to end on CPU (gloo, world_size 2, stub rollouts): shard files, barrier, rank-0 merge."""
    pytest.importorskip("torch")
    script = tmp_path / "regen_worker.py"
    script.write_text(REGEN_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29618")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                          "127.0.0.1", "--master-port", "29618", str(script), ROOT, str(tmp_path / "tree")],
                         capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "OK" in out.stdout


def test_bench_sensor_trace_error_against_the_oracle(oracle):
    """bench.py's sensor_trace_error: zero for the oracle's own traces (with every per-world parameter of BASELINE configs[2]:
    stiffness, shell damping, object offset), the perturbation otherwise, and an error key (never an exception) when it
    cannot run."""
    sys.path.insert(0, ROOT)
    import argparse
    import bench
    args = argparse.Namespace(tendon_damping=None)
    info = bench._model_info(blob_path("softbox"))
    assert info[:3] == (8, 118, 10) and np.allclose(info[3], [1.7, 0.0, 1.0])
    w = oracle.OracleWorld(oracle.OracleModel(open(blob_path("softbox"), "rb").read()))
    ks, ds, offs = [400.0, 900.0], [120.0, 180.0], [[0.01, -0.02, 0.03], [0.0, 0.04, -0.05]]
    rows = []
    for k, d, off in zip(ks, ds, offs):
        w.set_stiffness(k)
        for dof in range(8, 118):
            w.set_dof_damping(dof, d)
        w.set_body_pos(10, np.array([1.7, 0, 1.0]) + off)
        rows.append(w.episode()[0])
    out = bench.sensor_trace_error(args, blob_path("softbox"), np.array(rows), (ks, ds, offs))
    assert out["worlds"] == 2 and out["settle_rows_max_rel"] == 0.0 and out["row_max_rel"] == 0.0
    plain = bench.sensor_trace_error(args, blob_path("softbox"), np.array(rows), (ks, None, None))
    assert plain["row_max_rel"] > 1e-3                       # the damping / offset really change the traces
    bumped = np.array(rows) * (1 + 1e-3)
    out = bench.sensor_trace_error(args, blob_path("softbox"), bumped, (ks, ds, offs))
    assert 5e-4 < out["row_max_rel"] < 2e-3 and 0 < out["settle_rows_max_rel"] < 2e-3
    assert "error" in bench.sensor_trace_error(args, "/nonexistent.sgm", bumped, (ks, ds, offs))


def test_bench_world_params_do_not_depend_on_the_sharding():
    """BASELINE configs[2] parameters are functions of (seed, step, global world id): any shard draws the same values."""
    sys.path.insert(0, ROOT)
    import argparse
    import bench
    args = argparse.Namespace(randomise="all", fixed_stiffness=None, seed=3, damping_range=[100.0, 200.0], offset_range=0.05)
    k, d, off = bench.world_params(args, np.arange(0, 64), 5)
    k2, d2, off2 = bench.world_params(args, np.arange(32, 64), 5)
    assert np.array_equal(k[32:], k2) and np.array_equal(d[32:], d2) and np.array_equal(off[32:], off2)
    assert 300 <= k.min() and k.max() <= 1400 and 100 <= d.min() and d.max() <= 200 and np.abs(off).max() <= 0.05 and off.shape == (64, 3)
    assert not np.array_equal(k, bench.world_params(args, np.arange(0, 64), 6)[0])
    ks, ds, offs = bench.world_params(args, np.arange(8), 0, "stiffness")
    assert ds is None and offs is None
    args.fixed_stiffness = 700.0
    assert np.all(bench.world_params(args, np.arange(8), 0)[0] == 700.0)


def test_bench_dump_outputs_is_a_fixed_bounded_sample(tmp_path):
    """bench.py --dump-outputs: the whole trajectory buffer when it fits, otherwise the same seeded sample of worlds on every
    run, in the batch precision, under 64 MB in all, with the global ids of the worlds it holds."""
    torch = pytest.importorskip("torch")
    sys.path.insert(0, ROOT)
    import bench
    small = torch.arange(5 * 200 * 12, dtype=torch.float32).reshape(5, 200, 12)
    bench.dump_outputs(str(tmp_path / "small"), small, 10)
    assert np.array_equal(np.load(str(tmp_path / "small" / "traj.npy")), small.numpy())
    assert np.array_equal(np.load(str(tmp_path / "small" / "traj_worlds.npy")), np.arange(10.0, 15.0))
    big = torch.randn(4096, 200, 12, dtype=torch.float64, generator=torch.Generator().manual_seed(0))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), big, 100)
    files = sorted(os.listdir(str(tmp_path / "a")))
    assert files == ["traj.npy", "traj_worlds.npy"]
    assert sum(os.path.getsize(str(tmp_path / "a" / f)) for f in files) <= 64 * 10 ** 6
    ids = np.load(str(tmp_path / "a" / "traj_worlds.npy"))
    traj = np.load(str(tmp_path / "a" / "traj.npy"))
    assert ids.dtype == np.float64 and traj.dtype == np.float64 and 1000 < len(ids) < 4096 and (np.diff(ids) > 0).all()
    assert np.array_equal(traj, big.numpy()[ids.astype(int) - 100])
    for f in files:
        assert np.array_equal(np.load(str(tmp_path / "a" / f)), np.load(str(tmp_path / "b" / f)))


def test_regenerate_multi_rank_noise_flags_and_statistics(tmp_path):
    """ADVICE r1: the multi-rank path passes the noise seed to the */train files (a draw depends on the global world id only, so
    the merged file equals the single-rank one), counts every status flag, drops every flagged world, and writes the per-file
    statistics on rank 0 after the merge; a rollouts object with `prefetch` is asked for every shape once (stub rollouts)."""
    rg, ds, batched = pkg("regenerate"), pkg("dataset"), pkg("batched")
    tag = {"softball": 0.0, "softbox": 10000.0, "softcylinder": 20000.0}

    class Rollouts:
        def __init__(self):
            self.calls, self.prefetched = [], []

        def prefetch(self, files):
            self.prefetched.append(sorted({shape for _, parts in files for shape, _, _ in parts}))

        def __call__(self, shape, first, count, noise_seed=None):
            self.calls.append((shape, first, count, noise_seed))
            ids = np.arange(first, first + count)
            k = batched.world_uniform(3, ids, 300.0, 1400.0)
            x = np.broadcast_to(k[:, None, None], (count, 200, 12)) + tag[shape]
            if noise_seed is not None:                       # stand-in for the device noise: a function of (seed, shape, world id)
                x = x + (noise_seed + 1) * 1e-3 * (ids[:, None, None] % 17)
            st = np.where(ids % 6 == 1, 1, 0) | np.where(ids % 10 == 3, 2, 0) | np.where(ids % 15 == 7, 8, 0)
            yield x, k, st

    one = Rollouts()
    single = rg.regenerate(str(tmp_path / "one"), 11, 5, 4, one, log=lambda *_: None, noise_seed=5)
    assert one.prefetched == [["softball", "softbox", "softcylinder"]]
    many = Rollouts()
    stems = None
    for r in range(3):
        stems = rg.regenerate_shard(str(tmp_path / "many"), 11, 5, 4, many, r, 3, noise_seed=5)
    merged = rg.merge_shards(str(tmp_path / "many"), stems, 3, ds)
    noisy = {c[:3] for c in many.calls if c[3] == 5}
    assert noisy and all(c[3] is None or c[3] == 5 for c in many.calls)
    for m, s1 in zip(merged, single):
        xa, ya = ds.read_pickle(s1["file"])
        xb, yb = ds.read_pickle(m["file"])
        assert (xa == xb).all() and (ya == yb).all()
        for key in ("diverged", "capacity", "unsupported", "dropped", "samples"):
            assert m[key] == s1[key], (m["file"], key)
        sa, sb = np.load(s1["file"].replace(".pickle", ".stats.npz")), np.load(m["file"].replace(".pickle", ".stats.npz"))
        assert int(sb["n"]) == m["samples"] and int(sb["dropped"]) == m["dropped"]
        np.testing.assert_allclose(sb["mean"], xb.mean(axis=(0, 1)), rtol=1e-12)
        np.testing.assert_allclose(sb["std"], xb.std(axis=(0, 1)), rtol=1e-12)
    # flagged worlds (any of the three bits) are not in the files
    x, k = ds.read_pickle(single[0]["file"])                # sim_box/train: softbox worlds 0..10
    ids = np.arange(11)
    keep = (ids % 6 != 1) & (ids % 10 != 3) & (ids % 15 != 7)
    assert len(k) == int(keep.sum()) and single[0]["dropped"] == int((~keep).sum())
    # per-shape stiffness streams (DeviceRollouts.shape_seed): the three shapes do not share a label vector
    dr = rg.DeviceRollouts.__new__(rg.DeviceRollouts)
    dr.seed = 0
    assert len({dr.shape_seed(s) for s in rg.SHAPES}) == 3
