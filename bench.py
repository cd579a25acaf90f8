#!/usr/bin/env python
"""Benchmark of the soft-grip hot path on B200: world-steps/s of the batched squeeze-episode rollout.

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA kernels behind the C-ABI)
    python bench.py --impl reference --gpus N --steps K ...   # the CPU path (oracle port, all host cores)
    N>1:  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload = BASELINE.json configs[2] as written: `--worlds` = 65 536 worlds IN TOTAL, sharded W/N per rank (strong
scaling; `--weak` keeps `--worlds` per GPU instead), every world with its own stiffness U(300,1400) (ref:
environment/manenv.py:103-109), shell damping and object-centre offset (the two extensions configs[2] names; see
--damping-range / --offset-range), fp32 fast path, softbox model, no collective on the step path.  One "step" = one full
squeeze episode (reset + 1 + 200*7 = 1401 physics steps, ref: create_dataset.py:14-17,33-60) of the rank's shard
= one launch of the rollout kernel per GPU.  Other BASELINE configs: `--config 1` (4 096 worlds, fp64 verification
build, fixed stiffness, error against the oracle), `--model softball|softcylinder|softbox_refined --tendon-damping D`.

`value`   : device-timed (CUDA events on the launching stream, max over ranks), parameters resident in HBM.
`e2e`     : the same episode through sg_batch_rollout_host_params with pinned HOST buffers (H2D of the per-world
            parameters and D2H of the whole trajectory + status inside the timed region, wall clock, max over ranks).
`roofline`: HBM roofline of the rollout kernel on its algorithmic bytes (the kernel is latency/issue bound on
            the Gauss-Seidel sweep, so this fraction is tiny by construction; see DESIGN.md); `fp32_pipe` is the pipe view.
`cpu_baseline`: the fp64 oracle (a port, not libmujoco; -O3 -march=native) on the host cores, bounded sample, rank 0, N=1.
`variants`: (N=1) the same launch with stiffness-only randomisation, and with shell damping U(50,200) (below ~85 the
            softbox volume mode is linearly unstable, SURVEY App. E: those worlds are flagged diverged and counted).
`sensor_trace_error`: (N=1) worlds just simulated against the fp64 oracle with the same parameters.
`traj_kernels`: (N=1, outside the timed region) the HBM-bound kernels that post-process the trajectory buffer.
`--dump-outputs DIR`: the trajectories of the last timed step (a seeded sample of at most 56 MiB) as DIR/traj.npy; the
            inputs are a function of the arguments alone, so two builds run with the same arguments compare output for output.
"""
import argparse
import atexit
import ctypes as C
import functools
import importlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
if __name__ == "__main__":
    sys.dont_write_bytecode = True       # the benchmark leaves the tree as it found it (no __pycache__ of the modules it imports)

STEPS_PER_EPISODE = 1 + 200 * 7
METRIC = "world-steps/sec"


# ---------------------------------------------------------------------------------------------
# helpers shared with the tests (pure host logic)
# ---------------------------------------------------------------------------------------------
def shard_range(total, rank, world):
    """Contiguous block of worlds owned by `rank` (SURVEY section 8e)."""
    per = (total + world - 1) // world
    lo = min(total, rank * per)
    return lo, min(total, lo + per)


def _dist():
    import torch.distributed as dist
    return dist if (dist.is_available() and dist.is_initialized()) else None


def max_over_ranks(x, device):
    import torch
    d = _dist()
    t = torch.tensor([float(x)], dtype=torch.float64, device=device)
    if d is not None:
        d.all_reduce(t, op=d.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(x, device):
    import torch
    d = _dist()
    t = torch.tensor([float(x)], dtype=torch.float64, device=device)
    if d is not None:
        d.all_reduce(t, op=d.ReduceOp.SUM)
    return float(t.item())


def barrier():
    d = _dist()
    if d is not None:
        d.barrier()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.splitlines()[0].split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback"


# ---------------------------------------------------------------------------------------------
# per-world parameters of BASELINE.json configs[2] (counter-based per GLOBAL world id: invariant to the sharding)
# ---------------------------------------------------------------------------------------------
def world_params(args, ids, it, mode=None):
    """(stiffness[W], damping[W] | None, objoff[W,3] | None) of step `it` for the global world ids `ids`."""
    batched = importlib.import_module("soft-grip_b200.batched")
    mode = mode or args.randomise
    if args.fixed_stiffness is not None:
        k = np.full(len(ids), float(args.fixed_stiffness))
    else:
        k = batched.world_uniform(args.seed, ids, 300, 1400, stream=it)            # ref: manenv.py:103-109
    if mode == "stiffness":
        return k, None, None
    lo, hi = (50.0, 200.0) if mode == "all_damping_50_200" else args.damping_range
    d = batched.world_uniform(args.seed, ids, lo, hi, stream=100000 + it)
    r = args.offset_range
    off = np.stack([batched.world_uniform(args.seed, ids, -r, r, stream=200000 + 3 * it + c) for c in range(3)], axis=1)
    return k, d, np.ascontiguousarray(off)


# ---------------------------------------------------------------------------------------------
# CPU path (oracle port): used as cpu_baseline and as the --impl reference arm
# ---------------------------------------------------------------------------------------------
_W = {}


@functools.lru_cache(maxsize=None)
def native_oracle():
    """Path of the -O3 -march=native oracle, built once per run for the host this runs on.  It goes to a temporary
    directory, removed at exit, because the tree bench.py runs from may be read-only."""
    from oracle import sgoracle as so
    d = tempfile.mkdtemp(prefix="softgrip-bench-")
    atexit.register(shutil.rmtree, d, True)
    return so.build_native(d)


def _cpu_init(blob_path, tendon_damping=None, native=None):
    """Worker set-up; `native`: the library native_oracle() built in the parent (None: this process builds it)."""
    from oracle import sgoracle as so
    so.use_native(native or native_oracle())
    blob = open(blob_path, "rb").read()
    _W["m"] = so.OracleModel(blob)
    _W["w"] = so.OracleWorld(_W["m"])
    _W["blob"] = blob_path
    if tendon_damping is not None:
        _W["w"].set_tendon_damping(0, float(tendon_damping))


def _oracle_apply(w, model_info, k, d, off):
    """One world's parameters on the oracle, the way sg_batch_set_params applies them on the device: stiffness -> joints
    11..63 + tendon 0 (ref: manenv.py:12-13,103-109), damping -> every shell slider, offset -> the object's centre body."""
    w.set_stiffness(float(k))
    nfd, nv, obj_body, pos0 = model_info
    if d is not None:
        for i in range(nfd, nv):
            w.set_dof_damping(i, float(d))
    if off is not None:
        w.set_body_pos(obj_body, pos0 + np.asarray(off, dtype=np.float64))


def _model_info(blob_path):
    """(finger dofs, nv, body id of the composite's centre body, its model position) from the compiled blob."""
    mjcf = importlib.import_module("soft-grip_b200.mjcf")
    A = mjcf.load_blob(blob_path).arrays
    jt, jb = np.asarray(A["jnt_type"]), np.asarray(A["jnt_bodyid"])
    slide = np.nonzero(jt == 2)[0]                               # mjJNT_SLIDE: the composite's shell sliders
    obj_body = int(np.asarray(A["body_parentid"])[jb[slide[0]]])
    pos0 = np.asarray(A["body_pos"], dtype=np.float64).reshape(-1, 3)[obj_body].copy()
    nv = int(np.asarray(A["dof_bodyid"]).shape[0])
    return nv - len(slide), nv, obj_body, pos0


def _cpu_episodes(job):
    ks, ds, offs = job
    w = _W["w"]
    if "info" not in _W:
        _W["info"] = _model_info(_W["blob"])
    chk, n = 0.0, 0
    w.flops(reset=True)
    for i, k in enumerate(ks):
        _oracle_apply(w, _W["info"], k, None if ds is None else ds[i], None if offs is None else offs[i])
        rows, touch, st = w.episode()
        chk += float(np.abs(rows).sum())
        n += 1
    f = w.flops(reset=True)
    return chk, f


def _cpu_jobs(args, cores, per_core, it, mode=None):
    ids = np.arange(cores * per_core)
    k, d, off = world_params(args, ids, it, mode)
    return [(list(k[i::cores]), None if d is None else list(d[i::cores]), None if off is None else list(off[i::cores])) for i in range(cores)]


def cpu_throughput(args, blob_path, episodes_per_core, repeats=1, cores=None):
    """world-steps/s of the oracle with one process per host core on the bench's own workload; returns
    (value, cores, seconds, sample text, flops per world-step (PGS, all stages))."""
    from concurrent.futures import ProcessPoolExecutor
    cores = cores or len(os.sched_getaffinity(0))
    best = None
    with ProcessPoolExecutor(cores, initializer=_cpu_init, initargs=(blob_path, args.tendon_damping, native_oracle())) as ex:
        list(ex.map(_cpu_episodes, [([], None, None)] * cores))      # spin the workers up (model load excluded)
        for rep in range(repeats):
            jobs = _cpu_jobs(args, cores, episodes_per_core, 500000 + rep)
            t0 = time.perf_counter()
            res = list(ex.map(_cpu_episodes, jobs))
            dt = time.perf_counter() - t0
            val = cores * episodes_per_core * STEPS_PER_EPISODE / dt
            if best is None or val > best[0]:
                f = np.sum([r[1] for r in res], axis=0)
                best = (val, dt, (float(f[1] / max(1.0, f[0])), float(f[2] / max(1.0, f[0]))))
    sample = "%d processes x %d full squeeze episodes (%s, randomise=%s, fp64 oracle port, gcc -O3 -march=native)" % (
        cores, episodes_per_core, args.model, args.randomise)
    return best[0], cores, best[1], sample, best[2]


def sensor_trace_error(args, blob_path, rows, params):
    """The metric's second half ("sensor-trace error"): the sensor traces the bench just produced for a few worlds against
    the fp64 oracle run on the host with the same per-world parameters (the oracle as the checker, inside the cpu_baseline
    leg).  Relative to each channel's peak.  The 40 settle rows are contact-free and must agree tightly; over the squeeze
    contact make/break events amplify round-off (DESIGN.md section 4: the oracle run against itself from a 1e-7
    perturbation deviates as much), so the median row is the horizon statistic; tests/test_gpu.py asserts the same numbers."""
    try:
        _cpu_init(blob_path, args.tendon_damping)
        w = _W["w"]
        info = _model_info(blob_path)
        settle, med, worst = 0.0, [], 0.0
        ks, ds, offs = params
        for i, r in enumerate(rows):
            _oracle_apply(w, info, ks[i], None if ds is None else ds[i], None if offs is None else offs[i])
            want, _, st = w.episode()
            scale = np.abs(want).max(axis=0) + 1e-12
            err = (np.abs(np.asarray(r, dtype=np.float64) - want) / scale).max(axis=1)
            settle = max(settle, float(err[:40].max()))
            med.append(float(np.median(err)))
            worst = max(worst, float(err.max()))
        return {"worlds": len(med), "settle_rows_max_rel": settle, "row_median_rel": float(np.median(med)),
                "row_median_rel_worst_world": float(np.max(med)), "row_max_rel": worst,
                "against": "fp64 oracle port on the host (not libmujoco), same per-world parameters, relative to each channel's peak",
                "stated_tolerance": TRACE_TOLERANCE}
    except Exception as e:                                   # noqa: BLE001 -- informational key only
        return {"error": "%s: %s" % (type(e).__name__, e)}


# stated tolerances of the fast path against the fp64 oracle over the full horizon (DESIGN.md section 4; asserted by
# tests/test_gpu.py::test_fp32_trace_error_against_the_oracle on the same statistic)
TRACE_TOLERANCE = {"fp32": {"settle_rows_max_rel": 1e-4, "row_median_rel": 5e-2}, "fp64": {"settle_rows_max_rel": 1e-9, "row_median_rel": 5e-2}}


# ---------------------------------------------------------------------------------------------
def run_reference_arm(args, rank):
    """The reference's own CPU implementation of the path = the oracle port (MuJoCo is not installable here), with all the
    host threads it can use, on this arm's config; each step a bounded sample (cores x --ref-episodes-per-core episodes)."""
    if rank != 0:
        return
    blob = os.path.join(ROOT, "tests", "golden", args.model + ".sgm")
    from oracle import sgoracle as so
    so.build()
    cores = len(os.sched_getaffinity(0))
    from concurrent.futures import ProcessPoolExecutor
    times = []
    with ProcessPoolExecutor(cores, initializer=_cpu_init, initargs=(blob, args.tendon_damping, native_oracle())) as ex:
        list(ex.map(_cpu_episodes, [([], None, None)] * cores))
        for it in range(args.warmup + args.steps):
            jobs = _cpu_jobs(args, cores, args.ref_episodes_per_core, it)
            t0 = time.perf_counter()
            list(ex.map(_cpu_episodes, jobs))
            dt = time.perf_counter() - t0
            if it >= args.warmup:
                times.append(dt)
    total = sum(times)
    value = args.steps * cores * args.ref_episodes_per_core * STEPS_PER_EPISODE / total
    sample = "%d processes x %d full squeeze episodes per step (gcc -O3 -march=native)" % (cores, args.ref_episodes_per_core)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "world-steps/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak" if args.weak else "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, worlds_total=None, per_gpu=cores * args.ref_episodes_per_core,
                                      note="CPU path: fp64 oracle port of the MuJoCo step (not libmujoco), host cores only; each step is a bounded sample of the workload"),
            "cpu_baseline": {"value": value, "unit": "world-steps/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "world-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def workload_config(args, worlds_total, per_gpu, note=None):
    rand = {"stiffness": "stiffness U(300,1400) on joints 11..63 + tendon 0",
            "all": "stiffness U(300,1400) on joints 11..63 + tendon 0, shell damping U(%g,%g), object-centre offset U(+-%g) m per axis"
                   % (args.damping_range[0], args.damping_range[1], args.offset_range)}[args.randomise]
    if args.fixed_stiffness is not None:
        rand = "fixed stiffness %g" % args.fixed_stiffness + ("" if args.randomise == "stiffness" else "; " + rand.split(", ", 1)[1])
    cfg = {"workload": "BASELINE.json configs[%d]: %s model, %s, %s, full squeeze horizon (1401 physics steps, 200 sensor rows x 12 "
                       "channels per world), worlds sharded over the GPUs" % (args.config, args.model, rand,
                                                                             "fp32 fast path" if args.precision == 32 else "fp64 verification build"),
           "model": args.model, "worlds_total": worlds_total, "worlds_per_gpu_per_step": per_gpu,
           "physics_steps_per_world_per_step": STEPS_PER_EPISODE, "randomise": args.randomise,
           "sim_step": 7, "sim_start": 1, "rows": 200, "parallelism": "independent world shards, no collective on the step path",
           "l2": "256 MiB scratch buffer written between timed steps (L2 flush); kernel inputs are tiny, state lives in shared memory"}
    if getattr(args, "tendon_damping", None) is not None:
        cfg["tendon_damping"] = ("volume-tendon damper set to %g (model file: 100): the value at which this model is stable under the "
                                 "restated engine semantics, SURVEY App. E / section 8d cfg 3" % args.tendon_damping)
    if note:
        cfg["note"] = note
    return cfg


def measure_traj_kernels(torch, traj, flush, hbm_peak, reps=5):
    """Outside the timed region, N = 1 only: the HBM-bound kernels that post-process the trajectory buffer where the rollout
    left it (csrc/sg_traj.cuh: noise augmentation, channel statistics), each timed alone with CUDA events on the current
    stream after an L2 flush, four calls per timed region on a tensor several times the size of L2; achieved = algorithmic
    bytes (noise: read + write, statistics: read) / average time per call.
    Extra information next to the headline numbers: a failure here is reported in the key, never raised."""
    try:
        fn = importlib.import_module("soft-grip_b200.functions")
        out = torch.empty_like(traj)
        nbytes = traj.numel() * traj.element_size()
        ws, st_out = fn.stats_workspace(traj), torch.empty((2, traj.shape[-1]), dtype=torch.float64, device=traj.device)
        # buffers are allocated once, outside the timed region: what is timed is the launch(es) of the C-ABI call
        cases = (("sg_traj_noise_kernel<float>", lambda: fn.noised_modality(traj, seed=1, out=out), 2 * nbytes),
                 ("sg_traj_stats_partial_kernel<float> + final", lambda: fn.channel_mean_std(traj, workspace=ws, out=st_out), nbytes))
        res = {}
        for name, f, algo in cases:
            ms = []
            calls = 4          # per timed region: the 629 MB tensor is several times the 126 MB L2, so back-to-back passes stream from
                               # HBM every time, and the host-side cost of a call overlaps the previous launch
            for r in range(reps + 2):
                flush.fill_(r & 255)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(calls):
                    f()
                e1.record()
                torch.cuda.synchronize()
                if r >= 2:
                    ms.append(e0.elapsed_time(e1) / calls)
            avg = sum(ms) / len(ms)
            gbs = algo / (avg * 1e-3) / 1e9
            res[name] = {"ms": avg, "algorithmic_bytes": algo, "achieved_GBps": gbs, "peak_GBps": hbm_peak, "frac": gbs / hbm_peak}
        mean, std = fn.channel_mean_std(out)
        ref_std = (out - traj).double().std(dim=(0, 1), unbiased=False)
        res["check"] = {"noise_std_acc": float(ref_std[:6].mean()), "noise_std_gyro": float(ref_std[6:].mean()),
                        "stats_vs_torch_max_rel": float(((mean.reshape(-1) - out.double().mean(dim=(0, 1))).abs()
                                                         / (out.double().std(dim=(0, 1)) + 1e-30)).max())}
        return res
    except Exception as e:                                   # noqa: BLE001 -- informational key only
        return {"error": "%s: %s" % (type(e).__name__, e)}


DUMP_BYTES = 56 << 20


def dump_outputs(out_dir, traj, lo):
    """--dump-outputs: what the timed rollout returned in its last step, so that two builds can be compared output for output
    on identical inputs.  traj.npy: the trajectories [n, T, 12] in the batch precision of a fixed, seeded sample of this
    rank's worlds (all of them when they fit in DUMP_BYTES); traj_worlds.npy: their global world ids (float64)."""
    import torch
    W = traj.shape[0]
    n = min(W, DUMP_BYTES // (traj[0].numel() * traj.element_size()))
    idx = np.arange(W) if n == W else np.sort(np.random.default_rng(0).choice(W, n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "traj.npy"), traj[torch.as_tensor(idx, device=traj.device)].cpu().numpy())
    np.save(os.path.join(out_dir, "traj_worlds.npy"), (lo + idx).astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="softgrip", choices=["softgrip", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 4],
                    help="BASELINE.json configs index: 2 (default) = 65 536 worlds, everything randomised, fp32; 1 = 4 096 worlds, fixed "
                         "stiffness 700, fp64 verification build; 4 = stress (refined composite; give --worlds)")
    ap.add_argument("--model", default=None)
    ap.add_argument("--worlds", type=int, default=None, help="worlds in total (sharded W/N per rank); with --weak: per GPU")
    ap.add_argument("--weak", action="store_true", help="weak scaling: --worlds per GPU instead of in total")
    ap.add_argument("--precision", type=int, default=None, choices=[32, 64])
    ap.add_argument("--randomise", default=None, choices=["stiffness", "all"])
    ap.add_argument("--fixed-stiffness", type=float, default=None)
    ap.add_argument("--damping-range", type=float, nargs=2, default=[100.0, 200.0],
                    help="shell damping U(lo,hi): from the committed model value 100 to the reference's unused DEFAULT_DAMPING 200 "
                         "(ref: manenv.py:5); below ~85 the softbox volume mode is linearly unstable (SURVEY App. E)")
    ap.add_argument("--offset-range", type=float, default=0.05, help="object-centre offset U(+-r) m per axis")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--tendon-damping", type=float, default=None,
                    help="override the composite's volume-tendon damper for every world (softball / softcylinder: 50 is stable)")
    ap.add_argument("--cpu-episodes-per-core", type=int, default=16)
    ap.add_argument("--ref-episodes-per-core", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--trace-worlds", type=int, default=8)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the trajectories of the last one to DIR/*.npy (rank 0, CUDA path)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computed; the reference arm keeps no trajectories")
    if args.warmup < 3:
        args.warmup = 3                      # timing rules: W >= 3
    defaults = {2: ("softbox", 65536, 32, "all", None), 1: ("softbox", 4096, 64, "stiffness", 700.0), 4: ("softbox_refined", 16384, 32, "all", None)}[args.config]
    args.model = args.model or defaults[0]
    args.worlds = args.worlds or defaults[1]
    args.precision = args.precision or defaults[2]
    args.randomise = args.randomise or defaults[3]
    if args.fixed_stiffness is None:
        args.fixed_stiffness = defaults[4]
    if args.config == 4 and args.tendon_damping is None and args.model == "softbox_refined":
        args.tendon_damping = 20.0
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the CUDA path has no CPU fallback (use --impl reference for the CPU arm)")
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    batched = importlib.import_module("soft-grip_b200.batched")
    from importlib import import_module
    lib = import_module("soft-grip_b200._lib")

    # ---- sharding (SURVEY section 8e): contiguous blocks of global world ids, no collective on the step path ----
    if args.weak:
        W_total, lo = args.worlds * world, rank * args.worlds
        hi = lo + args.worlds
    else:
        W_total = args.worlds
        lo, hi = shard_range(W_total, rank, world)
    Wg = hi - lo
    tdtype = torch.float32 if args.precision == 32 else torch.float64
    esize = 4 if args.precision == 32 else 8
    blob = os.path.join(ROOT, "tests", "golden", args.model + ".sgm")
    env = batched.BatchedManEnv(blob, Wg, device=dev, dtype=tdtype, seed=args.seed, world_offset=lo)
    ev, val = batched.default_schedule(env.nu)
    T = ev.shape[0]
    sc = lib.SgSchedule(1, 7, T, ev.ctypes.data_as(C.POINTER(C.c_int)), val.ctypes.data_as(C.POINTER(C.c_double)))
    traj = torch.empty((Wg, T, env.nsd), dtype=tdtype, device=dev)
    ids = np.arange(lo, hi)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)
    tdamp = None if args.tendon_damping is None else np.full(Wg, args.tendon_damping)

    def push_params(it, mode=None):
        k, d, off = world_params(args, ids, it, mode)
        env.stiffness = torch.from_numpy(k).to(dev)
        env.set_params(damping=d, tendon_damping=tdamp, object_offset=off)     # resident in HBM before the timed region
        return k, d, off

    def one_step(it, timed, mode=None):
        push_params(it, mode)
        flush.fill_(it & 255)                           # L2 flush
        if timed:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
        lib.check(env.L.sg_batch_rollout(env.h, C.byref(sc), C.c_void_p(traj.data_ptr()), None, C.c_void_p(stream.cuda_stream)))
        if timed:
            e1.record(stream)
            return e0, e1
        return None

    for it in range(args.warmup):
        one_step(it, False)
    torch.cuda.synchronize(dev)
    barrier()
    launches0 = env.launch_count()
    env.status(clear=True)
    with ClockSampler(local_rank) as clk:
        evs = [one_step(args.warmup + it, True) for it in range(args.steps)]
        torch.cuda.synchronize(dev)
    barrier()
    launches = env.launch_count() - launches0
    ms_local = sum(a.elapsed_time(b) for a, b in evs)
    ms_total = max_over_ranks(ms_local, dev)
    st = env.status(clear=True)
    ndiv = sum_over_ranks(float(((st & batched.ST_DIVERGED) != 0).sum()), dev)
    nfull = sum_over_ranks(float(((st & (batched.ST_CON_FULL | batched.ST_UNSUPPORTED)) != 0).sum()), dev)
    finite = bool(torch.isfinite(traj).all().item())
    world_steps = float(W_total) * STEPS_PER_EPISODE * args.steps
    value = world_steps / (ms_total * 1e-3)
    last = args.warmup + args.steps - 1                  # `traj` still holds the last timed step
    pick = sorted(set(int(x) for x in np.linspace(0, Wg - 1, max(1, args.trace_worlds))))
    traj_pick = traj[pick].double().cpu().numpy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, traj, lo)                  # before the variants below reuse `traj`

    # ---- end to end through the C-ABI with pinned HOST buffers ----
    k_host = torch.empty(Wg, dtype=torch.float64).pin_memory()
    d_host = torch.empty(Wg, dtype=torch.float64).pin_memory() if args.randomise == "all" else None
    o_host = torch.empty((Wg, 3), dtype=torch.float64).pin_memory() if args.randomise == "all" else None
    traj_host = torch.empty((Wg, T, env.nsd), dtype=tdtype).pin_memory()
    status_host = np.zeros(Wg, dtype=np.int32)
    hp = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
    h2d = Wg * 8 * (1 + (4 if args.randomise == "all" else 0))
    d2h = Wg * (T * env.nsd * esize + 4)

    def e2e_step(it):
        k, d, off = world_params(args, ids, 1000 + it)
        k_host.copy_(torch.from_numpy(k))
        if d_host is not None:
            d_host.copy_(torch.from_numpy(d)); o_host.copy_(torch.from_numpy(off))
        lib.check(env.L.sg_batch_rollout_host_params(env.h, C.byref(sc), hp(k_host), hp(d_host), None, hp(o_host), hp(traj_host), None,
                                                     status_host.ctypes.data_as(C.c_void_p)))
    e2e_step(0)
    torch.cuda.synchronize(dev)
    barrier()
    t0 = time.perf_counter()
    for it in range(args.steps):
        e2e_step(1 + it)
    torch.cuda.synchronize(dev)
    e2e_s = max_over_ranks(time.perf_counter() - t0, dev)
    barrier()
    e2e_value = world_steps / e2e_s
    e2e_launches = args.steps

    # ---- variants (N = 1): what the randomisation costs / does ----
    variants = None
    if world == 1 and not args.no_variants and args.randomise == "all":
        variants = {}
        for name, mode in (("stiffness_only", "stiffness"), ("damping_50_200_and_offset", "all_damping_50_200")):
            one_step(2000, False, mode)
            torch.cuda.synchronize(dev)
            env.status(clear=True)
            e0, e1 = one_step(2001, True, mode)
            torch.cuda.synchronize(dev)
            stv = env.status(clear=True)
            ms = e0.elapsed_time(e1)
            variants[name] = {"value": Wg * STEPS_PER_EPISODE / (ms * 1e-3), "unit": "world-steps/s", "ms_per_step": ms, "steps": 1,
                              "worlds_diverged": int(((stv & batched.ST_DIVERGED) != 0).sum()),
                              "worlds_capacity_or_unsupported": int(((stv & (batched.ST_CON_FULL | batched.ST_UNSUPPORTED)) != 0).sum())}
        push_params(last)

    if rank != 0:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()
        return

    # ---- roofline of the rollout kernel (HBM; algorithmic bytes = parameters in + trajectory + status out) ----
    peaks, which = measured_peaks()
    bytes_per_world = 8 * (1 + (4 if args.randomise == "all" else 0)) + T * env.nsd * esize + 4
    launch_s = (ms_local * 1e-3) / args.steps
    achieved = Wg * bytes_per_world / launch_s / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            # measured per launch of `worlds_per_launch` worlds under ncu --set full; scaled to this launch's world count
            traffic = tj.get("dram_bytes_per_launch")
            if traffic is not None and tj.get("worlds_per_launch"):
                traffic = traffic * Wg / float(tj["worlds_per_launch"])
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                "traffic": traffic, "peak_source": which + " (MEASURED_PEAKS.json hbm_gbs)" if which == "measured" else "fallback 6650 GB/s",
                "kernel": "sg_step_kernel2<%s, %d> (rollout mode)" % ("float" if args.precision == 32 else "double", env.config()["lanes_per_world"]),
                "algorithmic_bytes_per_world_episode": bytes_per_world,
                "note": "latency/issue-bound Gauss-Seidel kernel: state stays in shared memory for the whole episode, so the HBM fraction is tiny by design; see fp32_pipe"}

    cpu = None
    flops = None
    trace_err = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import sgoracle as so
        so.build()
        k_l, d_l, o_l = world_params(args, ids, last)
        sel = (k_l[pick], None if d_l is None else d_l[pick], None if o_l is None else o_l[pick])
        trace_err = sensor_trace_error(args, blob, traj_pick, sel)
        v, cores, secs, sample, flops = cpu_throughput(args, blob, args.cpu_episodes_per_core)
        cpu = {"value": v, "unit": "world-steps/s", "cores": cores, "kind": "port", "sample": sample + ", %.1f s" % secs}

    traj_kernels = None
    if world == 1 and args.precision == 32:
        traj_kernels = measure_traj_kernels(torch, traj, flush, peaks["hbm_gbs"])

    line = {"metric": METRIC, "value": value, "unit": "world-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak" if args.weak else "strong", "vs_baseline": None,
            "dtype": "f32" if args.precision == 32 else "f64",
            "data": "synthetic", "config": workload_config(args, W_total, Wg),
            "e2e": {"value": e2e_value, "unit": "world-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "clocks": clk.summary(),
            "launch_geometry": env.config(), "worlds_diverged": int(ndiv), "worlds_capacity_or_unsupported": int(nfull), "trajectory_finite": finite}
    if flops:
        clock = (line["clocks"]["sm_mhz"] or 1965.0)
        peak = 148 * 128 * 2 * clock * 1e6 / 1e12 / (1 if args.precision == 32 else 64)     # fp64: 1/64 rate on B200
        line["fp32_pipe" if args.precision == 32 else "fp64_pipe"] = {
            "flops_per_world_step_all_stages": flops[1], "flops_per_world_step_pgs": flops[0],
            "count": "episode average over the cpu_baseline sample: PGS counted per executed row / block update by the oracle's op counter, "
                     "other stages by the closed-form count of SURVEY section 8d (oracle/sg_oracle.c sgo_flops_get)",
            "achieved_tflops": value / world * flops[1] / 1e12, "peak_tflops_at_sampled_clock": peak,
            "frac": value / world * flops[1] / 1e12 / peak}
    if variants is not None:
        line["variants"] = variants
    if traj_kernels is not None:
        line["traj_kernels"] = traj_kernels
    if trace_err is not None:
        line["sensor_trace_error"] = trace_err
    print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
