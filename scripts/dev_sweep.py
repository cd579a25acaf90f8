"""Dev tool: throughput of the rollout kernel over lanes-per-world / warps per CTA / the development switches.
usage: dev_sweep.py [model] [W] [rows] [configs...]   config = l<lpw>:n<warps per CTA>[:<letter><value>...], letters below"""
import importlib, os, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
batched = importlib.import_module("soft-grip_b200.batched")
name = sys.argv[1] if len(sys.argv) > 1 else "softbox"
W = int(sys.argv[2]) if len(sys.argv) > 2 else 8192
rows = int(sys.argv[3]) if len(sys.argv) > 3 else 60
cfgs = sys.argv[4:] or ["l8", "l4", "l16", "l32"]
blob = os.path.join(ROOT, "tests", "golden", name + ".sgm")
ev, val = batched.default_schedule(2) if rows == 200 else batched.default_schedule(2, n_settle=10, n_iter=rows - 10, open_close_div=(rows - 10) // 2)
ref = None
for cfg in cfgs:
    parts = {x[0]: int(x[1:]) for x in cfg.split(":")}
    os.environ["SOFTGRIP_LPW"] = str(parts.get("l", 8))
    # b0: plain list schedule of the equality sweep instead of the bank-conflict-aware one
    if parts.get("b", 1) == 0: os.environ["SOFTGRIP_NO_BANK_SCHEDULE"] = "1"
    else: os.environ.pop("SOFTGRIP_NO_BANK_SCHEDULE", None)
    # s0: no CTA barrier at the start of every physics step
    os.environ["SOFTGRIP_STEP_BARRIER"] = str(parts.get("s", 1))
    # m<n>: contact capacity per world
    if "m" in parts: os.environ["SOFTGRIP_MAXCON"] = str(parts["m"])
    else: os.environ.pop("SOFTGRIP_MAXCON", None)
    # t0 / t1: equality rows in shared memory / forced into tensor memory (default: the library decides)
    if "t" in parts: os.environ["SOFTGRIP_TMEM"] = str(parts["t"])
    else: os.environ.pop("SOFTGRIP_TMEM", None)
    # r0: contact records read from the scratch instead of the shared-memory ring
    if "r" in parts: os.environ["SOFTGRIP_RING"] = str(parts["r"])
    else: os.environ.pop("SOFTGRIP_RING", None)
    # d0: fixed shares of the world batches per persistent CTA instead of the dynamic hand-out
    if "d" in parts: os.environ["SOFTGRIP_DYNAMIC"] = str(parts["d"])
    else: os.environ.pop("SOFTGRIP_DYNAMIC", None)
    if "n" in parts: os.environ["SOFTGRIP_NW"] = str(parts["n"])
    else: os.environ.pop("SOFTGRIP_NW", None)
    dm = batched.DeviceModel(blob)
    for dt in (torch.float32,):
        try:
            env = batched.BatchedManEnv(dm, W, dtype=dt, seed=0)
        except Exception as e:
            print(cfg, "create failed:", e); continue
        best = 1e9
        for rep in range(3):
            torch.cuda.synchronize(); e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            # u1: every world gets the same stiffness (how much do unequal worlds in a warp / CTA cost?)
            traj, kk, st = env.rollout(schedule=(ev, val), stiffness=([700.0] * W if parts.get("u", 0) else None))
            e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1) / 1e3)
        t = traj.double().cpu().numpy()
        if ref is None: ref = t
        dev = np.median(np.abs(t - ref)) / np.abs(ref).max()
        print("%-12s W %d rows %d  %.3f s  %.3e world-steps/s  status!=0: %d  finite %s  median dev vs first %.2e" %
              (cfg, W, rows, best, W * (1 + 7 * rows) / best, int((st != 0).sum()), bool(np.isfinite(t).all()), dev), flush=True)
        del env
