"""Dev tool: SM cycles per phase of the step kernel (SOFTGRIP_PROF=1), split into the contact-free settle part and the
whole episode.  usage: dev_phase.py [model] [W] [configs...]   config = l<lpw>:n<warps>"""
import importlib, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ["SOFTGRIP_PROF"] = "1"
import torch
batched = importlib.import_module("soft-grip_b200.batched")
name = sys.argv[1] if len(sys.argv) > 1 else "softbox"
W = int(sys.argv[2]) if len(sys.argv) > 2 else 18944
cfgs = sys.argv[3:] or ["l8:n16"]
dm = batched.DeviceModel(os.path.join(ROOT, "tests", "golden", name + ".sgm"))
for cfg in cfgs:
    parts = {x[0]: int(x[1:]) for x in cfg.split(":")}
    os.environ["SOFTGRIP_LPW"] = str(parts.get("l", 8))
    if "n" in parts: os.environ["SOFTGRIP_NW"] = str(parts["n"])
    else: os.environ.pop("SOFTGRIP_NW", None)
    env = batched.BatchedManEnv(dm, W, dtype=torch.float32, seed=0)
    for label, sched in (("settle (40 rows, no contact)", batched.default_schedule(2, n_settle=40, n_iter=0)), ("full episode (200 rows)", batched.default_schedule(2))):
        env.rollout(schedule=sched); env.phase_cycles()          # warm-up, clears the counters
        torch.cuda.synchronize(); e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); traj, k, st = env.rollout(schedule=sched); e1.record(); torch.cuda.synchronize()
        ph = env.phase_cycles(); tot = float(sum(ph.values())) or 1.0
        nst = 1 + 7 * len(sched[0])
        print("%s %s: %.3f s, %.3e world-steps/s (clocks on), geometry %s" % (cfg, label, e0.elapsed_time(e1) / 1e3, W * nst / (e0.elapsed_time(e1) / 1e3), env.config()))
        print("   " + "  ".join("%s %.1f%%" % (k_, 100.0 * v / tot) for k_, v in ph.items()), " | cycles per warp-step %.0f" % (tot / (W / (32 // parts.get("l", 8)) * nst)), flush=True)
    del env
