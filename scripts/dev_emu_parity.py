"""Dev tool: single-step parity of the kernel source (run under the SIMT emulator, no GPU) against the oracle along
an oracle trajectory.  usage: dev_emu_parity.py [model] [64|32] [nsteps] [lpw] [stride]"""
import importlib, os, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "simt"))
from oracle import sgoracle as so
import emu
batched = importlib.import_module("soft-grip_b200.batched")
mjcf = importlib.import_module("soft-grip_b200.mjcf")

name = sys.argv[1] if len(sys.argv) > 1 else "softbox"
prec = int(sys.argv[2]) if len(sys.argv) > 2 else 64
nsteps = int(sys.argv[3]) if len(sys.argv) > 3 else 400
lpw = int(sys.argv[4]) if len(sys.argv) > 4 else 8
stride = int(sys.argv[5]) if len(sys.argv) > 5 else 1
blob = os.path.join(ROOT, "tests", "golden", name + ".sgm")
model = mjcf.load_blob(blob)
om = so.OracleModel(open(blob, "rb").read())
ow = so.OracleWorld(om)
ow.set_geom_mask(batched.geom_name_mask(model.names["geom"], "OBJ", ("g12", "g2")))
k = 700.0
ow.set_stiffness(k)
W = 32 // lpw + 1
env = emu.EmuBatch(blob, W, prec=prec, lpw=lpw)
env.set_params(stiffness=np.full(W, k))
env.set_debug_world(1)
print("info nv", env.info.nv, "levels", env.info.nlevels, "maxcon", env.info.maxcon, "smem32", env.info.smem_bytes32, "W", W, "lpw", lpw)
ow.reset()
worst = {}
def rel(a, b):
    return np.abs(a - b).max() / max(1e-12, np.abs(b).max())
t0 = time.time()
ctrl = [0.0, 0.0]
for t in range(nsteps):
    if t == 281: ow.set_ctrl([-0.2, -0.2]); ctrl = [-0.2, -0.2]
    if t == 841: ow.set_ctrl([0.2, 0.2]); ctrl = [0.2, 0.2]
    q, v, a, w = ow.get_state()
    st = ow.step()
    if t % stride:
        continue
    env.set_state(q, v, a, w)
    env.set_ctrl(ctrl)
    sens, touch = env.step(1)
    q2, v2, a2, w2 = ow.get_state()
    gq, gv, ga, gw = env.get_state()
    e = dict(q=rel(gq[1], q2), v=rel(gv[1], v2), act=np.abs(ga[1] - a2).max(), qacc=rel(gw[1], w2), sens=rel(sens[1], ow.sensordata()))
    same = all(np.array_equal(gq[1], gq[i]) and np.array_equal(gw[1], gw[i]) for i in range(W))
    ncon_o, nefc_o, it_o = ow.get_int("ncon"), ow.get_int("nefc"), ow.get_int("solver_iter")
    ncon_g, nefc_g, it_g = int(env.debug("ncon")[0]), int(env.debug("nefc")[0]), int(env.debug("solver_iter")[0])
    bad = (ncon_o != ncon_g) or (nefc_o != nefc_g) or (it_o != it_g and prec == 64) or max(e.values()) > (1e-8 if prec == 64 else 2e-2) or not same \
        or int(touch[1]) != ow.touch_mask()
    for kk, vv in e.items(): worst[kk] = max(worst.get(kk, 0), vv)
    if bad or t % (50 * stride) == 0:
        print(t, "ncon", ncon_o, ncon_g, "nefc", nefc_o, nefc_g, "iter", it_o, it_g, {kk: "%.2e" % vv for kk, vv in e.items()}, "touch", ow.touch_mask(), int(touch[1]),
              "st", st, env.status()[1], "same", same, "maxlev/tmax", int(env.debug("maxlev")[0]), "%.1fs" % (time.time() - t0), flush=True)
    if bad and "-k" not in sys.argv:
        fo, fg = ow.get("efc_force"), env.debug("efc_force")
        ao, ag = ow.get("efc_aref"), env.debug("efc_aref")
        Ro, Rg = ow.get("efc_R"), env.debug("efc_R")
        n = min(len(fo), len(fg))
        print(" efc_aref err", np.abs(ao[:n] - ag[:n]).max(), np.argmax(np.abs(ao[:n] - ag[:n])), " R err", np.abs(Ro[:n] - Rg[:n]).max(), np.argmax(np.abs(Ro[:n] - Rg[:n])),
              " force err", np.abs(fo[:n] - fg[:n]).max(), np.argmax(np.abs(fo[:n] - fg[:n])), "max |f|", np.abs(fo).max())
        do, dg = ow.get("con_dist"), env.debug("con_dist")
        print(" con_dist", do[:8], dg[:8])
        print(" qacc o", w2[:10], "\n qacc g", gw[1][:10])
        print(" qacc err by dof (top)", np.argsort(-np.abs(gw[1] - w2))[:8], np.sort(-np.abs(gw[1] - w2))[:8])
        break
print("worst", {kk: "%.3e" % vv for kk, vv in worst.items()}, "time %.1fs" % (time.time() - t0))
