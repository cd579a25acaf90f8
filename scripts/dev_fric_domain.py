"""Dev tool: the domain of friction_fast's arguments that the fp32 step kernel produces, measured under the SIMT emulator
(no GPU).  Builds the kernel source with -DSG_FRIC_DOMAIN into a temporary directory, steps the twelve golden softbox
snapshots and emulated softbox squeeze episodes at five stiffnesses in fp32, and prints the ranges of f0, |bc| kb / f0, the
condition of the normalised tangential block (all calls, and the calls that end inside the cone) and the warm start over
the root it settles on.  tests/test_primitives.py asserts its friction bounds on this domain (profiles/fric_domain.json).

usage: dev_fric_domain.py [out.json] [n_iter]"""
import importlib
import json
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIMT = os.path.join(ROOT, "tests", "simt")
CSRC = os.path.join(ROOT, "soft-grip_b200", "csrc")


def build(out_dir):
    flags = subprocess.check_output(["make", "-s", "-C", SIMT, "--eval", "print-%: ; @echo $($*)", "print-CXXFLAGS"], text=True).split()
    flags += ["-DSG_FRIC_DOMAIN", "-DSG_SMALL_BUILD=1"]
    objs = []
    for name, extra in (("api", []), ("inst_float_8", ["-DSG_INST_T=float", "-DSG_INST_LPW=8"]), ("inst_double_8", ["-DSG_INST_T=double", "-DSG_INST_LPW=8"])):
        src = os.path.join(CSRC, "sg_api.cu" if name == "api" else "sg_inst.cu")
        o = os.path.join(out_dir, name + ".o")
        subprocess.check_call(["g++"] + flags + extra + ["-x", "c++", "-c", "-o", o, src], cwd=SIMT)
        objs.append(o)
    so = os.path.join(out_dir, "libsoftgrip_simt_domain.so")
    subprocess.check_call(["g++", "-shared", "-o", so] + objs)
    return so


def child(so, n_iter):
    import ctypes as C
    sys.path.insert(0, ROOT)
    sys.path.insert(0, SIMT)
    import emu
    batched = importlib.import_module("soft-grip_b200.batched")
    L = C.CDLL(so)
    for name, (res, args) in importlib.import_module("soft-grip_b200._lib").SIGNATURES.items():
        getattr(L, name).restype = res
        getattr(L, name).argtypes = args
    emu._LIB = L
    golden = os.path.join(ROOT, "tests", "golden")
    st = np.load(os.path.join(golden, "softbox_states.npz"))
    env = emu.EmuBatch(os.path.join(golden, "softbox.sgm"), 1, prec=32, lpw=8)
    env.set_params(stiffness=[700.0])
    for i in range(len(st["step"])):
        env.set_state(st["q"][i], st["v"][i], st["act"][i], st["warm"][i])
        env.set_ctrl([st["ctrl"][i]] * 2)
        env.step(1)
    env.close()
    sched = batched.default_schedule(2, n_settle=2, n_iter=n_iter, open_close_div=4)
    ks = np.array([200.0, 500.0, 700.0, 1000.0, 1500.0])
    env = emu.EmuBatch(os.path.join(golden, "softbox.sgm"), len(ks), prec=32, lpw=8)
    env.set_params(stiffness=ks)
    _, _, status = env.rollout(sched)
    assert (status == 0).all(), status     # a diverged world would put its reset state into the domain
    env.close()


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "--child":
        child(sys.argv[2], int(sys.argv[3]))
        return
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(tempfile.gettempdir(), "fric_domain.json")
    n_iter = int(sys.argv[2]) if len(sys.argv) > 2 else 16
    tmp = tempfile.mkdtemp(prefix="sg_fric_domain_")
    try:
        so = build(tmp)
        if os.path.exists(out):
            os.remove(out)
        env = dict(os.environ, SG_FRIC_DOMAIN_OUT=out, PYTHONDONTWRITEBYTECODE="1")
        subprocess.check_call([sys.executable, os.path.abspath(__file__), "--child", so, str(n_iter)], env=env)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    d = json.loads(open(out).read().splitlines()[-1])
    print("calls %d, active %d, singular block %d" % (d["calls"], d["active"], d["singular"]))
    for q in ("f0", "bc_kb_over_f0", "cond", "cond_inactive", "warm_over_root"):
        h = d[q]["hist_log10_quarter"]
        print("%-15s n %9d  min %.3g  max %.3g  log10 bins %s .. %s" % (q, d[q]["n"], d[q]["min"], d[q]["max"], min(h, key=float, default="-"), max(h, key=float, default="-")))


if __name__ == "__main__":
    main()
