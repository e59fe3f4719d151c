#!/usr/bin/env python
"""Build -D variants of csrc/cnf_rk.cu (here, no GPU needed) and time config 3 at 2^20 trajectories with each (GPU box).
  build:  python tools/tune_cnf.py build           -> pnode_b200/csrc/tune/libcnf_*.so
  time :  python tools/tune_cnf.py time            (under gpurun) -> gpurun_out/tune_cnf.json"""
import copy
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "pnode_b200", "csrc")
TUNE = os.path.join(CSRC, "tune")

VARIANTS = {
    "ev4": {"CNF_EVAL_UNROLL": 4},
    "ev4_mb3": {"CNF_EVAL_UNROLL": 4, "CNF_ATT_MINB": 3},
    "ev2_mb3": {"CNF_EVAL_UNROLL": 2, "CNF_ATT_MINB": 3},
    "ev6": {"CNF_EVAL_UNROLL": 6},
}


def build():
    os.makedirs(TUNE, exist_ok=True)
    procs = []
    for name, defs in VARIANTS.items():
        out = os.path.join(TUNE, "libcnf_%s.so" % name)
        obj = os.path.join(TUNE, "cnf_%s.o" % name)
        cmd = ["nvcc", "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC",
               "-c", "cnf_rk.cu", "-o", obj] + ["-D%s=%s" % kv for kv in defs.items()]
        procs.append((name, out, obj, subprocess.Popen(cmd, cwd=CSRC, stderr=subprocess.PIPE, text=True)))
    objdir = os.path.join(CSRC, "_obj")
    others = [os.path.join(objdir, f) for f in os.listdir(objdir) if f.endswith(".o") and not f.startswith("cnf_rk")]
    for name, out, obj, p in procs:
        p.wait()
        if p.returncode != 0:
            print(name, "FAILED\n" + p.stderr.read()[-2000:])
            continue
        link = ["nvcc", "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a", "-o", out, obj] + \
            others + ["-lcuda"]
        r = subprocess.run(link, capture_output=True, text=True)
        print(name, "ok" if r.returncode == 0 else "LINK FAILED\n" + r.stderr[-2000:])
        os.remove(obj)


def time_one():
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch

    import bench_configs as bc
    from pnode import petsc_adjoint
    from pnode_b200.options import Options

    name, build_cfg = bc.config_table()["3L"]
    spec = build_cfg()
    Options.clear_all()
    Options.insert_args(spec["argv"])
    dev = torch.device("cuda:0")
    funcs = [spec["to_dev"](copy.deepcopy(f), dev) for f in spec["funcs"]]
    u0, t, target = spec["u0"].to(dev), spec["t"].to(dev), spec["target"].to(dev)
    ode = petsc_adjoint.ODEPetsc()
    ode.setupTS(u0, funcs[0], step_size=spec["step"], enable_adjoint=True, **spec["kw"])
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    tf = ta = 0.0
    reps = 6
    for i in range(reps + 2):
        funcs[0].zero_grad(set_to_none=True)
        torch.cuda.synchronize()
        ev[0].record()
        pred = ode.odeint_adjoint(u0, t)
        ev[1].record()
        (pred * target).sum().backward()
        ev[2].record()
        torch.cuda.synchronize()
        if i >= 2:
            tf += ev[0].elapsed_time(ev[1])
            ta += ev[1].elapsed_time(ev[2])
    g = torch.cat([p.grad.reshape(-1) for p in funcs[0].parameters()])
    print(json.dumps({"fwd_ms": tf / reps, "adj_ms": ta / reps, "chk": float(g.double().abs().sum())}))


def time_all():
    res = {}
    for name in VARIANTS:
        lib = os.path.join(TUNE, "libcnf_%s.so" % name)
        if not os.path.exists(lib):
            continue
        env = dict(os.environ, PNODE_B200_LIB=lib)
        p = subprocess.run([sys.executable, __file__, "one"], env=env, capture_output=True, text=True)
        try:
            res[name] = json.loads(p.stdout.strip().splitlines()[-1])
        except Exception:
            res[name] = {"error": (p.stderr or p.stdout)[-500:]}
        print(name, res[name], flush=True)
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    with open(os.path.join(ROOT, "gpurun_out", "tune_cnf.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    if sys.argv[1] == "build":
        build()
    elif sys.argv[1] == "one":
        time_one()
    else:
        time_all()
