#!/usr/bin/env python
"""Build -D variants of csrc/mlp_rk.cu (here, no GPU needed) and time them (on the GPU box).
  build:  python tools/tune_spiral.py build            -> gpurun_out/.. no; writes pnode_b200/csrc/tune/*.so
  time :  python tools/tune_spiral.py time [f64|f32]   (run under gpurun) -> gpurun_out/tune.json
Variants are listed in VARIANTS below."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "pnode_b200", "csrc")
TUNE = os.path.join(CSRC, "tune")

VARIANTS = {
    "base": {},
    "f64_tanh_v0": {"PNODE_F64_TANH_V": 0},       # relative-accuracy tanh (15 FP64 instructions)
    "f32_t1c2": {"PNODE_F32_TPT": 1, "PNODE_F32_CHUNKS": 2, "PNODE_F32_ADJ_CTAS": 5},
    "f32_t1c2_ag1": {"PNODE_F32_TPT": 1, "PNODE_F32_CHUNKS": 2, "PNODE_F32_ADJ_CTAS": 5, "PNODE_F32_ADJ_GROUP": 1},
    "f32_t1c2_ag2": {"PNODE_F32_TPT": 1, "PNODE_F32_CHUNKS": 2, "PNODE_F32_ADJ_CTAS": 5, "PNODE_F32_ADJ_GROUP": 2},
    "f32_t2c2": {"PNODE_F32_CHUNKS": 2, "PNODE_F32_ADJ_CTAS": 3},
    "f32_t2c3_a3": {"PNODE_F32_ADJ_CTAS": 3},
    "f32_t2c3_ag1": {"PNODE_F32_ADJ_GROUP": 1, "PNODE_F32_ADJ_CTAS": 3},
    "f32_fwd_g2": {"PNODE_F32_GROUP": 2, "PNODE_F32_ADJ_GROUP": 4},
    "f32_fwd_t1": {"PNODE_F32_TPT": 1, "PNODE_F32_CHUNKS": 2, "PNODE_F32_ADJ_CTAS": 5, "PNODE_F32_FWD_CTAS": 12},
    "f64_ag10": {"PNODE_F64_ADJ_GROUP": 10},
    "f64_adj2": {"PNODE_F64_ADJ_CTAS": 2},
    "f64_fwd4": {"PNODE_F64_FWD_CTAS": 4},
    "f64_fwd6": {"PNODE_F64_FWD_CTAS": 6},
    "f64_g10": {"PNODE_F64_GROUP": 10, "PNODE_F64_ADJ_GROUP": 5, "PNODE_F64_FWD_CTAS": 4},
    "f64_g10b": {"PNODE_F64_GROUP": 10, "PNODE_F64_ADJ_GROUP": 5, "PNODE_F64_FWD_CTAS": 3},
    "f64_ch3": {"PNODE_F64_CHUNKS": 3, "PNODE_F64_ADJ_CTAS": 4},
}


def build():
    """Part 0 of mlp_rk.cu (the spiral shape + the C entry points) is compiled per variant and linked against the objects of
    the in-tree build (pnode_b200/csrc/_obj, `python -m pnode_b200.build` first) for everything else."""
    os.makedirs(TUNE, exist_ok=True)
    objdir = os.path.join(CSRC, "_obj")
    others = [os.path.join(objdir, f) for f in sorted(os.listdir(objdir)) if f.endswith(".o") and f != "mlp_rk.o"]
    procs = []
    for name, defs in VARIANTS.items():
        obj = os.path.join(TUNE, "mlp_rk_%s.o" % name)
        cmd = ["nvcc", "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC",
               "-DPNODE_MLP_PART=0", "-c", "mlp_rk.cu", "-o", obj] + ["-D%s=%s" % kv for kv in defs.items()]
        procs.append((name, obj, subprocess.Popen(cmd, cwd=CSRC, stderr=subprocess.PIPE, text=True)))
        if len(procs) % 4 == 0:
            for _, _, p in procs[-4:]:
                p.wait()
    for name, obj, p in procs:
        err = p.stderr.read()
        p.wait()
        if p.returncode != 0:
            print(name, "FAILED\n" + err[-2000:])
            continue
        out = os.path.join(TUNE, "lib_%s.so" % name)
        link = ["nvcc", "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a", "-o", out, obj] + others + \
            ["-lcuda"]
        r = subprocess.run(link, capture_output=True, text=True)
        print(name, "ok" if r.returncode == 0 else "LINK FAILED\n" + r.stderr[-2000:])
        os.remove(obj)


def time_one(dtype):
    """Runs in a child process with PNODE_B200_LIB set."""
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch
    from _problems import SpiralFunc
    from pnode_b200 import tableaux
    from pnode_b200.fused import FusedMlpRK, recognise_mlp

    dt = torch.float64 if dtype == "f64" else torch.float32
    n = 1 << 20
    dev = torch.device("cuda:0")
    func = SpiralFunc(dtype=dt).to(dev)
    g = torch.Generator().manual_seed(0)
    u0 = ((torch.rand(n, 1, 2, generator=g, dtype=torch.float64) * 2 - 1) * 2).to(dt).to(dev)
    spec = recognise_mlp(func, u0)
    fused = FusedMlpRK(spec, tableaux.RK["4"], dt, dev)
    times = [0.025 * i for i in range(10)]
    gout = torch.randn(10, n * 2, dtype=dt, device=dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    tf = ta = 0.0
    reps = 8
    for i in range(reps + 2):
        torch.cuda.synchronize()
        ev[0].record()
        sol, ckpt, sched = fused.forward(u0.reshape(-1), times, 0.025, True)
        ev[1].record()
        lam, mu, _ = fused.adjoint(gout, ckpt, sched, n)
        ev[2].record()
        torch.cuda.synchronize()
        if i >= 2:
            tf += ev[0].elapsed_time(ev[1])
            ta += ev[1].elapsed_time(ev[2])
    print(json.dumps({"fwd_ms": tf / reps, "adj_ms": ta / reps, "chk": float(mu.double().abs().sum()),
                      "chk2": float(sol[-1].double().abs().sum())}))


def time_all(dtypes):
    res = {}
    for name in VARIANTS:
        lib = os.path.join(TUNE, "lib_%s.so" % name)
        if not os.path.exists(lib):
            continue
        for dtype in dtypes:
            if (name.startswith("f32") and dtype != "f32") or (name.startswith("f64") and dtype != "f64"):
                continue
            env = dict(os.environ, PNODE_B200_LIB=lib)
            p = subprocess.run([sys.executable, __file__, "one", dtype], env=env, capture_output=True, text=True)
            try:
                res["%s/%s" % (name, dtype)] = json.loads(p.stdout.strip().splitlines()[-1])
            except Exception:
                res["%s/%s" % (name, dtype)] = {"error": (p.stderr or p.stdout)[-500:]}
            print(name, dtype, res["%s/%s" % (name, dtype)], flush=True)
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    with open(os.path.join(ROOT, "gpurun_out", "tune.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    if sys.argv[1] == "build":
        build()
    elif sys.argv[1] == "one":
        time_one(sys.argv[2])
    else:
        time_all(sys.argv[2:] or ["f64", "f32"])
