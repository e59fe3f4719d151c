#!/usr/bin/env python
"""Exact-trace FFJORD solves (divergence_bf): the module path (D autograd calls per evaluation, a second backward through
them per adjoint stage) against the tensor-core evaluator (csrc/cnf_net.cu with D tangent chains), eager and replayed
from a CUDA graph.  One forward + adjoint pass = odeint_adjoint over [0, 1] with RK4, h = 0.25 (16 evaluations, 16 adjoint
stages) + backward.

    python tools/time_cnf_exact.py [--out FILE.jsonl] [--reps N] [--kernels]

Before timing, each shape checks the evaluator's outputs (trajectory, lambda, each parameter gradient) and the graph
replay's against eager execution bit for bit.  fp64: the evaluator's outputs are within 1e-10 of the module path's.  fp32:
both fp32 paths are compared with the module path run in fp64 on the same inputs; every output of the evaluator must be
within 1e-4 of it (the fp32 bar of the parity tests), and both paths' errors are recorded.  Prints the card's name, power
limit and SM clock, then one JSON line per shape with the median milliseconds per pass of each variant.  With --kernels,
one more eager evaluator pass per shape runs under torch.profiler (after the timed passes, so it does not slow them) and
the line gets the device time per kernel name of that pass."""
import argparse
import copy
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402
from _cnf_exact import exact_cnf  # noqa: E402
from _workloads import cnf_to  # noqa: E402

from pnode import petsc_adjoint  # noqa: E402
from pnode_b200.options import Options  # noqa: E402

SHAPES = [(2, (64, 64, 64), 1000, torch.float32), (2, (64, 64, 64), 1000, torch.float64),
          (43, (860, 860), 1000, torch.float32)]
FIXED = ["-ts_adapt_type", "none"]


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        line = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i",
                               str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60).stdout
        return dict(zip(q.split(","), (x.strip() for x in line.strip().split(","))))
    except (OSError, subprocess.SubprocessError):
        return {"name": torch.cuda.get_device_name()}


def inputs(B, D, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(B, D, generator=g, dtype=torch.float64)
    u0 = torch.cat((z.view(-1), torch.zeros(B, dtype=torch.float64))).to(dtype).cuda()
    gout = torch.randn(2, B * (D + 1), generator=g, dtype=torch.float64).to(dtype).cuda()
    return u0, gout


class Runner:
    def __init__(self, base, u0, gout, argv):
        Options.clear_all()
        Options.insert_args(FIXED + argv)
        self.func = cnf_to(copy.deepcopy(base), "cuda")
        self.u0, self.gout = u0, gout
        self.t = torch.tensor([0.0, 1.0], dtype=torch.float64).cuda()
        self.ode = petsc_adjoint.ODEPetsc()
        self.ode.setupTS(u0, self.func, step_size=0.25, method="rk4", enable_adjoint=True)

    def one_pass(self):
        for p in self.func.parameters():
            p.grad = None
        y0 = self.u0.clone().requires_grad_(True)
        out = self.ode.odeint_adjoint(y0, self.t)
        (out * self.gout).sum().backward()
        return out.detach(), y0.grad, [p.grad for p in self.func.parameters()]


def rel(a, b):
    return float((a.double() - b.double()).norm() / max(float(b.double().norm()), 1e-300))


def rel_each(p, q):
    """Relative errors of (trajectory, lambda, parameter gradient 0, 1, ...)."""
    return [rel(p[0], q[0]), rel(p[1], q[1])] + [rel(a, b) for a, b in zip(p[2], q[2])]


def to_f64(base):
    f = copy.deepcopy(base).to(torch.float64)
    f.base_func._e = f.base_func._e.to(torch.float64)
    f.y0 = tuple(x.to(torch.float64) for x in f.y0)
    return f


def bit_equal(p, q):
    return torch.equal(p[0], q[0]) and torch.equal(p[1], q[1]) and all(torch.equal(a, b) for a, b in zip(p[2], q[2]))


def median_ms(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ms = []
    for _ in range(reps):
        ev[0].record()
        fn()
        ev[1].record()
        torch.cuda.synchronize()
        ms.append(ev[0].elapsed_time(ev[1]))
    return statistics.median(ms), ms


def kernel_breakdown(fn):
    """Device time (ms) per kernel name of one call of fn, largest first, and the sum over all kernels."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    per = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            name = ev.name.split("(")[0].split("<")[0]
            per[name] = per.get(name, 0.0) + ev.device_time_total / 1e3
    total = sum(per.values())
    return {"total_kernel_ms": total,
            "ms_per_kernel": dict(sorted(((k, round(v, 4)) for k, v in per.items()), key=lambda kv: -kv[1])[:15])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--module-reps", type=int, default=3)
    ap.add_argument("--kernels", action="store_true")
    args = ap.parse_args()
    info = card()
    print(json.dumps({"card": info, "torch": torch.__version__}), flush=True)
    lines, failed = [], False
    for D, hidden, B, dtype in SHAPES:
        base = exact_cnf(B, D, hidden, dtype=dtype, seed=1)
        u0, gout = inputs(B, D, dtype, seed=2)
        module = Runner(base, u0, gout, ["-pnode_fused", "0"])
        ref = module.one_pass()
        evaluator = Runner(base, u0, gout, [])
        eager = evaluator.one_pass()
        assert evaluator.ode.path == "generic+cnf-net-rhs" and evaluator.ode._cb_ex.spec.trace == "exact"
        assert module.ode.path == "generic"
        if dtype == torch.float64:
            err_eval = rel_each(eager, ref)
            err_module = [0.0] * len(err_eval)
            values_ok = max(err_eval) < 1e-10
        else:
            ref64 = Runner(to_f64(base), u0.double(), gout.double(), ["-pnode_fused", "0"]).one_pass()
            err_eval, err_module = rel_each(eager, ref64), rel_each(ref, ref64)
            values_ok = max(err_eval) < 1e-4

        # CUDA graph of the whole pass: warm up on a side stream, capture, replay on new data, compare with eager
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(2):
                evaluator.one_pass()
        torch.cuda.current_stream().wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            captured = evaluator.one_pass()
        fresh = inputs(B, D, dtype, seed=3)[0]
        evaluator.u0.copy_(fresh)
        graph.replay()
        torch.cuda.synchronize()
        replayed = (captured[0].clone(), captured[1].clone(), [x.clone() for x in captured[2]])
        want = evaluator.one_pass()
        torch.cuda.synchronize()
        graph_ok = bit_equal(replayed, want)
        ok = values_ok and graph_ok
        failed = failed or not ok

        t_graph, _ = median_ms(graph.replay, 3, args.reps)
        t_eager, _ = median_ms(evaluator.one_pass, 3, args.reps)
        t_module, ms_module = median_ms(module.one_pass, 1, args.module_reps)
        line = {"D": D, "hidden": list(hidden), "B": B, "dtype": str(dtype).replace("torch.", ""), "scheme": "rk4 h=0.25",
                "evaluations": 16, "adjoint_stages": 16,
                "reference": "module path, fp64" if dtype == torch.float32 else "module path",
                "rel_err_evaluator": err_eval, "rel_err_module": err_module, "graph_bit_equal": graph_ok,
                "check_ok": ok, "ms_module": t_module, "ms_module_all": ms_module, "ms_eager": t_eager,
                "ms_graph": t_graph, "speedup_eager": t_module / t_eager, "speedup_graph": t_module / t_graph,
                "passes": {"module": args.module_reps, "eager": args.reps, "graph": args.reps}, "card": info}
        if args.kernels:
            line["evaluator_kernels"] = kernel_breakdown(evaluator.one_pass)
        print(json.dumps(line), flush=True)
        lines.append(line)
        del graph, captured, evaluator, module
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")
    if failed:
        sys.exit("an output check failed")


if __name__ == "__main__":
    main()
