#!/usr/bin/env python
"""Secondary measurement harness: every BASELINE.json config (1-5) through the drop-in on ONE B200, next to the oracle on the
host cores.  bench.py stays the contract (config 2); this script produces the per-config table of DESIGN.md section 6 /
profiles/r1_configs.jsonl.   python bench_configs.py [--configs 1,3,4,5] [--iters 10] [--cpu]

Per config one JSON line: trajectory-steps/s = batch * accepted steps / time(odeint_adjoint + backward), CUDA events, median of
`iters` after 3 warm-ups; which engine ran (fused / generic); algorithmic flops per trajectory-step from SURVEY.md section 8d
and the fraction of the measured peak of the pipe that bounds it.
"""
import argparse
import copy
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402


SEED_OFFSET = 0  # bench.py --gpus N: rank r draws its own shard of synthetic inputs (models stay identical)


def _time_gpu(step, iters, world=1):
    """Median over `iters` passes of the CUDA-event time of one pass; at world > 1 every pass is bracketed by a barrier and
    its time is the max over ranks."""
    import torch.distributed as dist

    for _ in range(3):
        step()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0.record()
        step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            tm = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            ms = float(tm.item())
        ts.append(ms)
    ts.sort()
    return ts[len(ts) // 2]


def _time_graph_replay(step, iters):
    """The same pass captured once in a CUDA graph (torch.cuda.graph around the caller's step) and replayed: what is left
    when the host side of the fixed-step paths (Python, ctypes, launch gaps) is taken out."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step()
    return _time_gpu(g.replay, iters)


def _time_cpu(step, reps=2):
    step()
    t0 = time.perf_counter()
    for _ in range(reps):
        step()
    return 1e3 * (time.perf_counter() - t0) / reps


def _make_step(ode_factory, funcs, u0, t, target, setup_kw, step_size, dev, each_call_setup=False, comm=None):
    fs = funcs
    kw = dict(setup_kw)
    if len(fs) == 2:
        kw["func2"] = fs[1]
    ode = ode_factory()
    if comm is not None:
        ode.comm = comm
    ode.setupTS(u0, fs[0], step_size=step_size, enable_adjoint=True, **kw)

    def step():
        for f in fs:
            f.zero_grad(set_to_none=True)
        if each_call_setup:  # FFJORD / CIFAR drivers call setupTS every forward (cnf.py:73, train-Cifar10.py:124)
            ode.setupTS(u0, fs[0], step_size=step_size, enable_adjoint=True, **kw)
        pred = ode.odeint_adjoint(u0, t)
        loss = torch.mean(torch.abs(pred - target))
        loss.backward()
        return ode

    return step, ode


def run_config(name, build, args, peaks, world=1, comm=None):
    """One config through the drop-in.  world > 1 (under torchrun, every rank calls this): the batch of `spec` is the PER-GPU
    batch (weak scaling), `comm` the run's BatchComm; the reported rate is the whole job's."""
    from pnode import petsc_adjoint
    from pnode_b200.options import Options

    spec = build()
    out = {"config": name, "dtype": spec["dtype"], "workload": spec["desc"], "n_gpus": world}
    Options.clear_all()
    Options.insert_args(spec["argv"])
    dev = torch.device("cuda", torch.cuda.current_device())
    to_dev = spec.get("to_dev", lambda f, d: f.to(d))
    funcs = [to_dev(copy.deepcopy(f), dev) for f in spec["funcs"]]
    u0, t, target = spec["u0"].to(dev), spec["t"].to(dev), spec["target"].to(dev)
    step, ode = _make_step(lambda: petsc_adjoint.ODEPetsc(), funcs, u0, t, target, spec["kw"], spec["step"], dev,
                           spec.get("each_call_setup", False), comm=comm)
    if comm is not None and world > 1 and spec.get("peer_reduce"):
        comm.enable_peer_reduce()
    ms = _time_gpu(step, args.iters, world)
    loop = ode._loop
    accepted = loop.steps
    attempts = len(loop.attempts)
    units = spec["batch"] * accepted * world
    cb = getattr(ode, "_cb_im", None)
    if getattr(cb, "native", None) is not None:
        out["rhs_evaluator"] = ("csrc/conv_mma.cu (tcgen05 implicit GEMM, 3xTF32)" if getattr(cb, "mma", False) else
                                "csrc/conv_block.cu") if cb.native else "library convolutions + csrc/bn_relu.cu"
    out.update({"path": ode.path, "ms_per_pass": ms, "accepted_steps": accepted, "attempts": attempts,
                "traj_steps_per_s": units / (ms * 1e-3)})
    flops = (spec["flops_per_unit"] * units + spec.get("flops_per_rejected", 0) * spec["batch"] * (attempts - accepted) * world) / world
    tfl = flops / (ms * 1e-3) / 1e12  # per GPU
    out["algorithmic_tflops"] = tfl
    hbm = spec["bytes_per_unit"] * units / world / (ms * 1e-3) / 1e9
    out["roofline"] = {"pipe": spec["pipe"], "peak_tflops": peaks[spec["pipe"]], "frac": tfl / peaks[spec["pipe"]],
                       "hbm_gbs": hbm, "hbm_peak_gbs": peaks["hbm_gbs"], "hbm_frac": hbm / peaks["hbm_gbs"]}
    if spec.get("tensor_ops_per_unit") and "dense-mlp" in str(ode.path):
        # tensor-pipe roofline of the sliced products: operations the tensor cores EXECUTE (21 int8 slice pairs per fp64 product,
        # 3 TF32 products per fp32 product) against the dense peak of that input type -- the measured bf16 peak of this pool
        # scaled by the nominal ratio of the type (int8 2x, tf32 0.5x; MEASURED_PEAKS.json has no int8 / tf32 entry)
        tops = spec["tensor_ops_per_unit"] * units / world / (ms * 1e-3) / 1e12
        ratio = 2.0 if spec["dtype"] == "f64" else 0.5
        out["roofline"]["tensor"] = {"pipe": "int8 tcgen05 (Ozaki digits, 21 slice pairs)" if spec["dtype"] == "f64" else
                                     "tf32 tcgen05 (3xTF32)", "executed_tops": tops,
                                     "peak_tops": ratio * peaks["bf16_tensor"], "frac": tops / (ratio * peaks["bf16_tensor"]),
                                     "peak_note": "%.1fx the measured bf16 peak (nominal type ratio)" % ratio}
    if world == 1 and ode.path != "generic" and not getattr(args, "no_graph", False):
        # fixed-step solves launch without reading the device, and the adaptive FFJORD solve decides on the device (recorded
        # as a fixed budget of attempts): the whole pass replays from a CUDA graph
        try:
            out["cuda_graph_replay_ms_per_pass"] = _time_graph_replay(step, args.iters)
        except Exception as exc:  # reported, never fatal for the bench line
            out["cuda_graph_replay_ms_per_pass"] = None
            out["cuda_graph_error"] = str(exc)[:200]
            torch.cuda.synchronize()
    if spec.get("also_generic") and ode.path != "generic" and world == 1 and not getattr(args, "no_generic", False):
        Options.insert_args(["-pnode_fused", "0"])
        funcs_g = [to_dev(copy.deepcopy(f), dev) for f in spec["funcs"]]
        step_g, ode_g = _make_step(lambda: petsc_adjoint.ODEPetsc(), funcs_g, u0, t, target, spec["kw"], spec["step"], dev,
                                   spec.get("each_call_setup", False))
        ms_g = _time_gpu(step_g, max(3, args.iters // 2))
        out["generic_path_ms_per_pass"] = ms_g
        out["fused_speedup_vs_generic_path"] = ms_g / ms
        Options.clear_all()
        Options.insert_args(spec["argv"])
    if args.cpu and world == 1 and spec.get("cpu_sample") is not None:
        from oracle import OracleODEPetsc

        torch.set_num_threads(os.cpu_count() or 1)
        cs = spec["cpu_sample"]()
        funcs_c = [copy.deepcopy(f) for f in cs["funcs"]]
        step_c, ode_c = _make_step(lambda: OracleODEPetsc(spec["argv"]), funcs_c, cs["u0"], cs["t"], cs["target"], cs["kw"],
                                   spec["step"], "cpu", spec.get("each_call_setup", False))
        ms_c = _time_cpu(step_c)
        acc_c = len([a for a in ode_c.ts.log if a[2]])
        out["cpu_baseline"] = {"traj_steps_per_s": cs["batch"] * acc_c / (ms_c * 1e-3), "cores": os.cpu_count(),
                               "kind": "port", "sample": cs["desc"], "ms_per_pass": ms_c}
        out["speedup_vs_cpu_port"] = out["traj_steps_per_s"] / out["cpu_baseline"]["traj_steps_per_s"]
    return out


# ----------------------------------------------------------------------------------------------------------------------


def cfg1():
    from _problems import SpiralFunc, spiral_inputs

    u0, t, target = spiral_inputs(20)
    return dict(desc="cfg1 ode_demo_petsc spiral: batch 20, batch_time 10, RK4 h=0.025, fp64", dtype="f64",
                argv=["-ts_adapt_type", "none", "-ts_trajectory_type", "memory"], funcs=[SpiralFunc()], u0=u0, t=t,
                target=target, kw=dict(method="rk4"), step=0.025, batch=20, flops_per_unit=6400, bytes_per_unit=160,
                pipe="fp64_fma", also_generic=True,
                cpu_sample=lambda: dict(funcs=[SpiralFunc()], u0=u0, t=t, target=target, kw=dict(method="rk4"), batch=20,
                                        desc="full size"))


def cfg2(dtype="f32", ntraj=1 << 20, lean=False):
    """lean: -ts_trajectory_solution_only 1 -- u_n per step in HBM (2 scalars per trajectory-step instead of 8), the stages
    recomputed inside the adjoint kernel (SURVEY.md 8f.1); the CPU baseline of the plain entry applies."""
    def build():
        from _problems import SpiralFunc

        td = torch.float32 if dtype == "f32" else torch.float64
        T, H = 10, 0.025
        g = torch.Generator().manual_seed(SEED_OFFSET)
        u0 = ((torch.rand(ntraj, 1, 2, generator=g, dtype=torch.float64) * 2 - 1) * 2).to(td)
        t = torch.arange(T, dtype=torch.float64) * H
        target = torch.randn(T, ntraj, 1, 2, generator=g, dtype=torch.float64).to(td)
        bs = 1 << 16
        w = 4 if dtype == "f32" else 8
        return dict(desc="cfg2 spiral MLP 2-50-2 on y**3, 2^%d trajectories, RK4 9 steps h=0.025, %s%s" %
                    (ntraj.bit_length() - 1, dtype, ", -ts_trajectory_solution_only 1 (u_n checkpoints, stages recomputed in "
                     "the adjoint kernel)" if lean else ""),
                    dtype=dtype, argv=["-ts_adapt_type", "none", "-ts_trajectory_type", "memory"] +
                    (["-ts_trajectory_solution_only", "1"] if lean else []), funcs=[SpiralFunc(dtype=td)],
                    u0=u0, t=t, target=target, kw=dict(method="rk4"), step=H, batch=ntraj, flops_per_unit=6400,
                    bytes_per_unit=(8 if lean else 20) * w, pipe="fp32_fma" if dtype == "f32" else "fp64_fma", peer_reduce=True,
                    cpu_sample=None if lean else lambda: dict(funcs=[SpiralFunc(dtype=td)], u0=u0[:bs].clone(), t=t, target=target[:, :bs].clone(),
                                            kw=dict(method="rk4"), batch=bs, desc="%d of %d trajectories" % (bs, ntraj)))

    return build


def _cnf(B, dtype, D=6, hidden=(60,), fixed_rk4=None):
    """FFJORD tabular CNF.  Default: the POWER shape of BASELINE config 3 (fused kernels, dopri5 adaptive).  Other shapes --
    e.g. the reference's own usage line, train_tabular.py:5: miniboone, D=43, two hidden layers of 860, RK4 h=0.25 -- run
    the generic stage loop with the tensor-core evaluator of csrc/cnf_net.cu; the same call also times the module path
    (-pnode_fused 0) for comparison."""
    from _workloads import CNFFunc, cnf_to

    def build():
        td = torch.float32 if dtype == "f32" else torch.float64
        g = torch.Generator().manual_seed(2 + SEED_OFFSET)
        mk = lambda b: dict(
            func=CNFFunc(b, D, hidden, dtype=td),
            u0=torch.cat((torch.randn(b, D, generator=g, dtype=torch.float64).view(-1),
                          torch.zeros(b, dtype=torch.float64))).to(td),
            target=torch.randn(2, b * (D + 1), generator=g, dtype=torch.float64).to(td))
        full = mk(B)
        t = torch.tensor([0.0, 1.0], dtype=torch.float64)
        bs = min(B, 1 << 14)

        def cpu_sample():
            s = mk(bs)
            return dict(funcs=[s["func"]], u0=s["u0"], t=t, target=s["target"], kw=dict(method="dopri5"), batch=bs,
                        desc="%d of %d samples" % (bs, B))

        if fixed_rk4 is not None:
            dims = (D,) + tuple(hidden) + (D,)
            f_f = 2 * 2 * sum(a * b for a, b in zip(dims[:-1], dims[1:]))  # network + Hutchinson VJP
            return dict(desc="FFJORD tabular CNF D=%d hidden %s, B=%d, RK4 h=%g, t=[0,1], Hutchinson trace, %s (ConcatSquash "
                             "network evaluator, csrc/cnf_net.cu)" % (D, "x".join(map(str, hidden)), B, fixed_rk4, dtype),
                        dtype=dtype, also_generic=True,
                        argv=["-ts_adapt_type", "none", "-ts_trajectory_type", "memory"], funcs=[full["func"]], u0=full["u0"],
                        t=t, target=full["target"], kw=dict(method="rk4"), step=fixed_rk4, batch=B, flops_per_unit=16 * f_f,
                        bytes_per_unit=(2 * 4 + 2) * (D + 1) * (4 if dtype == "f32" else 8),
                        pipe="fp32_fma" if dtype == "f32" else "fp64_fma", each_call_setup=True, to_dev=cnf_to,
                        cpu_sample=lambda: dict(funcs=[mk(min(B, 256))["func"]], u0=mk(min(B, 256))["u0"], t=t,
                                                target=mk(min(B, 256))["target"], kw=dict(method="rk4"), batch=min(B, 256),
                                                desc="%d of %d samples" % (min(B, 256), B)))
        return dict(desc="cfg3 FFJORD tabular CNF, POWER-shaped D=6 H=60, B=%d, dopri5 adaptive rtol=atol=1e-4, h0=0.05, "
                         "t=[0,1], Hutchinson trace, %s" % (B, dtype), dtype=dtype, argv=["-ts_trajectory_type", "memory"],
                    funcs=[full["func"]], u0=full["u0"], t=t, target=full["target"], kw=dict(method="dopri5"), step=0.05,
                    batch=B, flops_per_unit=69120, flops_per_rejected=17280, bytes_per_unit=112 * (4 if dtype == "f32" else 8),
                    pipe="fp32_fma" if dtype == "f32" else "fp64_fma", also_generic=B <= (1 << 16), each_call_setup=True,
                    to_dev=cnf_to, cpu_sample=cpu_sample, peer_reduce=True)

    return build


def cfg4(C=32, HW=32, Nt=1):
    def build():
        from _workloads import OdeConvBlock

        B = 256
        g = torch.Generator().manual_seed(3 + SEED_OFFSET)
        u0 = torch.randn(B, C, HW, HW, generator=g)
        target = torch.randn(1, B, C, HW, HW, generator=g)
        t = torch.tensor([1.0], dtype=torch.float64)
        bs = 32
        # SURVEY.md 8d: 75.5 Mflop and 96 C HW w bytes per trajectory-step (every layer reads its input and writes its output
        # once per RHS evaluation, adjoint = 3 evaluations' worth, stage checkpoints): block 1-2 are HBM-bound on CUDA cores
        return dict(desc="cfg4 CIFAR SqueezeNext ODE block: u [256,%d,%d,%d] fp32, RK4, t=[1.0], Nt=%d (h=%g), conv+BN(train)"
                         % (C, HW, HW, Nt, 1.0 / Nt), dtype="f32", argv=["-ts_adapt_type", "none", "-ts_trajectory_type", "memory"],
                    funcs=[OdeConvBlock(C)], u0=u0, t=t, target=target, kw=dict(method="rk4"), step=1.0 / Nt, batch=B,
                    flops_per_unit=75.5e6, bytes_per_unit=96 * C * HW * HW * 4, pipe="fp32_fma", each_call_setup=True,
                    cpu_sample=lambda: dict(funcs=[OdeConvBlock(C)], u0=u0[:bs].clone(), t=t, target=target[:, :bs].clone(),
                                            kw=dict(method="rk4"), batch=bs, desc="%d of %d samples" % (bs, B)))

    return build


def cfg5(N=1024, B=256, dtype="f64", ark="3"):
    from _workloads import KSExplicit, KSImplicit, ks_dx

    def build():
        td = torch.float64 if dtype == "f64" else torch.float32
        g = torch.Generator().manual_seed(4 + SEED_OFFSET)
        u0 = (0.5 * torch.randn(B, N, generator=g, dtype=torch.float64)).to(td)
        target = torch.randn(2, B, N, generator=g, dtype=torch.float64).to(td)
        t = torch.tensor([0.0, 0.2], dtype=torch.float64)
        H = N * 25 // 8
        kw = dict(method="imex", imex_form=True, batch_size=B, linear_solver="torch", fixed_jacobian_across_solves=True)
        f_ex = 2 * (2 * N * H + 3 * H * H)
        bs = 32
        ns = {"3": 4, "l2": 3}[ark]  # stages: ns explicit evaluations + ns - 1 implicit solves forward, as many VJPs / transposed solves back
        return dict(desc="cfg5 SINODE KS: N=%d, MLP hidden %d, batch %d, ARKIMEX-%s h=0.2 one step, torch LU-type solver, "
                         "-snes_type ksponly, %s" % (N, H, B, ark, dtype), dtype=dtype,
                    argv=["-ts_adapt_type", "none", "-snes_type", "ksponly", "-ts_trajectory_type", "memory",
                          "-ts_arkimex_type", ark],
                    funcs=[KSImplicit(ks_dx(N), dtype=td), KSExplicit(N, dtype=td)], u0=u0, t=t, target=target, kw=kw,
                    step=0.2, batch=B, flops_per_unit=4 * ns * f_ex + 2 * (ns - 1) * 2 * N * N,
                    bytes_per_unit=3 * ns * 37.3e6 * 8 / B,
                    pipe="fp64_fma" if dtype == "f64" else "fp32_fma", also_generic=True,
                    # executed by the products: 4 forward + 8 backward layer sweeps of F_f / 2 MACs, (21 | 3) slice pairs, 2 ops
                    tensor_ops_per_unit=3 * ns * (f_ex / 2) * (21 if dtype == "f64" else 3) * 2,
                    cpu_sample=lambda: dict(funcs=[KSImplicit(ks_dx(N), dtype=td), KSExplicit(N, dtype=td)],
                                            u0=u0[:bs].clone(), t=t, target=target[:, :bs].clone(),
                                            kw=dict(kw, batch_size=bs), batch=bs, desc="%d of %d samples" % (bs, B)))

    return build


def burgers(N=1024, B=200, dtype="f64"):
    """SURVEY.md 8f.3: the second SINODE driver (examples-sinode/Burgers/Burgers.py:134-195, 359-377): 3-tap stencil + MLP of
    width 9N/8, batch 200, 10 output times, ARKIMEX; run_a100_512.sh uses -ts_arkimex_type 1bee and a fixed step."""
    from _workloads import BurgersExplicit, BurgersImplicit

    def build():
        td = torch.float64 if dtype == "f64" else torch.float32
        g = torch.Generator().manual_seed(5 + SEED_OFFSET)
        x = torch.linspace(0, 1, N + 1, dtype=torch.float64)[:-1]
        u0 = (torch.sin(2 * torch.pi * x)[None, :] * (0.5 + torch.rand(B, 1, generator=g, dtype=torch.float64))).to(td)
        T, h = 10, 0.01
        t = torch.arange(T, dtype=torch.float64) * h
        target = torch.randn(T, B, N, generator=g, dtype=torch.float64).to(td)
        H = N * 9 // 8
        kw = dict(method="imex", imex_form=True, batch_size=B, linear_solver="torch", fixed_jacobian_across_solves=True)
        f_ex = 2 * (2 * N * H + 3 * H * H)
        bs = 25
        mk = lambda: [BurgersImplicit(N, dtype=td), BurgersExplicit(N, dtype=td)]
        return dict(desc="Burgers SINODE: N=%d, MLP width %d, batch %d, ARKIMEX 1bee h=0.01, 10 output times, torch solver, "
                         "-snes_type ksponly, %s" % (N, H, B, dtype), dtype=dtype,
                    argv=["-ts_adapt_type", "none", "-snes_type", "ksponly", "-ts_arkimex_type", "1bee", "-ts_trajectory_type",
                          "memory"], funcs=mk(), u0=u0, t=t, target=target, kw=kw, step=h, batch=B,
                    flops_per_unit=(3 + 3 * 3) * f_ex + 6 * 2 * N * N, bytes_per_unit=12 * 8 * (2 * N * H + 3 * H * H) / B,
                    pipe="fp64_fma" if dtype == "f64" else "fp32_fma", also_generic=True,
                    cpu_sample=lambda: dict(funcs=mk(), u0=u0[:bs].clone(), t=t, target=target[:, :bs].clone(),
                                            kw=dict(kw, batch_size=bs), batch=bs, desc="%d of %d samples" % (bs, B)))

    return build


def config_table():
    return {"1": ("cfg1", cfg1), "2S": ("cfg2-f32", cfg2("f32")), "2D": ("cfg2-f64", cfg2("f64")),
            "2L": ("cfg2-f64-solution-only", cfg2("f64", lean=True)), "3": ("cfg3", _cnf(1000, "f32")), "3L": ("cfg3-2^20", _cnf(1 << 20, "f32")),
            "3D": ("cfg3-f64", _cnf(1000, "f64")),
            "3M": ("ffjord-miniboone", _cnf(1000, "f32", 43, (860, 860), 0.25)), "4": ("cfg4", cfg4()), "4b": ("cfg4-block2", cfg4(64, 16)),
            "4n": ("cfg4-Nt4", cfg4(32, 32, 4)), "4c": ("cfg4-block3", cfg4(128, 8)), "4d": ("cfg4-block4", cfg4(256, 4)),
            "5": ("cfg5", cfg5()), "5S": ("cfg5-f32", cfg5(dtype="f32")), "5L": ("cfg5-l2", cfg5(ark="l2")),
            "B": ("burgers", burgers())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="1,3,3L,4,5")
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--cpu", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "configs.jsonl"))
    args = ap.parse_args()
    import ctypes as C

    from pnode_b200 import _lib

    lib = _lib.load()
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(
        os.path.join(ROOT, "MEASURED_PEAKS.json")) else {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}
    pk = {"hbm_gbs": peaks["hbm_gbs"], "bf16_tensor": peaks["bf16_tflops"]}
    for code, key in ((_lib.F32, "fp32_fma"), (_lib.F64, "fp64_fma")):
        fl, ms = C.c_double(), C.c_float()
        _lib.check(lib.pnode_peak_fma(code, 20000, C.byref(fl), C.byref(ms)))
        pk[key] = fl.value / (ms.value * 1e-3) / 1e12
    table = config_table()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "a") as fo:
        for c in args.configs.split(","):
            name, build = table[c]
            try:
                res = run_config(name, build, args, pk)
            except Exception as e:  # keep going: one failing config must not hide the others
                res = {"config": name, "error": repr(e)[:300]}
            res["peaks"] = pk
            line = json.dumps(res)
            print(line, flush=True)
            fo.write(line + "\n")


if __name__ == "__main__":
    main()
