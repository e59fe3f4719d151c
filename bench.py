#!/usr/bin/env python
"""bench.py -- fwd + discrete-adjoint trajectory-steps/s of the pnode hot path on B200 (BASELINE.json metric).

Workload (N=1): BASELINE.json configs[1] -- the spiral MLP ODE (Linear(2,50)-Tanh-Linear(50,2) on y**3,
examples-pnode/ode_demo_petsc.py:207-230) scaled to 2^20 synthetic trajectories, RK4, 10 output times = 9 steps of
h = 0.025, `odeint_adjoint` + `loss.backward()`.  A "step" of this bench is one such fwd+adjoint pass over the batch.
A trajectory-step = one sample advanced one accepted step forward plus its adjoint step (BASELINE.md section 3).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dtype f64|f32] [--impl reference] [--no-configs]
                    [--dump-outputs DIR]
`--dump-outputs DIR` writes what the last timed pass handed its caller (see dump_outputs) as DIR/<name>.npy; the inputs are
seeded, so two builds run with the same arguments can be compared output for output.
Besides the headline the line carries `parity` (a 32-trajectory slice against the CPU oracle; at N > 1 bit-equality of mu
across ranks) and `configs`: every BASELINE.json shape through the drop-in (bench_configs.py) -- ms per pass, rate, roofline,
bounded CPU baseline at N = 1; the sharding configs (3, 4, 5) weak-scaled at N > 1.
N>1: launched by torchrun, one rank per GPU, weak scaling (2^20 trajectories per GPU), the only collective is the NCCL
all-reduce of mu (252 scalars) inside backward.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402

NTRAJ = 1 << 20
T_OUT = 10
H = 0.025
NSTEPS = T_OUT - 1
STAGES = 4
DIM, HIDDEN = 2, 50
# DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) of ONE mlp_rk_adj_kernel launch on the default workload, from the
# `ncu --set full` captures summarised in profiles/r1_ncu_full_spiral_f64_v3.txt / r1_ncu_full_spiral_f32_v2.txt
NCU_ADJ_TRAFFIC = {("f64", 1 << 20): 772.183552e6 + 19.816192e6, ("f32", 1 << 20): 386.1e6 + 10.5e6}
METRIC = "fwd+adjoint trajectory-steps/sec"
UNIT = "trajectory-steps/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--dtype", choices=["f64", "f32"], default="f64")
    ap.add_argument("--impl", choices=["native", "reference"], default="native")
    ap.add_argument("--ntraj", type=int, default=NTRAJ, help="trajectories per GPU")
    ap.add_argument("--cpu-sample", type=int, default=1 << 19,
                    help="trajectories of the bounded CPU-baseline sample inside the native arm's line (the --impl reference "
                         "arm runs the full --ntraj batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config table (`configs` key of the JSON line)")
    ap.add_argument("--config-iters", type=int, default=5)
    ap.add_argument("--no-peer", action="store_true", help="N>1: all-reduce mu with NCCL instead of inside the adjoint kernel")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed pass to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def make_problem(ntraj, dtype, seed=0):
    """Synthetic inputs of SURVEY.md section 8d (cfg1/2), generated on the CPU so every arm sees identical data."""
    from _problems import SpiralFunc

    g = torch.Generator().manual_seed(seed)
    u0 = ((torch.rand(ntraj, 1, 2, generator=g, dtype=torch.float64) * 2 - 1) * 2).to(dtype)
    t = torch.arange(T_OUT, dtype=torch.float64) * H
    target = torch.randn(T_OUT, ntraj, 1, 2, generator=g, dtype=torch.float64).to(dtype)
    func = SpiralFunc(dtype=dtype)
    return func, u0, t, target


DUMP_TRAJ = 1 << 17  # trajectories in the --dump-outputs sample of the solution: 21 MB in fp64


def dump_outputs(path, pred, loss, func):
    """What one pass hands its caller, in the run's dtype: `solution`, the trajectory at the output times
    [T_OUT, n, 1, DIM] of a fixed seeded sample of n = min(batch, DUMP_TRAJ) trajectories in batch order; the scalar
    `loss`; `grad_<parameter>` for every parameter of the model."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    ntraj = pred.shape[1]
    idx = torch.randperm(ntraj, generator=torch.Generator().manual_seed(0))[:DUMP_TRAJ].sort().values
    arrays = {"solution": pred.detach()[:, idx.to(pred.device)], "loss": loss.detach()}
    arrays.update(("grad_" + name, p.grad) for name, p in func.named_parameters())
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a.cpu().numpy())


def headline_config(world, ntraj, exchange):
    """`config` of the JSON line: the SAME object for the native and the reference arm at equal --gpus / --ntraj."""
    w = 8
    return {"workload": "spiral MLP 2-50-2 on y**3 (BASELINE configs[1]), 2^20 trajectories per GPU, RK4 fixed "
                        "step, 10 output times = 9 steps of h=0.025, odeint_adjoint + loss.backward()",
            "ntraj_per_gpu": ntraj, "global_ntraj": world * ntraj, "method": "rk4", "steps_per_pass": NSTEPS,
            "parallelism": "batch-sharded dp%d; only exchange = all-reduce of mu (252 scalars), %s" % (world, exchange),
            "l2": "per-pass working set (stage checkpoints %.0f MB + grad_output %.0f MB in fp64) exceeds the 126 MB L2; "
                  "no explicit flush" % (ntraj * NSTEPS * STAGES * DIM * w / 1e6, ntraj * T_OUT * DIM * w / 1e6)}


def exchange_desc(world, peer):
    if world == 1:
        return "single rank"
    return "fused into the adjoint kernel over NVLink peer memory" if peer else "NCCL"


# ----------------------------------------------------------------------------------------------------------------------
# CPU arms: the oracle (reference-structured restatement; PETSc is not installable here -- BASELINE.md section 4)


def cpu_port_rate(ntraj, dtype, reps=1):
    from oracle import OracleODEPetsc

    torch.set_num_threads(os.cpu_count() or 1)
    func, u0, t, target = make_problem(ntraj, dtype)
    ode = OracleODEPetsc(["-ts_adapt_type", "none", "-ts_trajectory_type", "memory"])
    ode.setupTS(u0, func, step_size=H, method="rk4", enable_adjoint=True)

    def one():
        func.zero_grad()
        pred = ode.odeint_adjoint(u0, t)
        loss = torch.mean(torch.abs(pred - target))
        loss.backward()
        return loss.item()

    one()  # warm-up
    t0 = time.perf_counter()
    for _ in range(reps):
        one()
    dt = (time.perf_counter() - t0) / reps
    return ntraj * NSTEPS / dt, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dtype = torch.float64 if args.dtype == "f64" else torch.float32
    cores = os.cpu_count() or 1
    ntraj = args.ntraj  # the full per-GPU batch of the native arm: same config on both arms
    torch.set_num_threads(cores)
    from oracle import OracleODEPetsc

    func, u0, t, target = make_problem(ntraj, dtype)
    ode = OracleODEPetsc(["-ts_adapt_type", "none", "-ts_trajectory_type", "memory"])
    ode.setupTS(u0, func, step_size=H, method="rk4", enable_adjoint=True)

    def one(keep=False):
        func.zero_grad()
        pred = ode.odeint_adjoint(u0, t)
        loss = torch.mean(torch.abs(pred - target))
        loss.backward()
        return (pred.detach(), loss.detach()) if keep else None

    for _ in range(max(args.warmup, 1)):
        one()
    t0 = time.perf_counter()
    for i in range(args.steps):
        kept = one(keep=args.dump_outputs is not None and i == args.steps - 1)
    total = time.perf_counter() - t0
    if kept is not None:
        dump_outputs(args.dump_outputs, *kept, func)
        del kept
    value = ntraj * NSTEPS * args.steps / total
    sample = "all %d trajectories of one GPU's batch per step (same model, schedule, dtype), %d warm-up + %d timed passes" % (
        ntraj, max(args.warmup, 1), args.steps)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
        "config": headline_config(args.gpus, ntraj, exchange_desc(args.gpus, not args.no_peer)),
        "note": "reference-structured CPU restatement on the host cores (PETSc unavailable: not installed, unpinned, no "
                "network); at --gpus N > 1 rank 0 alone runs ONE GPU's batch",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------------


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.samples = []
        self._proc = None

    def __enter__(self):
        # one long-lived sampler process (100 ms period) for the whole timed region -- B200_PROFILING.md "clocks line"
        try:
            self._proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                                           "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                          stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self._proc = None
        time.sleep(0.25)
        return self

    def __exit__(self, *a):
        if self._proc is None:
            return
        time.sleep(0.15)
        self._proc.terminate()
        try:
            out, _ = self._proc.communicate(timeout=5)
        except Exception:
            self._proc.kill()
            out = ""
        for ln in (out or "").strip().splitlines():
            self.samples.append([x.strip() for x in ln.split(",")])

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[1]))
                mx.append(float(s[2]))
                for name, val in zip(names, s[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


def parity_check(args, dtype, dev, func, u0_h, t_h, target_h, world):
    """32 trajectories of this rank's batch: product on the GPU (single-rank solve, the fused sweeps) vs the CPU oracle."""
    import copy

    from oracle import OracleODEPetsc
    from pnode import petsc_adjoint

    n = 32
    u0s, tgts = u0_h[:n].clone(), target_h[:, :n].clone()
    res = []
    for where in ("cpu", "cuda"):
        f = copy.deepcopy(func).to("cpu" if where == "cpu" else dev)
        ode = OracleODEPetsc(["-ts_adapt_type", "none"]) if where == "cpu" else petsc_adjoint.ODEPetsc()
        d = "cpu" if where == "cpu" else dev
        ode.setupTS(u0s.to(d), f, step_size=H, method="rk4", enable_adjoint=True)
        y0 = u0s.to(d).clone().requires_grad_(True)
        pred = ode.odeint_adjoint(y0, t_h.to(d))
        torch.mean(torch.abs(pred - tgts.to(d))).backward()
        res.append((pred.detach().cpu().double(), y0.grad.cpu().double(),
                    torch.cat([p.grad.reshape(-1) for p in f.parameters()]).cpu().double()))
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max())
    errs = [rel(a, b) for a, b in zip(res[1], res[0])]
    tol = 1e-10 if dtype == torch.float64 else 1e-4
    out = {"oracle_slice": {"trajectories": n, "rel_err_trajectory": errs[0], "rel_err_lambda": errs[1], "rel_err_mu": errs[2],
                            "tolerance": tol, "ok": max(errs) < tol}}
    assert out["oracle_slice"]["ok"], "parity check against the oracle failed: %r" % (out,)
    return out


def per_config_table(args, world, rank, comm):
    """BASELINE.json "each named shape": one entry per config through the drop-in.  N = 1: every config with its bounded CPU
    baseline (rank 0).  N > 1: the configs that shard (3, 4, 5) weak-scaled, every rank taking part, whole-job rates."""
    import types

    import bench_configs as bc

    peaks, kind = measured_peaks()
    pk = {"hbm_gbs": peaks["hbm_gbs"], "bf16_tensor": peaks["bf16_tflops"], "source": kind}
    import ctypes as C

    from pnode_b200 import _lib

    lib = _lib.load()
    for code, key in ((_lib.F32, "fp32_fma"), (_lib.F64, "fp64_fma")):
        fl, ms = C.c_double(), C.c_float()
        _lib.check(lib.pnode_peak_fma(code, 20000, C.byref(fl), C.byref(ms)))
        pk[key] = fl.value / (ms.value * 1e-3) / 1e12
    names = ["1", "2S", "2L", "3", "3L", "4", "4n", "4b", "4c", "4d", "5", "5L", "5S"] if world == 1 else ["3L", "4", "5"]
    a = types.SimpleNamespace(iters=args.config_iters, cpu=(world == 1 and not args.no_cpu_baseline), no_generic=True)
    bc.SEED_OFFSET = 100 * rank
    table, out = bc.config_table(), {"peaks": pk}
    for c in names:
        name, build = table[c]
        try:
            r = bc.run_config(name, build, a, pk, world=world, comm=comm if world > 1 else None)
        except Exception as e:  # one failing config must not take the headline down with it
            r = {"error": repr(e)[:300]}
        keep = {k: r[k] for k in ("workload", "dtype", "path", "n_gpus", "ms_per_pass", "traj_steps_per_s", "accepted_steps",
                                  "attempts", "algorithmic_tflops", "roofline", "cpu_baseline", "speedup_vs_cpu_port",
                                  "rhs_evaluator", "cuda_graph_replay_ms_per_pass", "cuda_graph_error", "error")
                if k in r}
        out[name] = keep
    return out


def run_native(args):
    import torch.distributed as dist

    from pnode import petsc_adjoint
    from pnode_b200 import _lib
    from pnode_b200.options import Options

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the native arm has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    dtype = torch.float64 if args.dtype == "f64" else torch.float32
    w = 8 if dtype == torch.float64 else 4
    ntraj = args.ntraj

    Options.insert_args(["-ts_adapt_type", "none", "-ts_trajectory_type", "memory"])
    func, u0_h, t_h, target_h = make_problem(ntraj, dtype, seed=rank)
    func = func.to(dev)
    if world > 1:  # identical replicas of the model on every rank
        for p in func.parameters():
            dist.broadcast(p.data, 0)
    u0_pin, target_pin = u0_h.pin_memory(), target_h.pin_memory()
    t_dev = t_h.to(dev)
    u0_dev, target_dev = u0_pin.to(dev), target_pin.to(dev)

    ode = petsc_adjoint.ODEPetsc()
    if world > 1:
        from pnode_b200.parallel import BatchComm

        ode.comm = BatchComm()
        if not args.no_peer:
            ode.comm.enable_peer_reduce()
    ode.setupTS(u0_dev, func, step_size=H, method="rk4", enable_adjoint=True)

    # --dump-outputs: the pass numbered keep["at"] (the final timed one) keeps what it returned, detached so that its
    # stage checkpoints are freed with the autograd graph; every other pass keeps nothing
    keep = {"passes": 0, "at": None}

    def step_resident():
        func.zero_grad(set_to_none=True)
        pred = ode.odeint_adjoint(u0_dev, t_dev)
        loss = torch.mean(torch.abs(pred - target_dev))
        loss.backward()
        keep["passes"] += 1
        if keep["passes"] == keep["at"]:
            keep["out"] = (pred.detach(), loss.detach())
        return loss

    grads_host = torch.empty(ode.np, dtype=dtype).pin_memory()

    # end to end: host buffers in, host results out, every H2D / D2H copy inside the timed region.  Like any input
    # pipeline, the upload of pass i+1 (pinned memory, copy stream) overlaps the sweeps of pass i; each pass still moves its
    # own h2d_bytes_per_step and synchronises on its own loss value.
    copy_stream = torch.cuda.Stream(device=dev)
    staged = {}

    def upload():
        with torch.cuda.stream(copy_stream):
            u0 = u0_pin.to(dev, non_blocking=True)
            target = target_pin.to(dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        staged["next"] = (u0, target, ev)

    def step_e2e():
        func.zero_grad(set_to_none=True)
        if "next" not in staged:
            upload()
        u0, target, ev = staged.pop("next")
        torch.cuda.current_stream().wait_event(ev)
        u0.record_stream(torch.cuda.current_stream())
        target.record_stream(torch.cuda.current_stream())
        upload()  # next pass's inputs start moving now
        pred = ode.odeint_adjoint(u0, t_dev)
        loss = torch.mean(torch.abs(pred - target))
        loss.backward()
        off = 0
        for p in func.parameters():
            grads_host[off:off + p.numel()].copy_(p.grad.reshape(-1), non_blocking=True)
            off += p.numel()
        return loss.item()  # D2H of the scalar loss; synchronises

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            tmax = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            ms = float(tmax.item())
        return ms

    # ---- correctness bit carried by the line: (1) a 32-trajectory slice of this rank's batch through the product against the
    # CPU oracle; (2) at N > 1, mu after the in-kernel / NCCL all-reduce is bit-identical on every rank
    parity = parity_check(args, dtype, dev, func, u0_h, t_h, target_h, world)

    for _ in range(max(args.warmup, 3)):
        step_resident()
    assert ode.path == "fused-mlp-rk", "bench must run the fused CUDA sweep, got %r" % ode.path
    if world > 1:
        mu_now = torch.cat([p.grad.reshape(-1) for p in func.parameters()]).contiguous()
        gathered = [torch.empty_like(mu_now) for _ in range(world)]
        dist.all_gather(gathered, mu_now)
        parity["mu_bit_equal_across_ranks"] = all(torch.equal(gathered[0], gk) for gk in gathered[1:])
        assert parity["mu_bit_equal_across_ranks"], "mu differs between ranks after the all-reduce"
    fused = ode._fused
    l0 = fused.launches + ode._ops.launches
    if args.dump_outputs and rank == 0:
        keep["at"] = keep["passes"] + args.steps
    with ClockSampler(local) as clk:
        ms = timed(step_resident, args.steps)
    launches = fused.launches + ode._ops.launches - l0
    clocks = clk.summary()
    if "out" in keep:  # before the passes below overwrite the gradients
        dump_outputs(args.dump_outputs, *keep.pop("out"), func)
    total_units = world * ntraj * NSTEPS * args.steps
    value = total_units / (ms * 1e-3)

    for _ in range(3):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps)
    staged.clear()
    torch.cuda.synchronize()
    e2e_value = total_units / (ms_e2e * 1e-3)
    h2d = u0_pin.numel() * w + target_pin.numel() * w
    d2h = ode.np * w + w

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": args.dtype, "data": "synthetic",
        "config": headline_config(world, ntraj, exchange_desc(world, ode.comm is not None and ode.comm.peer is not None)),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches,
        "clocks": clocks,
        "parity": parity,
    }
    if not args.no_configs:
        line["configs"] = per_config_table(args, world, rank, ode.comm)

    if rank == 0:
        # ---- per-kernel timing of the two sweeps (CUDA events on the launching stream) + rooflines -----------------
        peaks, peak_kind = measured_peaks()
        u_flat = u0_dev.reshape(-1)
        times = [float(x) for x in t_h]
        gout = torch.randn(T_OUT, ntraj * DIM, dtype=dtype, device=dev)
        reps = max(args.steps, 5)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        tf = ta = 0.0
        for i in range(reps + 2):
            torch.cuda.synchronize()
            ev[0].record()
            sol, ckpt, sched = fused.forward(u_flat, times, H, True)
            ev[1].record()
            fused.adjoint(gout, ckpt, sched, ntraj)
            ev[2].record()
            torch.cuda.synchronize()
            if i >= 2:
                tf += ev[0].elapsed_time(ev[1])
                ta += ev[1].elapsed_time(ev[2])
        tf, ta = tf / reps, ta / reps
        units = ntraj * NSTEPS
        adj_bytes = units * (STAGES * DIM + DIM) * w + ntraj * DIM * w  # read Y_i + grad_output, write lambda
        fwd_bytes = units * (STAGES * DIM + DIM) * w + ntraj * DIM * w  # write Y_i + outputs, read u0
        adj_flops = units * STAGES * 3 * 2 * (2 * DIM * HIDDEN)  # recompute + input-grad + weight-grad (SURVEY 8d)
        fwd_flops = units * STAGES * 2 * (2 * DIM * HIDDEN)
        lib = _lib.load()
        import ctypes as C

        fl, pms = C.c_double(), C.c_float()
        _lib.check(lib.pnode_peak_fma(_lib.F64 if dtype == torch.float64 else _lib.F32, 20000, C.byref(fl), C.byref(pms)))
        fma_peak = fl.value / (pms.value * 1e-3) / 1e12
        ach = adj_bytes / (ta * 1e-3) / 1e9
        line["roofline"] = {"bound": "hbm", "kernel": "mlp_rk_adj_kernel", "achieved": ach, "peak": peaks["hbm_gbs"],
                            "unit": "GB/s", "frac": ach / peaks["hbm_gbs"],
                            "traffic": NCU_ADJ_TRAFFIC.get((args.dtype, ntraj)), "algorithmic_bytes": adj_bytes,
                            "peak_source": peak_kind,
                            "ms_per_launch": ta,
                            "note": "arithmetic intensity ~60 flop/B: the kernel is bound by the %s FMA/transcendental "
                                    "issue rate, not HBM -- see roofline_compute" % args.dtype}
        line["roofline_compute"] = {
            "pipe": "%s CUDA-core FMA" % args.dtype, "peak_tflops_measured": fma_peak,
            "adjoint": {"ms": ta, "algorithmic_tflops": adj_flops / (ta * 1e-3) / 1e12,
                        "frac": adj_flops / (ta * 1e-3) / 1e12 / fma_peak},
            "forward": {"ms": tf, "algorithmic_tflops": fwd_flops / (tf * 1e-3) / 1e12,
                        "frac": fwd_flops / (tf * 1e-3) / 1e12 / fma_peak, "hbm_gbs": fwd_bytes / (tf * 1e-3) / 1e9},
            "note": "algorithmic flops exclude tanh (400 evaluations per trajectory-step; fp64: 11 FP64 + 7 integer "
                    "instructions each).  ncu: an FP64 instruction holds the dispatch port two cycles, the port is busy "
                    "98.5 % of the forward sweep's cycles (issue-active + FP64 share) -- the sweep is bound by its "
                    "instruction count; the adjoint by shared-memory wavefronts (0.91 per cycle).  DESIGN.md section 8.6"}
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            rate, dt = cpu_port_rate(args.cpu_sample, dtype, reps=3)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": "%d of %d trajectories, 1 warm-up + 3 timed fwd+adjoint passes (%.1f s each), oracle = "
                                              "reference-structured CPU restatement (PETSc unavailable)" %
                                              (args.cpu_sample, ntraj, dt)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
