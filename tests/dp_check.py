"""Run under torchrun (N ranks, one per GPU): the batch-sharded fused spiral path vs a single-rank run of the full batch.
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29611 tests/dp_check.py
Also exercised by tests/test_gpu_dp.py when >= 2 GPUs are visible."""
import copy
import os
import sys

import torch
import torch.distributed as dist

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)


def main():
    from _problems import SpiralFunc, TimeMLP, rel_err, spiral_inputs
    from pnode import petsc_adjoint
    from pnode_b200.options import Options
    from pnode_b200.parallel import BatchComm, shard_batch

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    comm = BatchComm()
    if "--peer" in sys.argv:
        assert comm.enable_peer_reduce(), "peer-memory all-reduce could not be enabled"

    def run(func, u, go, t, method, step, comm_, argv):
        Options.clear_all()
        Options.insert_args(argv)
        f = copy.deepcopy(func).to(dev)
        ode = petsc_adjoint.ODEPetsc()
        ode.comm = comm_
        ode.setupTS(u.to(dev), f, step_size=step, method=method, enable_adjoint=True)
        y0 = u.to(dev).clone().requires_grad_(True)
        out = ode.odeint_adjoint(y0, t.to(dev))
        (out * go.to(dev)).sum().backward()
        torch.cuda.synchronize()
        return out.detach().cpu(), y0.grad.cpu(), [p.grad.cpu() for p in f.parameters()], ode

    # 1. fused spiral, fixed step (mu all-reduce only)
    B = 4099
    u0, t, gout = spiral_inputs(B)
    func = SpiralFunc()
    full = run(func, u0, gout, t, "rk4", 0.025, None, ["-ts_adapt_type", "none"])
    mine = run(func, shard_batch(u0, rank, world).contiguous(), shard_batch(gout, rank, world, dim=1).contiguous(), t,
               "rk4", 0.025, comm, ["-ts_adapt_type", "none"])
    assert mine[3].path == "fused-mlp-rk"
    assert rel_err(mine[0], shard_batch(full[0], rank, world, dim=1)) < 1e-13
    assert rel_err(mine[1], shard_batch(full[1], rank, world)) < 1e-12
    for a, b in zip(mine[2], full[2]):
        assert rel_err(a, b) < 1e-11, rel_err(a, b)

    # 1b. the same with -ts_trajectory_solution_only 1: u_n per step in HBM, stages recomputed inside the adjoint kernel
    lean = run(func, shard_batch(u0, rank, world).contiguous(), shard_batch(gout, rank, world, dim=1).contiguous(), t,
               "rk4", 0.025, comm, ["-ts_adapt_type", "none", "-ts_trajectory_solution_only", "1"])
    assert lean[3].path == "fused-mlp-rk" and lean[3]._fused.solution_only
    assert rel_err(lean[0], shard_batch(full[0], rank, world, dim=1)) < 1e-13
    assert rel_err(lean[1], shard_batch(full[1], rank, world)) < 1e-12
    for a, b in zip(lean[2], full[2]):
        assert rel_err(a, b) < 1e-11, rel_err(a, b)

    # 2. generic adaptive dopri5: one scalar all-reduce per attempt => same step sequence as the single-rank run
    g = torch.Generator().manual_seed(5)
    u1 = torch.randn(1000, 6, generator=g, dtype=torch.float64)
    go1 = torch.randn(3, 1000, 6, generator=g, dtype=torch.float64)
    t1 = torch.tensor([0.0, 0.4, 1.0], dtype=torch.float64)
    f1 = TimeMLP(d=6, hidden=16)
    argv = ["-ts_rtol", "1e-6", "-ts_atol", "1e-6"]
    full = run(f1, u1, go1, t1, "dopri5", 0.3, None, argv)
    mine = run(f1, shard_batch(u1, rank, world).contiguous(), shard_batch(go1, rank, world, dim=1).contiguous(), t1,
               "dopri5", 0.3, comm, argv)
    la, lb = full[3]._loop.attempts, mine[3]._loop.attempts
    assert [a[2] for a in la] == [b[2] for b in lb] and any(not a[2] for a in la)
    for a, b in zip(la, lb):
        assert abs(a[1] - b[1]) <= 1e-10 * abs(a[1])
    assert rel_err(mine[0], shard_batch(full[0], rank, world, dim=1)) < 1e-10
    for a, b in zip(mine[2], full[2]):
        assert rel_err(a, b) < 1e-10
    # 3. conv ODE block (BASELINE config 4), batch sharded: train-mode BatchNorm needs the statistics of the GLOBAL batch.  The
    #    kernels exchange exact integer totals over NVLink peer memory in their tail: every rank holds bit-identical statistics,
    #    and the sharded run reproduces the single-GPU run of the whole batch to rounding (the per-CTA partial sums group the
    #    pixels differently when the batch is split, nothing else differs).
    if "--peer" in sys.argv:
        from _workloads import OdeConvBlock

        # third case: the tensor-core evaluator (csrc/conv_mma.cu), statistics exchanged inside its finalize kernels
        for dtype, shape, tol, extra in ((torch.float64, (4 * world, 16, 8, 8), 1e-12, []),
                                         (torch.float32, (16 * world, 32, 16, 16), 2e-5, []),
                                         (torch.float32, (8 * world, 128, 4, 4), 2e-5, ["-pnode_convblock_mma", "1"])):
            g = torch.Generator().manual_seed(9)
            u2 = torch.randn(shape, generator=g, dtype=torch.float64).to(dtype)
            go2 = torch.randn((1,) + shape, generator=g, dtype=torch.float64).to(dtype)
            t2 = torch.tensor([1.0], dtype=torch.float64)
            f2 = OdeConvBlock(shape[1], dtype=dtype)
            argv = ["-ts_adapt_type", "none", "-pnode_convblock_native", "1"] + extra
            full = run(f2, u2, go2, t2, "rk4", 0.5, None, argv)
            mine = run(f2, shard_batch(u2, rank, world).contiguous(), shard_batch(go2, rank, world, dim=1).contiguous(), t2,
                       "rk4", 0.5, comm, argv)
            assert mine[3]._cb_im.native and mine[3]._cb_im._comm is comm and bool(mine[3]._cb_im.mma) == bool(extra)
            flat = lambda gs: torch.cat([q.double().reshape(-1) for q in gs])
            errs = (rel_err(mine[0], shard_batch(full[0], rank, world, dim=1)), rel_err(mine[1], shard_batch(full[1], rank, world)),
                    rel_err(flat(mine[2]), flat(full[2])))
            fa, fb = mine[3].funcIM, full[3].funcIM
            errs += (rel_err(fa.bn3.running_var.cpu(), fb.bn3.running_var.cpu()), rel_err(fa.bn5.running_mean.cpu(), fb.bn5.running_mean.cpu()))
            if rank == 0:
                print("conv block sharded vs full batch (%s): trajectory %.2e lambda %.2e mu %.2e running stats %.2e %.2e" %
                      ((str(dtype),) + errs), flush=True)
            assert max(errs) < tol, errs
            assert int(fa.bn3.num_batches_tracked) == int(fb.bn3.num_batches_tracked)
            # every rank holds the SAME statistics bit for bit (exact integer exchange): compare the BatchNorm buffers across ranks
            rv = fa.bn4.running_var.detach().clone()
            ref = rv.clone()
            dist.broadcast(ref, 0)
            assert torch.equal(rv, ref), "BatchNorm statistics differ across ranks"
    # 4. fused FFJORD CNF (BASELINE config 3), adaptive dopri5, batch sharded.  With the peer inbox the whole time loop runs on
    #    the device of every rank (error norm summed over NVLink in the attempt kernel); without it the host drives the loop
    #    with one NCCL scalar per attempt.  Either way: the step sequence of the single-GPU run of the whole batch.
    from _workloads import CNFFunc, cnf_to

    Bc, D = 96 * world + 0, 6
    assert Bc % world == 0
    fc = CNFFunc(Bc, D, (60,), dtype=torch.float64, seed=3)
    with torch.no_grad():
        for prm in fc.parameters():
            prm.mul_(4.0)  # stiffer: the first big step is rejected
    g = torch.Generator().manual_seed(9)
    zc = torch.randn(Bc, D, generator=g, dtype=torch.float64)
    gz = torch.randn(3, Bc, D, generator=g, dtype=torch.float64)
    gl = torch.randn(3, Bc, generator=g, dtype=torch.float64)
    tc = torch.tensor([0.0, 0.3, 1.0], dtype=torch.float64)
    argv = ["-ts_rtol", "1e-7", "-ts_atol", "1e-7"]

    def run_cnf(func, z, gz_, gl_, comm_):
        Options.clear_all()
        Options.insert_args(argv)
        f = cnf_to(copy.deepcopy(func), dev)
        nb = z.shape[0]
        u = torch.cat((z.reshape(-1), torch.zeros(nb, dtype=torch.float64))).to(dev)
        go = torch.cat((gz_.reshape(3, -1), gl_), dim=1).to(dev)
        ode = petsc_adjoint.ODEPetsc()
        ode.comm = comm_
        ode.setupTS(u, f, step_size=0.5, method="dopri5", enable_adjoint=True)
        y0 = u.clone().requires_grad_(True)
        out = ode.odeint_adjoint(y0, tc.to(dev))
        (out * go).sum().backward()
        torch.cuda.synchronize()
        split = lambda v: (v[..., : nb * D].reshape(v.shape[:-1] + (nb, D)).cpu(), v[..., nb * D:].cpu())
        return split(out.detach()), split(y0.grad), [p.grad.cpu() for p in f.parameters()], ode

    full = run_cnf(fc, zc, gz, gl, None)
    lo, hi = rank * (Bc // world), (rank + 1) * (Bc // world)
    fs = copy.deepcopy(fc)
    fs.base_func._e = fc.base_func._e[lo:hi].clone()
    fs.y0 = tuple(x[lo:hi].clone() for x in fc.y0)
    mine = run_cnf(fs, zc[lo:hi], gz[:, lo:hi], gl[:, lo:hi], comm)
    assert mine[3].path == "fused-cnf-rk" and full[3].path == "fused-cnf-rk"
    la, lb = full[3]._loop.attempts, mine[3]._loop.attempts
    assert [a[2] for a in la] == [b[2] for b in lb] and any(not a[2] for a in la), (la, lb)
    for a, b in zip(la, lb):
        assert abs(a[1] - b[1]) <= 1e-9 * abs(a[1]), (a, b)
    for k in (0, 1):  # trajectory, lambda: (z part, logp part)
        assert rel_err(mine[k][0], full[k][0][..., lo:hi, :]) < 2e-9, ("cnf z", k)
        assert rel_err(mine[k][1], full[k][1][..., lo:hi]) < 2e-9, ("cnf logp", k)
    for a, b in zip(mine[2], full[2]):
        assert rel_err(a, b) < 2e-9, rel_err(a, b)
    if rank == 0:
        print("cnf sharded vs full batch: %d attempts, device loop on every rank: %s" %
              (len(lb), comm.peer is not None), flush=True)

    # 5. SINODE pair (BASELINE config 5 in small: circulant implicit half + wide ReLU MLP on the tensor-core evaluator), batch
    #    sharded: no exchange inside the sweep; the MLP's parameter gradient is all-reduced LAYER BY LAYER on a side stream as
    #    the last vector-Jacobian product finishes each layer (BatchComm.allreduce_sum_layered)
    from _workloads import KSExplicit, KSImplicit, ks_dx

    N5, B5 = 64, 8 * world
    g = torch.Generator().manual_seed(4)
    u5 = 0.5 * torch.randn(B5, N5, generator=g, dtype=torch.float64)
    go5 = torch.randn(2, B5, N5, generator=g, dtype=torch.float64)
    t5 = torch.tensor([0.0, 0.2], dtype=torch.float64)
    f_im0, f_ex0 = KSImplicit(ks_dx(N5)), KSExplicit(N5, hidden=200)

    def run_ks(u, go, comm_, nb):
        Options.clear_all()
        Options.insert_args(["-ts_adapt_type", "none", "-snes_type", "ksponly"])
        f_im, f_ex = copy.deepcopy(f_im0).to(dev), copy.deepcopy(f_ex0).to(dev)
        ode = petsc_adjoint.ODEPetsc()
        ode.comm = comm_
        ode.setupTS(u.to(dev), f_im, step_size=0.1, method="imex", imex_form=True, func2=f_ex, batch_size=nb,
                    linear_solver="torch")
        y0 = u.to(dev).clone().requires_grad_(True)
        out = ode.odeint_adjoint(y0, t5.to(dev))
        (out * go.to(dev)).sum().backward()
        torch.cuda.synchronize()
        return out.detach().cpu(), y0.grad.cpu(), [p.grad.cpu() for p in f_ex.parameters()], ode

    full = run_ks(u5, go5, None, B5)
    before = comm.collectives
    mine = run_ks(shard_batch(u5, rank, world).contiguous(), shard_batch(go5, rank, world, dim=1).contiguous(), comm,
                  B5 // world)
    assert "dense-mlp" in mine[3].path, mine[3].path
    assert mine[3]._cb_ex.record_layer_events
    assert comm.collectives - before >= len(mine[3]._cb_ex.lins), "mu was not all-reduced layer by layer"
    assert rel_err(mine[0], shard_batch(full[0], rank, world, dim=1)) < 1e-11
    assert rel_err(mine[1], shard_batch(full[1], rank, world)) < 1e-10
    for a, b in zip(mine[2], full[2]):
        assert rel_err(a, b) < 1e-10, rel_err(a, b)
    if rank == 0:
        print("KS pair sharded vs full batch: mu all-reduced in %d layer slices" % len(mine[3]._cb_ex.lins), flush=True)

    if comm.peer is not None:
        # the in-kernel all-reduce must be bit-identical on every rank and repeatable (epochs / double buffering)
        for rep in range(5):
            again = run(func, shard_batch(u0, rank, world).contiguous(), shard_batch(gout, rank, world, dim=1).contiguous(),
                        t, "rk4", 0.025, comm, ["-ts_adapt_type", "none"])
            flat = torch.cat([g.reshape(-1) for g in again[2]]).cuda()
            ref = flat.clone()
            dist.broadcast(ref, 0)
            assert torch.equal(flat, ref), "mu differs across ranks"
        assert comm.peer["epoch"] >= 6
    dist.barrier()
    if rank == 0:
        print("dp_check ok: world=%d collectives=%d peer=%s" % (world, comm.collectives, comm.peer is not None))
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
