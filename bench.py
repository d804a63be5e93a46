#!/usr/bin/env python
"""Benchmark of the hot path: one MNIST neural-ODE TRAINING step (forward adaptive Tsit5 solve
with the randomly-sampled local regulariser, classifier head + cross-entropy, continuous
adjoint + regulariser pullback, gradient all-reduce, Adam) on synthetic data.

    python bench.py --gpus N --steps K --warmup W            # this repo (libLRNDE.so)
    python bench.py --impl reference --gpus N --steps K ...  # CPU restatement of the reference
    python bench.py --steps K --dump-outputs DIR             # also write the last timed step's results as DIR/*.npy

The native arms load libLRNDE.so as `python -c 'import __graft_entry__ as g; g.build()'` left it and write
nothing into the tree.

Metric (BASELINE.json): MNIST neural-ODE train samples/s (+ NFE/s).  Workload: the
"mnist_ode batch-scaling sweep" config at 8192 samples per GPU (weak scaling: 8192 x N, i.e.
8192 ... 65536 over 1 ... 8 GPUs), reference tolerances abstol = reltol = 1.4e-8, :unbiased
:error_estimate regulariser, w_reg = 2.5 (experiments/mnist_ode/mlp.yml, SURVEY 8d).

The Julia reference cannot run here (no julia binary in the image), so `--impl reference` and
the `cpu_baseline` leg time the numpy oracle (oracle/, "port") on the host cores.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark runs from the tree build() left, which may be read-only: no __pycache__

D, H, NCLS = 784, 100, 10
TOL = 1.4e-8
W_REG = 2.5
LR = 1e-3
PHYS_TOL = 1.4e-8      # experiments/physionet/physionet.yml:8-9


def flops_per_feval(B):
    return 2.0 * B * (H * (D + 1) + D * (H + 1))          # SURVEY 8d


def iteration_flops(B, nfe_fwd, nf_bwd):
    """forward f-evals cost F_f, adjoint RHS evals ~3 F_f (recompute layer 1, two data GEMMs,
    two weight-gradient GEMMs; the W2*h product is skipped), regulariser pullback 6 x 3 F_f."""
    return flops_per_feval(B) * (nfe_fwd + 3.0 * nf_bwd + 18.0)


# ---------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, f"/tmp/lrnde_clocks_{os.getpid()}.csv"

    def start(self):
        if os.environ.get("LRNDE_NO_CLOCKS"):      # diagnostic: measure the sampler's own perturbation
            return
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=self.f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            p = [s.strip() for s in line.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm)}
        try:
            os.remove(self.path)
        except OSError:
            pass
        return out


# ---------------------------------------------------------------------------------- reference arm
def oracle_iteration(B, seed=0, reps=1):
    """One training iteration (fwd + head + adjoint + reg pullback) of the CPU restatement on a
    bounded sample of the workload.  Returns (seconds per iteration, nfe, nf_bwd)."""
    import oracle as orc
    om = orc.mnist_ode_model(D, H)
    rng = np.random.default_rng(seed)
    ps = orc.glorot_uniform_params(om, rng)
    Wc = (rng.uniform(-1, 1, (NCLS, D)) * np.sqrt(6.0 / (D + NCLS))).astype(np.float32)
    x = rng.random((D, B), dtype=np.float32)
    y = rng.integers(0, NCLS, B)
    node = orc.NeuralODE(om, regularize="unbiased", save_start=False, abstol=TOL, reltol=TOL, maxiters=10000)
    st = node.initialstates(np.random.default_rng(seed + 1))
    best, nfe, nfb = None, 0, 0
    for _ in range(reps):
        t0 = time.perf_counter()
        sol, st2, aux = node.forward(x, ps, st)
        u = sol.u[-1]
        z = Wc @ u
        z = z - z.max(0)
        sm = np.exp(z) / np.exp(z).sum(0)
        sm[y, np.arange(B)] -= 1
        d_u = (Wc.T @ (sm / B)).astype(np.float32)
        d_x, d_ps = node.backward(aux, [None, d_u], W_REG, ps)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
        nfe, nfb = st2["nfe"], aux["bsol"].nf
    return best, nfe, nfb


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    Bs = args.ref_batch
    for _ in range(max(args.warmup, 0) and 1):
        oracle_iteration(Bs)
    times = []
    nfe = nfb = 0
    for _ in range(max(1, args.steps)):
        dt, nfe, nfb = oracle_iteration(Bs)
        times.append(dt)
    ms = 1e3 * float(np.mean(times))
    val = Bs / (ms / 1e3)
    cores = os.cpu_count()
    sample = (f"{Bs} of the {args.batch}-sample per-GPU batch, same model/tolerances/regulariser; numpy "
              f"float32 oracle (CPU restatement of the reference, not Julia), BLAS threads = all {cores} cores")
    line = {
        "impl": "reference", "metric": "mnist_ode_train_samples_per_s", "value": val, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "nfe_per_s": nfe / (ms / 1e3),
        "config": workload_config(args, args.gpus),
        "sample": {"batch": Bs, "of_batch_per_gpu": args.batch,
                   "note": "every step of this arm is one training iteration on a bounded sample of the workload (the "
                           "full 8192-sample batch takes ~25 s per iteration in numpy); samples/s is size-normalised"},
        "cpu_baseline": {"value": val, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_config(args, n):
    return {"workload": "mnist_ode batch-scaling sweep (BASELINE configs[4]); TD-MLP 785=>100 tanh, 101=>784; "
                        "Tsit5 + :unbiased :error_estimate local reg; fwd + head + adjoint + Adam; the diffeqsol_to_array "
                        "layer after the functor is fused (only u(t2) crosses the C ABI)",
            "batch_per_gpu": args.batch, "global_batch": args.batch * n, "abstol": TOL, "reltol": TOL,
            "w_reg": W_REG, "precision": args.precision,
            "l2": "inputs larger than L2: every attempt streams the [D,B] state arrays (2-4 x 25.7 MB at 8192/GPU) and the "
                  "hidden tape (28 x 29 MB) from HBM; no flush needed"}


# ---------------------------------------------------------------------------------- this repo
DUMP_BYTES = 64 * 10**6     # cap on what --dump-outputs writes in all


def dump_outputs(path, outputs, per_sample):
    """Writes every entry of `outputs` as path/<name>.npy: tensors in float32, Python numbers as float64 scalars.  The
    arrays named in `per_sample` carry one row per sample; when everything together would exceed DUMP_BYTES, they are
    cut to a fixed seeded choice of rows (the same rows in every run with the same batch size)."""
    import torch
    arrs = {k: v.detach().float() if isinstance(v, torch.Tensor) else np.float64(v) for k, v in outputs.items()}
    fixed = 128 * len(arrs) + sum(4 * v.numel() if isinstance(v, torch.Tensor) else v.nbytes   # 128: .npy header
                                  for k, v in arrs.items() if k not in per_sample)
    n = arrs[per_sample[0]].shape[0]
    rows = min(n, (DUMP_BYTES - fixed) // sum(4 * arrs[k][0].numel() for k in per_sample))
    if rows < n:
        pick = torch.from_numpy(np.sort(np.random.default_rng(0).choice(n, rows, replace=False)))
        for k in per_sample:
            arrs[k] = arrs[k].index_select(0, pick.to(arrs[k].device))
    os.makedirs(path, exist_ok=True)
    for k, v in arrs.items():
        np.save(os.path.join(path, k + ".npy"), v.cpu().numpy() if isinstance(v, torch.Tensor) else v)


def _native_loop(pkg, torch, dist, args, B, world, rank, dev, ctx, steps, warmup, e2e_steps, keep_step=None):
    """The training iteration at batch B per GPU: returns (ms per step device-resident, ms per step through host
    buffers, info of the last step, kernel launches inside the timed region, nfe sum).  keep_step: index of the
    device-resident step whose results are returned under "outputs" (u(t2), gradients, updated parameters, loss)."""
    lib = pkg.lib()
    chk = pkg._lib.check
    chain = pkg.TDChain(pkg.Chain(pkg.Dense(D, H, "tanh"), pkg.Dense(H, D)))
    # return_last_only: the diffeqsol_to_array layer that follows the functor in the reference's classifier
    # (experiments/src/construct.jl:198) is fused, so only u(t2) crosses the boundary
    node = pkg.NeuralODE(chain, regularize="unbiased", save_start=False, abstol=TOL, reltol=TOL,
                         maxiters=10000, precision=args.precision, loop_mode=args.loop_mode, ctx=ctx,
                         return_last_only=True)
    P = pkg.nparams(chain)
    rng = np.random.default_rng(0)                       # same weights on every rank
    ps_h = node.initialparameters(rng)
    Wc_h = np.concatenate([((rng.uniform(-1, 1, (NCLS, D)) * np.sqrt(6.0 / (D + NCLS))).astype(np.float32)).ravel(order="F"),
                           np.zeros(NCLS, np.float32)])
    drng = np.random.default_rng(1000 + rank)             # different data per rank
    pin = lambda shape, dt=torch.float32: torch.empty(shape, dtype=dt).pin_memory()
    xb_h = pin((B, D))
    xb_h.numpy()[...] = drng.random((B, D), dtype=np.float32)
    y_hp = pin((B,), torch.int32)
    y_hp.numpy()[...] = drng.integers(0, NCLS, B).astype(np.int32)
    # e2e leg: two page-locked input buffers (same synthetic batch), so that batch i+1 is staged while step i computes
    xb_h2, y_hp2 = pin((B, D)), pin((B,), torch.int32)
    xb_h2.copy_(xb_h)
    y_hp2.copy_(y_hp)
    hbufs = [(xb_h, y_hp), (xb_h2, y_hp2)]
    st0 = node.initialstates(np.random.default_rng(7))    # same t1 stream on every rank

    ps = torch.from_numpy(ps_h).to(dev)
    Wc = torch.from_numpy(Wc_h).to(dev)
    xb = xb_h.to(dev)
    y = y_hp.to(dev)
    opt = {k: torch.zeros_like(v) for k, v in (("m_ps", ps), ("v_ps", ps), ("m_wc", Wc), ("v_wc", Wc))}
    d_u = torch.empty((B, D), dtype=torch.float32, device=dev)
    d_Wc = torch.empty_like(Wc)
    loss = C.c_float()
    launches = {"n": 0}
    info = {}
    kept = {}
    # host side of the e2e leg: page-locked buffers, as a host application (the Julia caller) would keep
    hb = {"ps": pin((P,)), "Wc": pin((Wc.numel(),)), "dps": pin((P,)), "dwc": pin((Wc.numel(),))}
    hb["ps"].copy_(ps)
    hb["Wc"].copy_(Wc)
    mh = ctx.model_handle(chain)
    Stats = pkg._lib.Stats

    def adam(i, gp, gw):
        if world > 1:                # parameter gradients: one all-reduce per iteration, inside the library
            chk(lib.lrnde_allreduce_sum(ctx._h, gp.data_ptr(), gp.numel()))
            chk(lib.lrnde_allreduce_sum(ctx._h, gw.data_ptr(), gw.numel()))
        chk(lib.lrnde_adam_step(ctx._h, ps.data_ptr(), gp.data_ptr(), opt["m_ps"].data_ptr(),
                                opt["v_ps"].data_ptr(), P, LR, 0.9, 0.999, 1e-8, i + 1))
        chk(lib.lrnde_adam_step(ctx._h, Wc.data_ptr(), gw.data_ptr(), opt["m_wc"].data_ptr(),
                                opt["v_wc"].data_ptr(), Wc.numel(), LR, 0.9, 0.999, 1e-8, i + 1))

    def step(i, st, resident=True):
        """One training iteration.  resident=True: device pointers, layer by layer; False: HOST buffers through
        the C ABI (lrnde_classifier_grad: the e2e leg)."""
        if resident:
            sol, st2 = node(xb.t(), ps, st)
            u_last = sol.u[-1].t()                           # (B, D) contiguous block of u_save
            chk(lib.lrnde_head_ce(ctx._h, Wc.data_ptr(), u_last.data_ptr(), y.data_ptr(), B, D, NCLS, 0,
                                  C.byref(loss), d_u.data_ptr(), d_Wc.data_ptr()))
            if world > 1:            # global-mean loss: lambda(t2) = dL/du carries 1 / world
                d_u.mul_(1.0 / world)
                d_Wc.mul_(1.0 / world)
            d_x, d_ps = node.backward(sol, [d_u.t()], W_REG)
            launches["n"] += sol.stats.gpu_launches + sol.bwd_stats.gpu_launches + 6
            adam(i, d_ps, d_Wc)
            fs, bs = sol.stats, sol.bwd_stats
            nfe, reg, retcode = st2["nfe"], float(st2["reg_val"]), sol.retcode
            if i == keep_step:       # u_last, d_x and d_ps are fresh per step; d_Wc, ps and Wc are rewritten in place
                kept.update(u_final=u_last, d_x=d_x.t(), d_ps=d_ps, d_wc=d_Wc.clone(), ps=ps.clone(), wc=Wc.clone(),
                            loss=float(loss.value), reg_val=reg, nfe=float(nfe))
            sol.free()
        else:
            # t1 is host-sampled exactly as the layer functor does (neural_ode.jl:69-71)
            o, _ = node._opts("unbiased", 0.0, 0.0, True, True)
            import copy
            rng2 = copy.deepcopy(st["rng"])
            o.t1 = float(np.float32(rng2.random(dtype=np.float32)))
            stats = Stats()
            xc, yc = hbufs[i % 2]
            xn, yn = hbufs[(i + 1) % 2]
            # input pipeline: the next batch goes host -> device on the library's copy stream while this step computes
            chk(lib.lrnde_prefetch_inputs(ctx._h, xn.data_ptr(), yn.data_ptr(), B, D))
            chk(lib.lrnde_classifier_grad(ctx._h, mh, C.byref(o), hb["ps"].data_ptr(), hb["Wc"].data_ptr(),
                                          xc.data_ptr(), yc.data_ptr(), B, NCLS, W_REG, 1.0 / world, C.byref(loss),
                                          hb["dps"].data_ptr(), hb["dwc"].data_ptr(), C.byref(stats)))
            gp = hb["dps"].to(dev, non_blocking=True)
            gw = hb["dwc"].to(dev, non_blocking=True)
            adam(i, gp, gw)
            hb["ps"].copy_(ps, non_blocking=True)            # the updated parameters back to the host application
            hb["Wc"].copy_(Wc, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
            fs = bs = stats
            nfe, reg, retcode = stats.nfe, float(stats.reg_val), pkg._lib.RETCODES.get(stats.retcode, "?")
            st2 = dict(st, rng=rng2, nfe=nfe, reg_val=np.float32(reg))
        info.update(nfe=nfe, nf_bwd=bs.nf_bwd, reg=reg, naccept=fs.naccept, nreject=fs.nreject,
                    nacc_b=bs.naccept_bwd, nrej_b=bs.nreject_bwd, loss=float(loss.value) + W_REG * reg, retcode=retcode,
                    phases_us=dict(fwd_solve=fs.reserved[0], saves=fs.reserved[1], reg_step=fs.reserved[2],
                                   adjoint=bs.reserved[3], reg_pullback=bs.reserved[4], fwd_setup=fs.reserved[5]))
        return st2

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def timed(nsteps, st, resident, i0):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(nsteps)]
        sync_all()
        e0.record()
        nfe_sum = 0
        for i in range(nsteps):
            st = step(i0 + i, st, resident)
            nfe_sum += info["nfe"]
            marks[i].record()
        e1.record()
        sync_all()
        ms = e0.elapsed_time(e1)
        prev = e0
        per_step = []
        for m in marks:
            per_step.append(round(prev.elapsed_time(m), 3))
            prev = m
        info["per_step_ms"] = per_step
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, st, nfe_sum

    import copy
    # buffers of the state snapshot taken at the start of the timed region (allocated before the warm-up so that the
    # timed steps see a settled allocator)
    snap = dict(ps=torch.empty_like(ps), Wc=torch.empty_like(Wc), opt={k: torch.empty_like(v) for k, v in opt.items()}, st=None)
    st = st0
    for i in range(warmup):
        st = step(i, st, True)
    launches["n"] = 0
    # the e2e leg below repeats exactly these iterations (same parameters, optimiser state and t1 stream), so that the
    # two legs take the same solver steps and differ only in where the buffers live
    for k, v in (("ps", ps), ("Wc", Wc)):
        snap[k].copy_(v)
    for k, v in opt.items():
        snap["opt"][k].copy_(v)
    snap["st"] = copy.deepcopy(st)

    def restore():
        ps.copy_(snap["ps"])
        Wc.copy_(snap["Wc"])
        for k, v in opt.items():
            v.copy_(snap["opt"][k])
        hb["ps"].copy_(ps)
        hb["Wc"].copy_(Wc)
        torch.cuda.synchronize(dev)
        return copy.deepcopy(snap["st"])

    ms_total, st, nfe_sum = timed(steps, st, True, warmup)
    n_launch = launches["n"]
    fwd_info = dict(info)
    per_step_ms = list(info.get("per_step_ms", []))
    ms_e = float("nan")
    if e2e_steps:
        i_w = warmup - 1 if warmup > 0 else 1
        chk(lib.lrnde_prefetch_inputs(ctx._h, hbufs[i_w % 2][0].data_ptr(), hbufs[i_w % 2][1].data_ptr(), B, D))   # batch of the warm step
        step(i_w, restore(), False)                         # warm (leaves the batch of iteration `warmup` staged)
        ms_e, _, _ = timed(e2e_steps, restore(), False, warmup)
        ms_e /= e2e_steps
    e2e_info = dict(info) if e2e_steps else {}
    PW = NCLS * D + NCLS
    h2d = 4 * (B * D + B + P + PW) + 4 * (P + PW)            # x, labels, ps, Wc in; the host gradients back up for the optimiser
    d2h = 4 * (P + PW + 1) + 4 * (P + PW)                    # d_ps, d_Wc, loss out; the updated parameters
    return dict(ms=ms_total / steps, ms_total=ms_total, ms_e2e=ms_e, info=fwd_info, e2e_info=e2e_info, launches=n_launch, nfe_sum=nfe_sum,
                per_step_ms=per_step_ms, outputs=kept,
                h2d=h2d, d2h=d2h, node=node, chain=chain, ps=ps, xb=xb, P=P)


def run_native(args):
    import torch
    import __graft_entry__ as entry
    pkg = entry.load_package()
    lib = pkg.lib()
    chk = pkg._lib.check

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)     # barrier + max-over-ranks of the timings only

    if args.scaling == "strong":
        if args.global_batch % world:
            raise SystemExit("--global-batch must be divisible by the number of GPUs")
        args.batch = args.global_batch // world
    B = args.batch
    ctx = pkg.Context(local, torch.cuda.current_stream(dev).cuda_stream)
    if world > 1:
        def gather(blob):
            out = [None] * world
            dist.all_gather_object(out, blob)
            return out
        ctx.setup_group(rank, world, B * world, gather)

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()         # before the warm-up: nvidia-smi's own start-up (~1 s of driver calls) must not
                               # land inside the timed region; it keeps sampling every 200 ms through it
    e2e_steps = max(0, min(args.steps, args.e2e_steps))
    try:
        r = _native_loop(pkg, torch, dist, args, B, world, rank, dev, ctx, args.steps, args.warmup, e2e_steps,
                         keep_step=args.warmup + args.steps - 1 if args.dump_outputs else None)
    finally:                   # the nvidia-smi sampler must not outlive a failed run
        clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, r["outputs"], per_sample=("u_final", "d_x"))
    ms, ms_e, fwd_info = r["ms"], r["ms_e2e"], r["info"]
    value = B * world / (ms / 1e3)
    e2e = {"value": B * world / (ms_e / 1e3), "unit": "samples/s", "h2d_bytes_per_step": r["h2d"],
           "d2h_bytes_per_step": r["d2h"], "ms_per_step": ms_e, "steps": e2e_steps,
           "last_step": {k: r["e2e_info"].get(k) for k in ("naccept", "nacc_b", "nfe", "phases_us")},
           "call": "lrnde_classifier_grad with host buffers (x, labels, ps, Wc in; loss, d_ps, d_Wc out) + gradient "
                   "all-reduce + Adam; pinned host memory; every step also issues lrnde_prefetch_inputs for the next batch "
                   "(one x + labels host-to-device copy per step, on the library's copy stream, overlapped with the step)"}

    # ---- roofline (SURVEY 8d): one Tsit5 attempt of the forward solve and of the adjoint solve, timed live with
    # CUDA events on the library's stream (lrnde_profile_step / LRNDE_PROFILE_ADJ hook), against the algorithmic
    # work of the reference's step: forward 6 F_f flop and 9 * 4 * D * B bytes (read u_n, k1; write k2..k7, u_{n+1});
    # adjoint 18 F_f flop and (8 + 2 * 7) * 4 * D * B + 2 * 7 * 4 * P bytes.
    node, chain, ps, xb, P = r["node"], r["chain"], r["ps"], r["xb"], r["P"]
    peaks = {}
    pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk_path):
        peaks = json.load(open(pk_path))
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    tf32_peak = peaks.get("bf16_tflops", 1590.0) / 2.0
    o, _k = node._opts("none", 0.0, 0.0, True, False)          # keep_tape: the training configuration of the engine
    us = (C.c_float * 3)()
    chk(lib.lrnde_profile_step(ctx._h, ctx.model_handle(chain), C.byref(o), ps.data_ptr(), xb.data_ptr(), B, 20, us))
    # the adjoint attempt: one more backward with the event hook switched on
    ua = (C.c_float * 5)()
    if world == 1:     # (in a group the repeated attempts would replay the mu exchange out of sequence)
        os.environ["LRNDE_PROFILE_ADJ"] = "20"
        sol, _st = node(xb.t(), ps, node.initialstates(np.random.default_rng(7)))
        node.backward(sol, [torch.full((B, D), 1.0 / B, device=dev).t()], W_REG)
        sol.free()
        os.environ.pop("LRNDE_PROFILE_ADJ", None)
        chk(lib.lrnde_profile_adjoint_last(ua))
    Ff = flops_per_feval(B)
    arr = 4.0 * D * B
    Kaug = H + 2
    fwd_t, adj_t = us[2] * 1e-6, (ua[4] * 1e-6 if ua[4] > 0 else float("nan"))
    fwd_bytes, fwd_flops = 9.0 * arr, 6.0 * Ff
    adj_bytes, adj_flops = 22.0 * arr + 14.0 * 4.0 * P, 18.0 * Ff
    # DRAM bytes per launch from the committed ncu --set full captures of this build at 8192 samples
    # (profiles/r2_traffic.json, made by scratch/ncu_traffic.py from profiles/r2_*_ncu_full.txt's reports):
    # the forward attempt = chain_kernel + kgemm_kernel<2,0> (lean tape)
    traffic, traffic_detail = None, None
    tr_path = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if os.path.exists(tr_path) and B == 8192:
        kt = json.load(open(tr_path))
        get = lambda name: next((v["dram_bytes_per_launch"] for k, v in kt.items() if name in k), None)
        parts = {n: get(n) for n in ("chain_kernel<1>", "kgemm_kernel<2, 0>", "adj_chain_kernel", "pairacc_kernel",
                                     "adj_reduce_kernel", "adj_mu_kernel")}
        if parts["chain_kernel<1>"] and parts["kgemm_kernel<2, 0>"]:
            traffic = parts["chain_kernel<1>"] + parts["kgemm_kernel<2, 0>"]
        traffic_detail = {"source": "profiles/r2_traffic.json (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch)",
                          "per_kernel": parts}
    # per-kernel figures with the bytes each launch really has to move in this design
    zarr = 4.0 * 128 * B                                         # one hidden-space array [B][128]
    kern = {
        "fused::chain_kernel (forward stages in hidden space)": dict(us=us[0], bytes=(2 + 7 + 7 + 1) * zarr,
                                                                    flops=6 * 2.0 * H * Kaug * B),
        "fused::kgemm_kernel<6,0> (k_2..k_7 = W2a h, u_{n+1}, residual; lean tape)": dict(
            us=us[1], bytes=4 * arr + 6 * 2 * 4.0 * 104 * B, flops=6 * 2.0 * D * Kaug * B),
        "ladj::adj_chain_kernel (adjoint stages in hidden space)": dict(us=ua[0], bytes=(48 + 4 * 6 + 6 + 12) * zarr,
                                                                        flops=6 * 2 * 2.0 * H * Kaug * B),
        "fused::kgemm_kernel<2,1> (lambda_{n+1} = lambda_n - dt W1^T Delta, residual)": dict(
            us=ua[1], bytes=2 * arr + 2 * 2 * 4.0 * 104 * B, flops=2 * 2.0 * D * H * B),
        "ladj::pairacc_kernel (batch contractions of the mu block)": dict(
            us=ua[2], bytes=2 * arr + 26 * zarr + 2 * 7 * 2 * zarr, flops=(13 * 2 + 2 * 7 * 2) * 2.0 * 128 * 128 * B),
        "ladj::adj_reduce_kernel + adj_mu_kernel": dict(us=ua[3], bytes=26e6, flops=4 * 2.0 * H * Kaug * D),
    }
    for k, v in kern.items():
        t = v["us"] * 1e-6
        v["hbm_frac"] = (v["bytes"] / t / 1e9 / hbm_peak) if t > 0 else None
        v["tensor_frac_3xtf32"] = (3.0 * v["flops"] / t / 1e12 / tf32_peak) if t > 0 else None
        v["us"] = round(v["us"], 2)
    hbm_frac, ten_frac = fwd_bytes / fwd_t / 1e9 / hbm_peak, fwd_flops / fwd_t / 1e12 / tf32_peak
    bound = "hbm" if hbm_frac >= ten_frac else "tensor"
    roof = {"bound": bound,
            "kernel": "one Tsit5 attempt of the forward solve (fused::chain_kernel + fused::kgemm_kernel), timed with CUDA "
                      "events; algorithmic work of SURVEY 8(d): 6 F_f flop, 9 * 4 * D * B bytes",
            "achieved": (fwd_bytes / fwd_t / 1e9) if bound == "hbm" else fwd_flops / fwd_t / 1e12,
            "peak": hbm_peak if bound == "hbm" else tf32_peak, "unit": "GB/s" if bound == "hbm" else "TFLOP/s",
            "frac": max(hbm_frac, ten_frac), "traffic": traffic, "traffic_detail": traffic_detail,
            "peak_source": ("MEASURED_PEAKS.json (STREAM copy; bf16 burst / 2 = TF32 dense)" if peaks else "fallback"),
            "forward_step": {"us": round(us[2], 2), "us_solve_loop": round(fwd_info["phases_us"]["fwd_solve"] /
                                                                        max(1, fwd_info["naccept"] + fwd_info["nreject"]), 2),
                             "algorithmic_bytes": fwd_bytes, "algorithmic_flops": fwd_flops, "hbm_frac": hbm_frac,
                             "tensor_frac": ten_frac},
            "adjoint_step": (None if not ua[4] > 0 else
                             {"us": round(ua[4], 2), "algorithmic_bytes": adj_bytes, "algorithmic_flops": adj_flops,
                              "hbm_frac": adj_bytes / adj_t / 1e9 / hbm_peak, "tensor_frac": adj_flops / adj_t / 1e12 / tf32_peak}),
            "iteration_tensor_frac": iteration_flops(B, fwd_info["nfe"], fwd_info["nf_bwd"]) / (ms * 1e-3) / 1e12 / tf32_peak,
            "kernels": kern}

    # ---- BASELINE configs[0]: the reference's own shape (batch 128), same iteration, measured in the same run
    secondary = None
    if world == 1 and not args.no_secondary and B != 128:
        r2 = _native_loop(pkg, torch, dist, args, 128, 1, 0, dev, ctx, max(5, args.steps), 3, 3)
        i2 = r2["info"]
        secondary = {"mnist_ode_b128": {
            "workload": "BASELINE configs[0]: mnist_ode batch 128 (the reference's own shape), same iteration",
            "value": 128 / (r2["ms"] / 1e3), "unit": "samples/s", "ms_per_step": r2["ms"],
            "e2e_value": 128 / (r2["ms_e2e"] / 1e3), "e2e_ms_per_step": r2["ms_e2e"],
            "steps_fwd": [i2["naccept"], i2["nreject"]], "steps_bwd": [i2["nacc_b"], i2["nrej_b"]],
            "nfe_per_step": i2["nfe"], "phases_us": i2["phases_us"], "gpu_launches_per_step": r2["launches"] / max(5, args.steps)}}

    # ---- BASELINE configs[3]: the cifar10 node core at batch 256 (tensor-core conv engine), measured in the same run
    if secondary is not None:
        try:
            secondary["cifar10_b256"] = cifar10_secondary(torch, dev)
        except Exception as exc:   # the headline line must not depend on the secondary workload
            secondary["cifar10_b256"] = {"error": repr(exc)[:200]}

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            Bs = args.ref_batch
            dt, nfe_c, nfb_c = oracle_iteration(Bs)
            cpu = {"value": Bs / dt, "unit": "samples/s", "cores": os.cpu_count(), "kind": "port",
                   "sample": f"1 iteration on {Bs} of the {B} samples ({dt:.1f} s), numpy float32 oracle, all host cores via BLAS",
                   "nfe": int(nfe_c)}
        line = {
            "metric": "mnist_ode_train_samples_per_s", "value": value, "unit": "samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "per_step_ms": r["per_step_ms"], "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32" if args.precision == "fp32" else "tf32x3",
            "data": "synthetic", "config": workload_config(args, world),
            "parity_regime": "noise (abstol = reltol = 1.4e-8 sits below Float32 resolution: the embedded error estimate "
                             "is rounding-dominated, step sequences of two Float32 implementations agree statistically; "
                             "strict step-sequence parity is asserted on the truncation-dominated fixtures of tests/)",
            "nfe_per_s": r["nfe_sum"] / (r["ms_total"] / 1e3) * world, "nfe_per_step": fwd_info["nfe"],
            "nf_bwd_per_step": fwd_info["nf_bwd"], "steps_fwd": [fwd_info["naccept"], fwd_info["nreject"]],
            "steps_bwd": [fwd_info["nacc_b"], fwd_info["nrej_b"]], "loss": fwd_info["loss"],
            "retcode": fwd_info["retcode"], "phases_us": fwd_info["phases_us"],
            "e2e": e2e, "gpu_launches": int(r["launches"]), "clocks": clk, "roofline": roof, "cpu_baseline": cpu,
            "secondary": secondary,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------- mnist_sde (secondary)
def sde_setup(B, use_oracle):
    Ds, Hs = 32, 64
    kw = dict(regularize="unbiased", abstol=0.14, reltol=0.14, save_start=False, maxiters=10000, seed=0)
    rng = np.random.default_rng(0)
    if use_oracle:
        import oracle as orc
        od = orc.MLP([orc.Dense(Ds, Hs, "tanh"), orc.Dense(Hs, Ds, "identity")], time_dependent=False)
        og = orc.MLP([orc.Dense(Ds, Ds, "identity")], time_dependent=False)
        layer = orc.NeuralDSDE(od, og, **kw)
        ps = np.concatenate([orc.glorot_uniform_params(od, rng), orc.glorot_uniform_params(og, rng)])
    else:
        import __graft_entry__ as entry
        pkg = entry.load_package()
        layer = pkg.NeuralDSDE(pkg.Chain(pkg.Dense(Ds, Hs, "tanh"), pkg.Dense(Hs, Ds)), pkg.Chain(pkg.Dense(Ds, Ds)), **kw)
        ps = layer.initialparameters(rng)
    x = np.random.default_rng(1).random((Ds, B), dtype=np.float32)
    return layer, ps, x


def run_sde(args):
    """BASELINE configs[1]: neural SDE (diagonal noise) with local regularisation, state 32 x 128
    (experiments/src/construct.jl:202-210): forward SOSRI solve + regulariser step + TrackerAdjoint
    pullback of sum(u(t2))/B + w_reg * reg_val.  Secondary workload (one JSON line, same contract)."""
    B = args.sde_batch
    if args.impl == "reference":
        layer, ps, x = sde_setup(B, True)
        st = layer.initialstates(np.random.default_rng(7))
        ts = []
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            out, st2, aux = layer.forward(x, ps, st)
            layer.backward(aux, [None, np.ones_like(x) / B], W_REG, ps)
            if i >= args.warmup:
                ts.append(time.perf_counter() - t0)
        ms = 1e3 * float(np.mean(ts))
        val = B / (ms / 1e3)
        print(json.dumps({"impl": "reference", "metric": "mnist_sde_train_samples_per_s", "value": val, "unit": "samples/s",
                          "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": {"workload": "mnist_sde (BASELINE configs[1])", "batch": B},
                          "cpu_baseline": {"value": val, "unit": "samples/s", "cores": os.cpu_count(), "kind": "port",
                                           "sample": "the whole workload"},
                          "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    import torch
    layer, ps, x = sde_setup(B, False)
    dev = torch.device("cuda", 0)
    xt, pt = torch.from_numpy(x).to(dev), torch.from_numpy(ps).to(dev)
    cot_t = torch.ones((32, B), device=dev) / B
    cot_h = np.ones((32, B), np.float32) / B
    st = layer.initialstates(np.random.default_rng(7))
    info = {}

    def step(resident):
        sol, st2 = layer(xt if resident else x, pt if resident else ps, st)
        layer.backward(sol, [None, cot_t if resident else cot_h], W_REG)
        info.update(nfe=st2["nfe_drift"], acc=sol.stats.naccept, rej=sol.stats.nreject, launches=sol.stats.gpu_launches + 3)
        sol.free()

    def timed(n, resident):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(n):
            step(resident)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n
    clocks = ClockSampler(0)
    clocks.start()
    for _ in range(max(3, args.warmup) + 20):
        step(True); step(False)
    ms = timed(args.steps, True)
    clk = clocks.stop()
    ms_e = timed(args.steps, False)
    olayer, ops, ox = sde_setup(B, True)
    ost = olayer.initialstates(np.random.default_rng(7))
    t0 = time.perf_counter()
    out, st2, aux = olayer.forward(ox, ops, ost)
    olayer.backward(aux, [None, cot_h], W_REG, ops)
    dt = time.perf_counter() - t0
    print(json.dumps({"metric": "mnist_sde_train_samples_per_s", "value": B / (ms / 1e3), "unit": "samples/s", "n_gpus": 1,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                      "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": {"workload": "mnist_sde (BASELINE configs[1]): NeuralDSDE drift 32-64-32 tanh, diffusion "
                                             "Dense(32=>32), SOSRI + RSwM3, :unbiased local reg, tol 0.14; fwd + TrackerAdjoint",
                                 "batch": B, "l2": "working set 16 KB per array: cache resident by construction"},
                      "nfe_per_step": info["nfe"], "steps_fwd": [info["acc"], info["rej"]],
                      "e2e": {"value": B / (ms_e / 1e3), "unit": "samples/s", "ms_per_step": ms_e,
                              "h2d_bytes_per_step": 4 * (32 * B * 2 + ps.size), "d2h_bytes_per_step": 4 * (32 * B * 3 + ps.size)},
                      "gpu_launches": int(info["launches"] * args.steps), "clocks": clk,
                      "roofline": {"bound": "latency", "kernel": "sde_solve_kernel (persistent cooperative kernel, one grid.sync "
                                   "per attempt)", "achieved": None, "peak": None, "unit": None, "frac": None, "traffic": None,
                                   "us_per_attempt": 1e3 * ms / max(1, info["acc"] + info["rej"])},
                      "cpu_baseline": {"value": B / dt, "unit": "samples/s", "cores": os.cpu_count(), "kind": "port",
                                       "sample": f"the whole workload, 1 iteration ({dt:.2f} s), numpy float32 oracle"}}))


# ---------------------------------------------------------------------------------- physionet (secondary)
def physionet_setup(B, T):
    in_dim, Hh, Lg, Nn = 37, 40, 50, 20                     # experiments/src/config.jl:31-34
    rng = np.random.default_rng(8)
    mask = (rng.random((in_dim, T, B)) < 0.2).astype(np.float32)
    mask[0, 0, :] = 1
    data = rng.standard_normal((in_dim, T, B)).astype(np.float32) * mask
    dt = np.zeros((1, T, B), np.float32)
    dt[0, 1:, :] = np.diff(np.sort(rng.random((T, B)), axis=0), axis=0)
    x = np.concatenate([data, mask, dt], axis=0)
    ts = np.sort(np.concatenate([[0.0], rng.uniform(0.02, 1.0, T - 1)])).astype(np.float32)
    return dict(in_dim=in_dim, H=Hh, Lg=Lg, Nn=Nn, x=x, data=data, mask=mask, ts=ts, rng=rng,
                dyn=[(Nn, Hh, "tanh"), (Hh, Nn, "tanh")] * 4,
                kw=dict(regularize="unbiased", abstol=PHYS_TOL, reltol=PHYS_TOL, maxiters=10000, saveat=list(ts)))


def run_physionet(args):
    """BASELINE configs[2]: latent ODE (GRU encoder + ODE decoder), 37 features, irregular series, batch 256;
    one training iteration = encoder -> rec_to_gen -> reparameterise -> NeuralODE (saveat = T observation times,
    :unbiased local reg) -> gen_to_data -> loss, and the whole reverse pass.  Secondary workload."""
    B, T = args.phys_batch, args.phys_T
    S = physionet_setup(B, T)
    w_reg, w_kl = 0.5, 0.1
    import oracle as orc
    from oracle.lrnde_latent_oracle import _net_fwd, _net_vjp
    rng = S["rng"]
    F = 2 * S["in_dim"] + 1
    ps_gru = orc.gru_init(rng, F, S["H"], S["Lg"])
    om = orc.MLP([orc.Dense(*l) for l in S["dyn"]], time_dependent=False, input_act="tanh")
    ps_node = (orc.glorot_uniform_params(om, rng) * 2).astype(np.float32)

    def chain_ps(dims):
        out = []
        for (i, o) in dims:
            a = np.sqrt(6.0 / (i + o))
            out += [rng.uniform(-a, a, (o, i)).astype(np.float32).ravel(order="F"), np.zeros(o, np.float32)]
        return np.concatenate(out)
    ps_r2g, ps_g2d = chain_ps([(2 * S["Lg"], S["Lg"]), (S["Lg"], 2 * S["Nn"])]), chain_ps([(S["Nn"], S["in_dim"])])

    def oracle_iter():
        def layers(ps, dims):
            out, off = [], 0
            for (i, o, a) in dims:
                W = ps[off:off + o * i].reshape((o, i), order="F"); wo = off; off += o * i
                b = ps[off:off + o]; bo = off; off += o
                out.append((W, b, a, wo, bo))
            return out
        x, data, mask = S["x"], S["data"], S["mask"]
        h, car = orc.gru_recurrence(ps_gru, x, F, S["H"], S["Lg"])
        Lr = layers(ps_r2g, [(2 * S["Lg"], S["Lg"], "tanh"), (S["Lg"], 2 * S["Nn"], "identity")])
        Ld = layers(ps_g2d, [(S["Nn"], S["in_dim"], "identity")])
        z = _net_fwd(Lr, h)
        eps = orc.philox_normal(13, 2, 0, S["Nn"] * B).reshape((S["Nn"], B), order="F")
        y0, mu, ls = orc.reparameterize(z, eps, True)
        on = orc.NeuralODE(om, **S["kw"])
        sol, st, aux = on.forward(y0, ps_node, on.initialstates(np.random.default_rng(2)))
        ser = np.stack(sol.u, axis=1)
        pred = _net_fwd(Ld, ser.reshape(S["Nn"], -1, order="F")).reshape((S["in_dim"], T, B), order="F")
        msum = mask.sum(axis=(0, 1))
        dpred = ((pred * mask - data * mask) * mask / 1e-4 / msum / B).astype(np.float32)
        g = np.zeros_like(ps_g2d)
        dser = _net_vjp(Ld, ser.reshape(S["Nn"], -1, order="F"), dpred.reshape(S["in_dim"], -1, order="F"), g).reshape(ser.shape, order="F")
        dy0, _ = on.backward(aux, [dser[:, i, :] for i in range(T)], w_reg, ps_node)
        dz = np.concatenate([dy0 + w_kl * mu / (S["Nn"] * B), dy0 * eps * np.exp(ls / 2) / 2 + w_kl * (np.exp(ls) - 1) / (2 * S["Nn"] * B)]).astype(np.float32)
        g2 = np.zeros_like(ps_r2g)
        dh = _net_vjp(Lr, h, dz, g2)
        orc.gru_recurrence_backward(ps_gru, x, F, S["H"], S["Lg"], car, dh)
        return st["nfe"]

    if args.impl == "reference":
        ts_ = []
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter(); oracle_iter()
            if i >= args.warmup:
                ts_.append(time.perf_counter() - t0)
        ms = 1e3 * float(np.mean(ts_)); val = B / (ms / 1e3)
        print(json.dumps({"impl": "reference", "metric": "physionet_train_samples_per_s", "value": val, "unit": "samples/s",
                          "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": {"workload": "physionet latent ODE (BASELINE configs[2])", "batch": B, "T": T},
                          "cpu_baseline": {"value": val, "unit": "samples/s", "cores": os.cpu_count(), "kind": "port", "sample": "the whole workload"},
                          "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    import torch
    import __graft_entry__ as entry
    pkg = entry.load_package()
    dev = torch.device("cuda", 0)
    cell = pkg.LatentGRUCell(S["in_dim"], S["H"], S["Lg"])
    rec = pkg.Recurrence(cell)
    r2g = pkg.Chain(pkg.Dense(2 * S["Lg"], S["Lg"], "tanh"), pkg.Dense(S["Lg"], 2 * S["Nn"]))
    g2d = pkg.Chain(pkg.Dense(S["Nn"], S["in_dim"]))
    node = pkg.NeuralODE(pkg.Chain(*[pkg.Dense(*l) for l in S["dyn"]], input_activation="tanh"),
                         precision=args.precision, **S["kw"])
    rp = pkg.ReparameterizeLayer(seed=13)
    to = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    dv = dict(x=to(S["x"]), data=to(S["data"]), mask=to(S["mask"]), gru=to(ps_gru), r2g=to(ps_r2g), g2d=to(ps_g2d), node=to(ps_node))
    hv = dict(x=S["x"], data=S["data"], mask=S["mask"], gru=ps_gru, r2g=ps_r2g, g2d=ps_g2d, node=ps_node)
    info = {}

    def step(resident):
        v = dv if resident else hv
        h, st_rec = rec(v["x"], v["gru"])
        z = pkg.mlp_forward(r2g, v["r2g"], h)
        y0, st_rp = rp(z, None, dict(training=True))
        y0c = y0.contiguous() if resident else np.ascontiguousarray(y0)
        sol, st_node = node(y0c, v["node"], node.initialstates(np.random.default_rng(2)))
        ser = pkg.diffeqsol_to_timeseries(sol)
        pred = pkg.mlp_forward(g2d, v["g2d"], ser)
        loss, nll, kl, d_pred, d_mu, d_ls = pkg.latent_loss(pred, v["data"], v["mask"], st_rp["mu0"], st_rp["logsigma2"], w_kl)
        d_ser, d_g2d = pkg.mlp_backward(g2d, v["g2d"], ser, d_pred)
        cots = [d_ser[:, i, :].contiguous() if resident else np.ascontiguousarray(d_ser[:, i, :]) for i in range(T)]
        d_y0, d_node = node.backward(sol, cots, w_reg)
        d_z = rp.backward(z, d_y0, d_mu, d_ls)
        d_h, d_r2g = pkg.mlp_backward(r2g, v["r2g"], h, d_z)
        rec.backward(st_rec, d_h)
        info.update(nfe=st_node["nfe"], loss=loss + w_reg * float(st_node["reg_val"]),
                    launches=sol.stats.gpu_launches + sol.bwd_stats.gpu_launches + 16,
                    phases_us=dict(fwd_solve=sol.stats.reserved[0], saves=sol.stats.reserved[1], reg_step=sol.stats.reserved[2],
                                   adjoint=sol.bwd_stats.reserved[3], reg_pullback=sol.bwd_stats.reserved[4],
                                   fwd_setup=sol.stats.reserved[5], bwd_setup=sol.bwd_stats.reserved[5]),
                    steps_bwd=[sol.bwd_stats.naccept_bwd, sol.bwd_stats.nreject_bwd], nf_bwd=sol.bwd_stats.nf_bwd)
        rec.free(st_rec); sol.free()

    def timed(n, resident):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record()
        for _ in range(n):
            step(resident)
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n
    clocks = ClockSampler(0)
    clocks.start()
    for _ in range(max(3, args.warmup)):
        step(True); step(False)
    ms = timed(args.steps, True)
    clk = clocks.stop()
    ms_e = timed(args.steps, False)
    t0 = time.perf_counter(); nfe_o = oracle_iter(); dt = time.perf_counter() - t0
    print(json.dumps({"metric": "physionet_train_samples_per_s", "value": B / (ms / 1e3), "unit": "samples/s", "n_gpus": 1,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                      "vs_baseline": None, "dtype": "tf32x3", "data": "synthetic",
                      "config": {"workload": "physionet latent ODE (BASELINE configs[2]): GRU encoder 37/40/50, ODE decoder 8 x Dense(20<->40, tanh), "
                                             "saveat at T irregular times, :unbiased local reg; fwd + full reverse pass", "batch": B, "T": T,
                                 "l2": "working set a few MB: cache resident by construction"},
                      "nfe_per_step": info["nfe"], "loss": info["loss"], "phases_us": info["phases_us"],
                      "steps_bwd": info["steps_bwd"], "nf_bwd_per_step": info["nf_bwd"],
                      "e2e": {"value": B / (ms_e / 1e3), "unit": "samples/s", "ms_per_step": ms_e,
                              "h2d_bytes_per_step": int(4 * (S["x"].size * 3 + ps_gru.size + ps_node.size)), "d2h_bytes_per_step": int(4 * (S["Nn"] * T * B * 3))},
                      "gpu_launches": int(info["launches"] * args.steps), "clocks": clk,
                      "roofline": {"bound": "latency", "kernel": "adjoint solve with T lambda jumps (tiny state 20 x B): launch / latency bound",
                                   "achieved": None, "peak": None, "unit": None, "frac": None, "traffic": None},
                      "cpu_baseline": {"value": B / dt, "unit": "samples/s", "cores": os.cpu_count(), "kind": "port",
                                       "sample": f"the whole workload, 1 iteration ({dt:.2f} s), numpy float32 oracle", "nfe": int(nfe_o)}}))


# ---------------------------------------------------------------------------------- cifar10 node core (secondary)
def measured_peaks():
    pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peaks = json.load(open(pk_path)) if os.path.exists(pk_path) else {}
    return {"hbm": peaks.get("hbm_gbs", 6650.0), "bf16_burst": peaks.get("bf16_tflops", 1590.0),
            "source": "MEASURED_PEAKS.json" if peaks else "fallback of B200_PROFILING.md"}


def cifar10_setup(B, use_oracle, W=32, loop_mode=0):
    kw = dict(regularize="unbiased", abstol=1e-4, reltol=1e-4, save_start=False, maxiters=10000)
    rng = np.random.default_rng(0)
    if use_oracle:
        import oracle as orc
        from oracle.lrnde_conv_oracle import cifar10_node_core, glorot_uniform_conv_params
        net = cifar10_node_core(W, W)
        layer = orc.NeuralODE(net, **kw)
        ps = glorot_uniform_conv_params(net, rng)
        D = net.state_dims
    else:
        import __graft_entry__ as entry
        pkg = entry.load_package()
        chain = pkg.TDConvChain(pkg.ConvChain(pkg.Conv(8, 64, True, "gelu"), pkg.Conv(64, 64, True, "gelu"),
                                              pkg.Conv(64, 8), width=W, height=W))
        layer = pkg.NeuralODE(chain, return_last_only=True, loop_mode=loop_mode, **kw)
        ps = layer.initialparameters(rng)
        D = chain.state_dims
    x = np.random.default_rng(1).standard_normal((D, B)).astype(np.float32)
    return layer, ps, x


def cifar10_secondary(torch, dev, B=256, steps=3):
    """Compact block for the default line: training iteration and in-solve f evaluation of the cifar10 node core
    (`python bench.py --workload cifar10` prints the full line with e2e, roofline and CPU baseline)."""
    layer, ps, x = cifar10_setup(B, False)
    D = x.shape[0]
    xt, pt = torch.from_numpy(x).to(dev), torch.from_numpy(ps).to(dev)
    cot_t = torch.ones((D, B), device=dev) / B
    st = layer.initialstates(np.random.default_rng(7))
    info = {}

    def step():
        sol, st2 = layer(xt, pt, st)
        layer.backward(sol, [cot_t], W_REG)
        info.update(nfe=int(st2["nfe"]), nf_bwd=int(sol.bwd_stats.nf_bwd), retcode=sol.retcode)
        sol.free()
    for _ in range(3):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    sol, _ = layer(xt, pt, st)
    sol.free()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(3):
        sol, _ = layer(xt, pt, st)
        sol.free()
    e1.record()
    torch.cuda.synchronize()
    us_f = 1e3 * e0.elapsed_time(e1) / (3.0 * info["nfe"])
    F_f = 2.0 * 9 * 1024 * (9 * 64 + 65 * 64 + 65 * 8)
    tf32_peak = measured_peaks()["bf16_burst"] / 2.0
    return {"workload": "BASELINE configs[3]: cifar10 node core, TDChain(Conv 9=>64 + BN gelu, Conv 65=>64 + BN gelu, Conv 65=>8), "
                        "state 32x32x8, batch 256, tol 1e-4, fwd + adjoint; tcgen05 implicit-GEMM convolutions in 3xTF32",
            "value": B / (ms / 1e3), "unit": "samples/s", "ms_per_step": ms, "nfe_per_step": info["nfe"],
            "nf_bwd_per_step": info["nf_bwd"], "retcode": info["retcode"], "us_per_feval": us_f,
            "tensor_frac_of_tf32_peak": F_f * B / (us_f * 1e-6) / 1e12 / tf32_peak}


def run_cifar10(args):
    """BASELINE configs[3]: conv-dynamics neural ODE, state 32x32x8 (after the AugmenterLayer), batch 256, local
    regularisation, tol 1e-4 (experiments/src/construct.jl:212-223): forward Tsit5 solve + regulariser step +
    adjoint pullback of sum(u(t2))/B + w_reg * reg_val.  The augment / BatchNorm(8) / classifier layers either
    side of the NeuralODE are not part of this workload.  Secondary workload (one JSON line, same contract)."""
    B = args.cifar_batch
    F_f = 2.0 * 9 * 1024 * (9 * 64 + 65 * 64 + 65 * 8)          # flop per f evaluation per sample
    wl = ("cifar10 node core (BASELINE configs[3]): TDChain(Conv 9=>64 + BN gelu, Conv 65=>64 + BN gelu, Conv 65=>8), "
          "3x3 pad 1, state 32x32x8, Tsit5 + :unbiased local reg, tol 1e-4; fwd + adjoint")
    if args.impl == "reference":
        Bs = args.cifar_ref_batch
        layer, ps, x = cifar10_setup(Bs, True)
        st = layer.initialstates(np.random.default_rng(7))
        ts = []
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            out, st2, aux = layer.forward(x, ps, st)
            layer.backward(aux, [np.zeros_like(x), np.ones_like(x) / Bs], np.float32(W_REG), ps)
            if i >= args.warmup:
                ts.append(time.perf_counter() - t0)
        ms = 1e3 * float(np.mean(ts))
        val = Bs / (ms / 1e3)
        print(json.dumps({"impl": "reference", "metric": "cifar10_train_samples_per_s", "value": val, "unit": "samples/s",
                          "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": {"workload": wl, "batch": B},
                          "cpu_baseline": {"value": val, "unit": "samples/s", "cores": os.cpu_count(), "kind": "port",
                                           "sample": f"batch {Bs} of the same workload per step"},
                          "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    import torch
    layer, ps, x = cifar10_setup(B, False, loop_mode=args.loop_mode)
    D = x.shape[0]
    dev = torch.device("cuda", 0)
    xt, pt = torch.from_numpy(x).to(dev), torch.from_numpy(ps).to(dev)
    cot_t = torch.ones((D, B), device=dev) / B
    x_pin = torch.from_numpy(x).pin_memory().numpy()
    cot_h = torch.ones((D, B)).div_(B).pin_memory().numpy()
    st = layer.initialstates(np.random.default_rng(7))
    info = {}

    def step(resident):
        sol, st2 = layer(xt if resident else x_pin, pt if resident else ps, st)
        layer.backward(sol, [cot_t if resident else cot_h], W_REG)
        b = sol.bwd_stats
        info.update(nfe=st2["nfe"], acc=sol.stats.naccept, rej=sol.stats.nreject, nf_bwd=b.nf_bwd,
                    bacc=b.naccept_bwd, brej=b.nreject_bwd, launches=sol.stats.gpu_launches + b.gpu_launches,
                    reg=float(st2["reg_val"]), retcode=sol.retcode)
        sol.free()

    def timed(n, resident):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(n):
            step(resident)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n
    clocks = ClockSampler(0)
    clocks.start()
    for _ in range(max(3, args.warmup)):
        step(True)
    step(False)
    ms = timed(args.steps, True)
    clk = clocks.stop()
    ms_e = timed(max(1, min(args.steps, args.e2e_steps)), False)
    # roofline probe: one f evaluation (3 convolutions + 2 BatchNorm reductions), CUDA events around 10 calls
    for _ in range(3):
        layer.dynamics(xt, pt, 0.5)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(10):
        layer.dynamics(xt, pt, 0.5)
    e1.record()
    torch.cuda.synchronize()
    us_f_call = 1e3 * e0.elapsed_time(e1) / 10      # through the C ABI: includes the per-call setup (weight images, buffers)
    # ... and inside a solve: the forward pass of the layer (main solve + regulariser step: nfe evaluations with their
    # stage combinations, BatchNorm reductions, error norms and controller launches), CUDA events around 3 passes
    nfe_f = []
    sol, _ = layer(xt, pt, st)          # untimed: the pool blocks of a forward pass are back in place after the probe above
    sol.free()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(3):
        sol, st2 = layer(xt, pt, st)
        nfe_f.append(int(st2["nfe"]))
        sol.free()
    e1.record()
    torch.cuda.synchronize()
    us_f = 1e3 * e0.elapsed_time(e1) / float(sum(nfe_f))
    peaks = measured_peaks()
    tf32_peak = peaks["bf16_burst"] / 2.0
    ach = F_f * B / (us_f * 1e-6) / 1e12
    traffic = None
    tr_path = os.path.join(ROOT, "profiles", "r2_traffic_cifar10.json")
    if B == 256 and os.path.exists(tr_path):   # ncu --set full of the same kernels at batch 256 (scratch/ncu_traffic.py)
        tr = json.load(open(tr_path))
        traffic = tr.get("dram_bytes_per_feval")
    cpu = None
    if not args.no_cpu_baseline:
        Bs = args.cifar_ref_batch
        olayer, ops, ox = cifar10_setup(Bs, True)
        ost = olayer.initialstates(np.random.default_rng(7))
        t0 = time.perf_counter()
        out, st2, aux = olayer.forward(ox, ops, ost)
        olayer.backward(aux, [np.zeros_like(ox), np.ones_like(ox) / Bs], np.float32(W_REG), ops)
        dt = time.perf_counter() - t0
        cpu = {"value": Bs / dt, "unit": "samples/s", "cores": os.cpu_count(), "kind": "port",
               "sample": f"1 iteration at batch {Bs} ({dt:.1f} s), numpy float32 oracle", "nfe": int(st2["nfe"])}
    print(json.dumps({"metric": "cifar10_train_samples_per_s", "value": B / (ms / 1e3), "unit": "samples/s", "n_gpus": 1,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
                      "scaling": "weak", "vs_baseline": None, "dtype": "tf32x3", "data": "synthetic",
                      "config": {"workload": wl, "batch": B,
                                 "l2": "hidden activations 2 x 67 MB per f evaluation at batch 256: larger than L2"},
                      "nfe_per_step": info["nfe"], "nfe_per_s": info["nfe"] / (ms / 1e3), "nf_bwd_per_step": info["nf_bwd"],
                      "steps_fwd": [info["acc"], info["rej"]], "steps_bwd": [info["bacc"], info["brej"]],
                      "reg_val": info["reg"], "retcode": info["retcode"],
                      "e2e": {"value": B / (ms_e / 1e3), "unit": "samples/s", "ms_per_step": ms_e,
                              "h2d_bytes_per_step": 4 * (2 * D * B + ps.size), "d2h_bytes_per_step": 4 * (2 * D * B + ps.size)},
                      "gpu_launches": int(info["launches"] * args.steps), "clocks": clk,
                      "roofline": {"bound": "tensor", "kernel": "one f evaluation inside the forward solve: convtc::pack_kernel x 3 (stage "
                                   "combination / BatchNorm + gelu, tf32 hi/lo split) + convtc::conv_kernel x 3 (tcgen05 implicit GEMM, "
                                   "3xTF32; the three MMAs per algorithmic one are NOT counted as work) + bn_finalize x 2; time = "
                                   "forward pass of the layer / nfe", "achieved": ach, "peak": tf32_peak,
                                   "unit": "TFLOP/s", "frac": ach / tf32_peak,
                                   "frac_of_3xtf32_issue_capacity": 3.0 * ach / tf32_peak,
                                   # dram read + write of the pack / conv kernels of one evaluation at batch 256, ncu --set full
                                   # (profiles/r2_traffic_cifar10.json); algorithmic: u in, z1 / z2 out and in, du out
                                   "traffic": traffic,
                                   "algorithmic_bytes_per_feval": 4.0 * 1024 * B * (8 + 64 + 64 + 64 + 64 + 8),
                                   "us_per_feval": us_f, "us_per_feval_through_the_c_abi": us_f_call,
                                   "peak_source": peaks["source"] + " (bf16 burst / 2 = TF32 dense)"},
                      "cpu_baseline": cpu}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--batch", type=int, default=8192, help="samples per GPU")
    ap.add_argument("--precision", default="auto", choices=["auto", "fp32", "tf32x3", "tf32"])
    ap.add_argument("--loop-mode", type=int, default=0)
    ap.add_argument("--ref-batch", type=int, default=512, help="bounded sample for the CPU reference")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the batch-128 (BASELINE configs[0]) block")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --batch samples per GPU; strong: --global-batch split over the GPUs")
    ap.add_argument("--global-batch", type=int, default=65536)
    ap.add_argument("--workload", default="mnist_ode", choices=["mnist_ode", "mnist_sde", "physionet", "cifar10"],
                    help="mnist_ode (default, the headline metric) or a secondary config")
    ap.add_argument("--phys-batch", type=int, default=256)
    ap.add_argument("--phys-T", type=int, default=49)
    ap.add_argument("--sde-batch", type=int, default=128)
    ap.add_argument("--cifar-batch", type=int, default=256)
    ap.add_argument("--cifar-ref-batch", type=int, default=4, help="bounded sample for the CPU oracle")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (u(t2) and d_x per sample, "
                         "d_ps, d_wc, the updated ps and wc, loss, reg_val, nfe) as DIR/<name>.npy, at most 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload != "mnist_ode" or args.impl != "native"):
        ap.error("--dump-outputs covers the default workload (--workload mnist_ode --impl native)")
    if args.workload == "mnist_sde":
        run_sde(args)
    elif args.workload == "physionet":
        run_physionet(args)
    elif args.workload == "cifar10":
        run_cifar10(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
