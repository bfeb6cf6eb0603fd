#!/usr/bin/env python
"""Throughput of the BPRMF / WARP training path (BASELINE configs[2] C3 and configs[3] C4): positives per second of whole
epochs (negative sampling + update kernels + optimizer step) -- same JSON contract as bench.py, which delegates here for
`bench.py --algo bpr|warp`.

  python bench.py --algo warp --workload c4            (WARP d=64, 1M x 100k, 50M nnz, adagrad, max_trials=500)
  python bench.py --algo bpr  --workload c3            (BPRMF d=128, 10M x 1M, 500M positives, sgd)
  torchrun ... bench.py --algo bpr --workload c3 --gpus 8
  python bench.py --algo bpr --workload c3 --impl reference   (CPU arm: the oracle on the host threads, bounded sample)

Under torchrun (one rank per GPU) the users are sharded by nonzeros (parallel/dist.py::ShardedSGD): gradient-
accumulating configurations all-reduce the accumulators once per epoch; plain-SGD BPR sums the item deltas of the epoch
(user rows are owner-only and are not exchanged during training).
"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)

SGD_WORKLOADS = {
    "c3": dict(algo="bpr", users=10_000_000, items=1_000_000, nnz=500_000_000, d=128,
               desc="BPRMF d=128 10Mx1M 500M positives (BASELINE configs[2])"),
    "c3_small": dict(algo="bpr", users=1_000_000, items=100_000, nnz=50_000_000, d=128,
                     desc="1/10-scale C3 (debug only)"),
    "c4": dict(algo="warp", users=1_000_000, items=100_000, nnz=50_000_000, d=64,
               desc="WARP d=64 1Mx100k 50M nnz (BASELINE configs[3])"),
    "c4_small": dict(algo="warp", users=100_000, items=20_000, nnz=5_000_000, d=64, desc="1/10-scale C4 (debug only)"),
}


def sgd_options(algo, d, epochs, optimizer=None):
    """The reference defaults (buffalo/algo/options.py:221-252 BPRMF, :286-311 WARP) with d / num_iters of the config."""
    from buffalo_b200.algo import options
    base = dict(options._BPRMF if algo == "bpr" else options._WARP)
    for k in ("model_path", "data_opt", "accelerator", "hyper_threads", "evaluation_period"):
        base.pop(k, None)
    base.update(d=d, num_iters=epochs, random_seed=7, compute_loss_on_training=True, num_workers=1)
    if optimizer:
        base["optimizer"] = optimizer
    if algo == "warp":
        base.update(use_bias=False, reg_b=0.0, num_negative_samples=1, verify_neg=True, sampling_power=0.0)
    return base


def algorithmic_bytes(algo, d, nnz, users, items, optimizer, mean_trials):
    """Per epoch.  BPR sgd: a warp walks one user's positives back to back, so the user row is read and written once
    per USER; the positive and the negative item row are read and updated per sample (4 x 4d), plus key + draw.
    WARP: per positive the positive row + E[trials] sampled rows are read (Q is 25.6 MB at C4 = L2-resident, so these
    are L2 reads, not HBM), three gradient rows are accumulated; the optimizer + projection pass streams theta, grad,
    state of P and Q."""
    if algo == "bpr":
        per = 4 * 4 * d + 12
        tot = nnz * per + users * 2 * 4 * d
        if optimizer != "sgd":
            tot += (users + items) * 4 * d * (6 if optimizer == "adagrad" else 8)
        return tot
    per = 4 * d * (2 + mean_trials) + 3 * 2 * 4 * d + 12
    return nnz * per + (users + items) * 4 * d * 8


def main(args):
    import torch
    import torch.distributed as dist
    import bench
    from buffalo_b200 import _cabi, backend
    from buffalo_b200.parallel.dist import ShardedSGD
    w = SGD_WORKLOADS[args.workload]
    algo, d = w["algo"], w["d"]
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    threads, tinfo = bench.host_threads()
    if args.impl == "reference":
        if rank != 0:
            return 0
        return reference_arm(args, w, threads, tinfo)
    assert torch.cuda.is_available(), "needs a GPU: there is no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    wl = bench.make_workload(dict(users=w["users"], items=w["items"], nnz=w["nnz"]), dev, seed=2025 if algo == "bpr" else 2026)
    U, I, nnz = wl["U"], wl["I"], wl["nnz"]
    steps, warmup = args.steps, args.warmup
    opt = sgd_options(algo, d, steps + warmup, args.optimizer)
    optimizer = opt["optimizer"]
    g = backend.CuSGD(algo)
    assert g.init(opt)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1)
    # reference initialisation: abs(N(0, 1/d^2)) for BPRMF (bpr.py:84-97), N(0, 1/d^2) for WARP (warp.py:79-92)
    P = torch.randn(U, d, device=dev, generator=gen) * (1.0 / d ** 2)
    Q = torch.randn(I, d, device=dev, generator=gen) * (1.0 / d ** 2)
    if algo == "bpr":
        P, Q = P.abs_(), Q.abs_()
    P, Q = P.contiguous(), Q.contiguous()
    Qb = torch.zeros(I, 1, device=dev)
    shard = ShardedSGD(None, None, P, Q, Qb, wl["r_indptr"], rank, world, dist if world > 1 else None)
    g.bind_factors(P, Q, Qb, shard.local_positives(wl["r_indptr"]))
    g.bind_csr(wl["r_indptr"], wl["r_keys"])
    g.launch_workers()
    grads = None
    if optimizer != "sgd" or algo == "warp":
        grads = [g.grad_tensor(0, P.shape), g.grad_tensor(1, Q.shape)] + ([g.grad_tensor(2, (I,))] if algo == "bpr" else [])
        grads += [g.count_tensor(0, U), g.count_tensor(1, I)]
    trials = None
    if algo == "warp" and world == 1:
        trials = torch.zeros(nnz, dtype=torch.int32, device=dev)
        negs = torch.zeros(nnz, dtype=torch.int32, device=dev)
        g.set_trace(trials, negs)
    drv = ShardedSGD(g.add_jobs_device, g.update_parameters_device, P, Q, Qb, wl["r_indptr"], rank, world,
                     dist if world > 1 else None, grads=grads)
    drv.begin()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(warmup):
        drv.epoch()
    barrier()
    sampler = bench.ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = _cabi.lib().bfl_kernel_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(steps):
        drv.epoch()
    e1.record()
    barrier()
    launches = _cabi.lib().bfl_kernel_launch_count() - launches0
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    drv.finalize()
    if args.dump_outputs and rank == 0:
        bench.dump_outputs(args.dump_outputs, dict(P=P, Q=Q, Qb=Qb) if algo == "bpr" else dict(P=P, Q=Q))
    mean_trials = None
    if trials is not None:
        tt = trials.to(torch.float32)
        mean_trials = float(tt[tt > 0].mean().item()) if bool((tt > 0).any()) else 0.0
    loss, updates = g.read_stats() if algo == "warp" else (float("nan"), 0)
    finite = bool(torch.isfinite(P).all().item() and torch.isfinite(Q).all().item())
    value = nnz * steps / (ms / 1e3)
    peak, peak_src = bench.measured_peak()
    alg = algorithmic_bytes(algo, d, nnz, U, I, optimizer, mean_trials if mean_trials is not None else 2.0)
    achieved = alg * steps / (ms / 1e3) / 1e9 / world      # per GPU (every rank streams its own share)
    tfile = os.path.join(ROOT, "profiles", "traffic_%s.json" % args.workload)
    traffic = json.load(open(tfile)) if (world == 1 and os.path.isfile(tfile)) else None
    out = {"metric": "positives/sec (nnz/s) %s d=%d" % ("BPRMF" if algo == "bpr" else "WARP", d), "value": value,
           "unit": "nnz/s", "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms / steps,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": w["desc"], "users": U, "items": I, "nnz": nnz, "d": d, "optimizer": optimizer,
                      "max_trials": opt.get("max_trials"), "parallelism": "users sharded by nonzeros x%d" % world,
                      "l2_policy": "factor matrices + CSR larger than L2 (C3); C4: Q is L2-resident by design"},
           "gpu_launches": int(launches), "clocks": clocks, "finite": finite,
           "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                        "traffic": (traffic or {}).get("dram_bytes_per_epoch"), "traffic_source": (traffic or {}).get("source"),
                        "peak_source": peak_src, "kernel": "epoch (sample + apply / accumulate + optimizer), per GPU",
                        "algorithmic_bytes_per_epoch": alg,
                        "note": "WARP C4: Q (25.6 MB) is L2-resident; the bound is L2 latency + RNG, not HBM" if algo == "warp" else
                                "user rows counted once per user (a warp walks one user's positives back to back)"},
           "warp": {"mean_trials": mean_trials, "loss_rank0": loss, "updates_rank0": updates} if algo == "warp" else None}
    if world == 1 and not args.no_e2e:
        out["e2e"] = e2e_host(args, w, wl, opt, P, Q)
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            out["cpu_baseline"] = cpu_sample_run(w, wl, opt, threads, tinfo, args.cpu_seconds)
        except Exception as e:
            out["cpu_baseline"] = {"value": None, "error": str(e)}
    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def e2e_host(args, w, wl, opt, Pd, Qd):
    """The same epochs through the reference-facing host-pointer ABI (initialize_model / set_placeholder / add_jobs per
    chunk / update_parameters, bpr.py:170-188): the CSR keys go H2D every epoch, the factors come back D2H every epoch."""
    import torch
    from buffalo_b200 import backend
    algo, d = w["algo"], w["d"]
    U, I, nnz = wl["U"], wl["I"], wl["nnz"]
    g = backend.CuSGD(algo)
    assert g.init(opt)
    P = Pd.cpu().pin_memory().numpy()
    Q = Qd.cpu().pin_memory().numpy()
    Qb = np.zeros((I, 1), np.float32)
    indptr = wl["r_indptr"].cpu().numpy()
    keys = wl["r_keys"].cpu().pin_memory().numpy()
    g.initialize_model(P, Q, Qb, nnz)
    limit = int(4098 * 1024 * 1024 / 16 / 2)
    g.set_placeholder(indptr, limit)
    g.launch_workers()
    cuts, start = [], 0
    while start < U:
        beg = 0 if start == 0 else int(indptr[start - 1])
        nxt = min(max(int(np.searchsorted(indptr, beg + limit, side="right")), start + 1), U)
        cuts.append((start, nxt, beg, int(indptr[nxt - 1])))
        start = nxt

    def epoch():
        for a, b, beg, end in cuts:
            g.add_jobs(a, b, indptr, keys[beg:end])
        g.update_parameters()
    epoch()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        epoch()
    g.wait_until_done()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return {"value": nnz * args.steps / dt, "unit": "nnz/s", "h2d_bytes_per_step": int(nnz * 4),
            "d2h_bytes_per_step": int((U + I) * d * 4 + I * 4), "ms_per_step": dt * 1e3 / args.steps,
            "api": "bfl_sgd_add_jobs (host CSR chunks) + bfl_sgd_update_parameters (factors copied back)"}


def cpu_sample_run(w, wl, opt, threads, tinfo, target_s, warmup=0, steps=1):
    """The oracle (restated bpr.cc / warp.cc) on the host threads over a contiguous user range sized to ~target_s."""
    import oracle
    oracle.build()
    algo, d = w["algo"], w["d"]
    U, I = wl["U"], wl["I"]
    indptr = wl["r_indptr"].cpu().numpy().astype(np.int64)
    rng = np.random.default_rng(5)
    Q = (rng.normal(size=(I, d)) / d ** 2).astype(np.float32)
    rows = 2000
    best = None
    for _ in range(5):
        rows = int(min(rows, U))
        lo = int(rng.integers(0, max(1, U - rows)))
        hi = lo + rows
        beg = int(indptr[lo - 1]) if lo else 0
        end = int(indptr[hi - 1])
        keys = wl["r_keys"][beg:end].cpu().numpy().astype(np.int32)
        sub_ind = (indptr[lo:hi] - beg).astype(np.int64)
        P = (rng.normal(size=(rows, d)) / d ** 2).astype(np.float32)
        o = oracle.OracleSGD(warp=(algo == "warp"), use_lut=(algo == "bpr"))
        o.init(dict(opt, num_workers=threads, num_iters=1 + warmup + steps))
        Qc, Qb = Q.copy(), np.zeros((I, 1), np.float32)
        o.initialize_model(P, Qc, Qb, len(keys))
        t0 = time.perf_counter()
        o.add_jobs(0, rows, sub_ind, keys)
        o.update_parameters()
        t = time.perf_counter() - t0
        best = dict(t=t, nnz=len(keys), rows=rows)
        if t >= 0.5 * target_s or rows >= U:
            break
        rows = int(rows * max(2.0, min(30.0, 0.8 * target_s / max(t, 1e-3))))
    v = best["nnz"] / best["t"]
    return {"value": v, "unit": "nnz/s", "cores": threads, "threads_used": threads, "thread_info": tinfo, "kind": "port",
            "sample": "one epoch over a random contiguous range of %d users (%d positives) with the full item matrix, "
                      "optimizer step over that range + all items included; %.1f s" % (best["rows"], best["nnz"], best["t"]),
            "seconds": best["t"]}


def reference_arm(args, w, threads, tinfo):
    import torch
    import bench
    algo, d = w["algo"], w["d"]
    device = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
    ww = dict(users=w["users"], items=w["items"], nnz=w["nnz"])
    if device.type == "cpu":
        ww.update(users=w["users"] // 50, nnz=w["nnz"] // 50)
    wl = bench.make_workload(ww, device, seed=2025 if algo == "bpr" else 2026) if device.type == "cuda" else bench.make_workload_cpu(ww)
    opt = sgd_options(algo, d, args.steps + args.warmup, args.optimizer)
    vals = []
    for i in range(args.warmup + args.steps):
        cb = cpu_sample_run(w, wl, opt, threads, tinfo, args.cpu_seconds)
        if i >= args.warmup:
            vals.append(cb)
    v = float(np.mean([c["value"] for c in vals]))
    cb = dict(vals[-1], value=v)
    out = {"impl": "reference", "metric": "positives/sec (nnz/s) %s d=%d" % ("BPRMF" if algo == "bpr" else "WARP", d),
           "value": v, "unit": "nnz/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": w["nnz"] / v * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": w["desc"], "users": w["users"], "items": w["items"], "nnz": w["nnz"], "d": d,
                      "optimizer": opt["optimizer"], "max_trials": opt.get("max_trials"), "sampled": cb["sample"]},
           "cpu_baseline": cb, "e2e": {"value": v, "unit": "nnz/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)
    return 0


if __name__ == "__main__":
    import bench
    sys.exit(bench.main())
