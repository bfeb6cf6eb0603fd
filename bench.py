#!/usr/bin/env python
"""bench.py -- interactions/sec of the ALS training hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            (our CUDA path; N>1 under torchrun)
  python bench.py --impl reference --gpus N --steps K ...   (CPU reference arm: the restated oracle)

A "step" is one ALS iteration (user half-epoch + item half-epoch, Gram precompute included) over the
synthetic CSR of BASELINE.json configs[1]: ALS d=128 on 10M x 1M, 1B nnz (SURVEY.md 8d generator C2).
`value` = nnz * steps / device time with everything resident in HBM; `e2e` = the same iteration driven
through the reference-facing host-pointer C ABI (bfl_als_partial_update: pinned-host CSR chunks H2D,
updated factor rows D2H inside the timed region).  One JSON line on stdout (rank 0).

`--dump-outputs DIR` writes, after the timed steps, the factor matrices the last timed step left behind as
DIR/<name>.npy (see dump_outputs); the workload and the initial factors are seeded, so two builds run with the same
arguments can be compared output for output.  Rows of more than 1536 nonzeros are summed chunk by chunk with float
atomics, so two runs of one build already differ: on C2 with --warmup 3 --steps 3 by up to 2.3e-3 of the largest
entry of P and of Q (one B200, 1000 W power limit).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: nothing is cached next to the sources

WORKLOADS = {
    # name: users, items, nnz, d, mean degree generator
    "c2": dict(users=10_000_000, items=1_000_000, nnz=1_000_000_000, d=128,
               desc="ALS d=128 10Mx1M 1B-nnz synthetic CSR (BASELINE configs[1])"),
    "c2_small": dict(users=1_000_000, items=100_000, nnz=100_000_000, d=128,
                     desc="1/10-scale C2 (debug only; NOT the headline workload)"),
    "c5": dict(users=5_000_000, items=500_000, nnz=2_000_000_000, d=256, zipf=1.1,
               desc="ALS d=256 Zipf(1.1) items 5Mx500k ~2B-nnz synthetic CSR (BASELINE configs[4])"),
    "c5_small": dict(users=500_000, items=50_000, nnz=200_000_000, d=256, zipf=1.1,
                     desc="1/10-scale BASELINE configs[4] (d=256, Zipf(1.1) items; debug only)"),
    "c5_d128": dict(users=500_000, items=50_000, nnz=200_000_000, d=128, zipf=1.1,
                    desc="1/10-scale Zipf(1.1) workload at d=128 (long-row path of the tensor-core kernel; debug only)"),
    "tiny": dict(users=20_000, items=5_000, nnz=1_000_000, d=128, desc="smoke-scale (debug only)"),
}
ALS_OPT = dict(d=128, optimizer="manual_cg", num_workers=1, compute_loss_on_training=False, alpha=8.0, reg_u=0.1,
               reg_i=0.1, block_size=32, adaptive_reg=False, num_cg_max_iters=3, eps=1e-10, cg_tolerance=1e-10,
               num_iters=1)  # d>=128 => iALS++ (als.cc:46); options of benchmark/test_performance.py:18-22


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------------
# workload (generated on the device; torch is plumbing only)
# ------------------------------------------------------------------------------------------------
def make_workload(w, device, seed=2024):
    """Row degrees ~ clipped lognormal (mean nnz/users, max 10k), items uniform, keys sorted within rows
    (the reference sorts by (row, col), fileio.hpp:330-341), values 1.0.  Returns dict of device tensors:
    rowwise (indptr_end, keys), colwise (indptr_end, keys), shared vals."""
    import torch
    if w.get("zipf"):
        return make_workload_zipf(w, device, seed=2027)
    U, I, nnz = w["users"], w["items"], w["nnz"]
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    sigma = 1.0
    mu = np.log(nnz / U) - 0.5 * sigma * sigma
    deg = torch.exp(torch.randn(U, device=device, generator=g, dtype=torch.float32) * sigma + mu)
    deg = torch.clamp(deg, max=10000.0)
    deg = torch.clamp((deg * (nnz / float(deg.sum().item()))).round().to(torch.int64), min=0)
    diff = int(nnz - int(deg.sum().item()))
    if diff != 0:  # spread the rounding remainder over the first |diff| rows with room
        idx = torch.nonzero(deg > (1 if diff < 0 else 0))[: abs(diff), 0]
        deg[idx] += 1 if diff > 0 else -1
    nnz = int(deg.sum().item())
    rows = torch.repeat_interleave(torch.arange(U, device=device, dtype=torch.int64), deg)
    cols = torch.randint(0, I, (nnz,), device=device, generator=g, dtype=torch.int64)
    key = rows * I + cols
    del rows, cols
    key = torch.sort(key).values
    r_keys = (key % I).to(torch.int32)
    rows = key // I
    del key
    r_indptr = torch.cumsum(deg, 0)
    key2 = r_keys.to(torch.int64) * U + rows
    del rows
    key2 = torch.sort(key2).values
    c_keys = (key2 % U).to(torch.int32)
    c_cols = key2 // U
    del key2
    c_indptr = torch.cumsum(torch.bincount(c_cols, minlength=I), 0)
    del c_cols
    vals = torch.ones(nnz, device=device, dtype=torch.float32)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return dict(U=U, I=I, nnz=nnz, r_indptr=r_indptr, r_keys=r_keys, c_indptr=c_indptr, c_keys=c_keys, vals=vals)


def make_workload_zipf(w, device, seed=2027):
    """SURVEY.md 8(d) generator C5: per-user degree ~ clipped lognormal, items ~ Zipf(alpha) over the item range by
    inverse-CDF sampling, duplicates within a user removed (so an item's degree is capped at the number of users), keys
    sorted within rows, values 1.0.  The draw count is inflated by the expected duplicate rate so that the
    de-duplicated matrix lands near the nominal nnz; the actual nnz is reported."""
    import torch
    U, I, nnz, alpha = w["users"], w["items"], w["nnz"], float(w["zipf"])
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    pmf = torch.arange(1, I + 1, device=device, dtype=torch.float64) ** (-alpha)
    pmf /= pmf.sum()
    mean_deg = nnz / U
    # expected distinct items among m draws: sum_k 1 - (1 - p_k)^m ; pick the per-user draw count whose expectation is mean_deg
    lo, hi = mean_deg, mean_deg * 4
    for _ in range(30):
        mid = 0.5 * (lo + hi)
        if float((1.0 - torch.exp(mid * torch.log1p(-pmf))).sum().item()) < mean_deg:
            lo = mid
        else:
            hi = mid
    inflate = hi / mean_deg
    sigma = 0.5
    mu = np.log(mean_deg * inflate) - 0.5 * sigma * sigma
    deg = torch.exp(torch.randn(U, device=device, generator=g, dtype=torch.float32) * sigma + mu)
    deg = torch.clamp(deg, max=float(I) / 4).round().to(torch.int64)
    cdf = torch.cumsum(pmf, 0).to(torch.float32)
    cdf[-1] = 1.0
    # torch.sort takes < 2^31 elements: the rowwise CSR is generated in user ranges of <= 2^29 draws (rows partition the
    # key space, so sorted ranges concatenate), the colwise CSR by item ranges of the finished matrix
    LIMIT = int(w.get("_chunk_limit", 1 << 29))
    cum = torch.cumsum(deg, 0)
    draws = int(cum[-1].item())
    r_keys_parts, r_cnt_parts = [], []
    u0 = 0
    while u0 < U:
        base = int(cum[u0 - 1].item()) if u0 else 0
        u1 = int(torch.searchsorted(cum, torch.tensor([base + LIMIT], device=device, dtype=cum.dtype)).item())
        u1 = min(max(u1, u0 + 1), U)
        dg = deg[u0:u1]
        n = int(dg.sum().item())
        rows = torch.repeat_interleave(torch.arange(u0, u1, device=device, dtype=torch.int64), dg)
        u = torch.rand(n, device=device, generator=g, dtype=torch.float32)
        col = torch.searchsorted(cdf, u).clamp_(max=I - 1)
        del u
        key = rows * I + col
        del rows, col
        key = torch.unique_consecutive(torch.sort(key).values)
        r_keys_parts.append((key % I).to(torch.int32))
        r_cnt_parts.append(torch.bincount(key // I - u0, minlength=u1 - u0))
        del key
        u0 = u1
    r_keys = torch.cat(r_keys_parts)
    del r_keys_parts
    r_indptr = torch.cumsum(torch.cat(r_cnt_parts), 0)
    del r_cnt_parts, cum, deg
    nnz = int(r_keys.numel())
    # colwise: item degrees, then per item range a stable sort of the range's entries by item (they are met in row order)
    c_cnt = torch.zeros(I, device=device, dtype=torch.int64)
    for s0 in range(0, nnz, 1 << 30):
        c_cnt += torch.bincount(r_keys[s0:s0 + (1 << 30)].to(torch.int64), minlength=I)
    c_indptr = torch.cumsum(c_cnt, 0)
    c_keys = torch.empty(nnz, device=device, dtype=torch.int32)
    i0 = 0
    while i0 < I:
        base = int(c_indptr[i0 - 1].item()) if i0 else 0
        i1 = int(torch.searchsorted(c_indptr, torch.tensor([base + LIMIT], device=device, dtype=c_indptr.dtype)).item())
        i1 = min(max(i1, i0 + 1), I)
        end = int(c_indptr[i1 - 1].item())
        idx_parts = []
        for s0 in range(0, nnz, 1 << 30):   # positions (in row order) of the entries whose item lies in [i0, i1)
            seg = r_keys[s0:s0 + (1 << 30)]
            idx_parts.append(torch.nonzero((seg >= i0) & (seg < i1)).flatten() + s0)
        idx = torch.cat(idx_parts)
        del idx_parts
        order = torch.sort(r_keys[idx], stable=True).indices
        idx = idx[order]
        del order
        c_keys[base:end] = torch.searchsorted(r_indptr, idx, right=True).to(torch.int32)   # row of entry position idx
        del idx
        i0 = i1
    vals = torch.ones(nnz, device=device, dtype=torch.float32)
    if device.type == "cuda":
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
    return dict(U=U, I=I, nnz=nnz, r_indptr=r_indptr, r_keys=r_keys, c_indptr=c_indptr, c_keys=c_keys, vals=vals,
                inflate=inflate, draws=draws)


def init_factors_t(rows, d, device, seed):
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    # abs(N(0, 1/d^2)) (buffalo/algo/als.py:85-86)
    return torch.abs(torch.randn(rows, d, device=device, generator=g, dtype=torch.float32) * (1.0 / d ** 2)).contiguous()


DUMP_BYTES_PER_ARRAY = 16 << 20  # at most four arrays per path: 64 MB in all


def dump_outputs(out_dir, arrays, seed=0):
    """Writes each output matrix as <out_dir>/<name>.npy (float32): all of it when it fits in DUMP_BYTES_PER_ARRAY,
    else a sample of its rows, the same sorted rows on every run (np.random.default_rng(seed), drawn in dict order)."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(seed)
    for name, F in arrays.items():
        rows = F.shape[0]
        n = min(rows, DUMP_BYTES_PER_ARRAY // (4 * F[0].numel()))
        if n < rows:
            F = F[torch.from_numpy(np.sort(rng.choice(rows, size=n, replace=False))).to(F.device)]
        np.save(os.path.join(out_dir, name + ".npy"), F.float().cpu().numpy())
    log("wrote %s to %s" % (", ".join(k + ".npy" for k in arrays), out_dir))


def algorithmic_bytes(nnz, rows, d):
    """SURVEY.md 8(d): per nnz 4d + 8 (opposite row + key + val); per updated row 12d + 8
    (indptr, warm-start read, write; the Gram read belongs to the precompute kernel)."""
    return nnz * (4 * d + 8) + rows * (12 * d + 8)


class ClockSampler(object):
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception as e:  # nvidia-smi missing
            log("clock sampler unavailable:", e)
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[5:9]):
                    if v.lower() == "active":
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------
# CPU arm: the restated oracle on the host cores (the reference cannot be built here, DESIGN.md)
# ------------------------------------------------------------------------------------------------
def host_threads():
    """Threads the CPU arm may really use: the scheduler affinity mask capped by the cgroup CPU quota (os.cpu_count()
    ignores both; an oversubscribed OpenMP team made the round-1 reference number swing 6.5x between boxes)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:  # cgroup v2, then v1
        if os.path.isfile("/sys/fs/cgroup/cpu.max"):
            q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
            if q != "max":
                quota = float(q) / float(p)
        elif os.path.isfile("/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / p
    except Exception:
        quota = None
    used = n if quota is None else max(1, min(n, int(quota + 0.5)))
    return used, {"affinity": n, "cgroup_quota": quota, "os_cpu_count": os.cpu_count()}


def cpu_sample_inputs(wl, Ph, Qh, frac, seed=99):
    """Bounded sample of the SAME workload: a seeded random subset of the rows of each orientation (compacted into a
    small CSR + a gathered copy of their factor rows) against the FULL opposite factor matrix."""
    rng = np.random.default_rng(seed)
    out = {}
    for axis, (ind, keys, rows_total, F) in enumerate([(wl["r_indptr"], wl["r_keys"], wl["U"], Ph),
                                                       (wl["c_indptr"], wl["c_keys"], wl["I"], Qh)]):
        n_rows = max(1, int(rows_total * frac))
        pick = np.sort(rng.choice(rows_total, size=n_rows, replace=False))
        hind = ind.cpu().numpy().astype(np.int64) if hasattr(ind, "cpu") else np.asarray(ind, np.int64)
        beg = np.where(pick > 0, hind[np.maximum(pick - 1, 0)], 0)
        end = hind[pick]
        lens = end - beg
        sind = np.cumsum(lens).astype(np.int64)
        n = int(sind[-1])
        # gather the picked rows' keys on whatever device holds them
        import torch
        idx = np.repeat(beg - np.concatenate(([0], sind[:-1])), lens) + np.arange(n, dtype=np.int64)
        kk = keys[torch.from_numpy(idx).to(keys.device)].cpu().numpy().astype(np.int32) if hasattr(keys, "device") \
            else np.asarray(keys)[idx].astype(np.int32)
        out[axis] = dict(rows=n_rows, indptr=sind, keys=kk, vals=np.ones(n, np.float32), nnz=n,
                         F=np.ascontiguousarray(F[pick]), nnz_total=int(hind[-1]))
    out["P"], out["Q"] = Ph, Qh
    return out


def cpu_run(sample, opt, threads):
    """One bounded CPU 'step'.  The Gram of each FULL opposite matrix and the row solves of the sample are timed
    separately and extrapolated to the full job:  T_full = T_gram(both) + sum_axis T_solve_sample / (sample nnz /
    total nnz);  value = nnz / T_full with nnz counted ONCE per iteration, like the GPU arm."""
    import oracle
    t_gram, t_solve, t_full_solve = 0.0, 0.0, 0.0
    for axis in (0, 1):
        s = sample[axis]
        o = oracle.OracleALS()
        o.init(dict(opt, num_workers=threads))
        if axis == 0:
            o.initialize_model(s["F"].copy(), sample["Q"])
        else:
            o.initialize_model(sample["P"], s["F"].copy())
        t0 = time.perf_counter()
        o.precompute(axis)
        t1 = time.perf_counter()
        o.partial_update(0, s["rows"], s["indptr"], s["keys"], s["vals"], axis)
        t2 = time.perf_counter()
        t_gram += t1 - t0
        t_solve += t2 - t1
        t_full_solve += (t2 - t1) * (s["nnz_total"] / max(1, s["nnz"]))
    return dict(t_gram_s=t_gram, t_solve_s=t_solve, t_full_s=t_gram + t_full_solve,
                frac=[sample[a]["nnz"] / max(1, sample[a]["nnz_total"]) for a in (0, 1)],
                sample_nnz=sample[0]["nnz"] + sample[1]["nnz"])


def size_cpu_sample(wl, Ph, Qh, opt, threads, target_s):
    """Grow the row fraction until one CPU step lasts about target_s seconds (bounded sample)."""
    frac = 2e-4
    for _ in range(5):
        sample = cpu_sample_inputs(wl, Ph, Qh, frac)
        r = cpu_run(sample, opt, threads)
        t = r["t_gram_s"] + r["t_solve_s"]
        if t >= 0.5 * target_s or frac >= 0.05:
            break
        grow = (0.8 * target_s - r["t_gram_s"]) / max(r["t_solve_s"], 1e-3)
        frac = min(0.05, frac * max(1.5, min(20.0, grow)))
    return frac, sample


def cpu_report(r, total_nnz, threads, tinfo, frac, kind="port"):
    v = total_nnz / r["t_full_s"]
    desc = ("seeded random %.4f%% of the user rows and of the item rows (%d nnz) solved against the full opposite "
            "factors; Gram of both full matrices timed separately; extrapolated T_full = T_gram + T_solve/frac"
            % (frac * 100, r["sample_nnz"]))
    return v, {"value": v, "unit": "nnz/s", "cores": threads, "threads_used": threads, "thread_info": tinfo,
               "kind": kind, "sample": desc, "t_gram_s": r["t_gram_s"], "t_solve_s": r["t_solve_s"],
               "frac": r["frac"], "t_full_extrapolated_s": r["t_full_s"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--algo", default="als", choices=["als", "bpr", "warp"],
                    help="als (default; the headline metric) or the BPRMF / WARP epochs of BASELINE configs[2], [3]")
    ap.add_argument("--optimizer", default=None, help="bpr/warp only: sgd | adagrad | adam (default: the reference's)")
    ap.add_argument("--workload", default=os.environ.get("BFL_BENCH_WORKLOAD"),
                    help="als: %s; bpr: c3, c3_small; warp: c4, c4_small" % ", ".join(sorted(WORKLOADS)))
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--kernel-mode", type=int, default=0, help="0 auto (d=128: tcgen05 kernel + SIMT class 0), 1 generic kernels, 2 tuned SIMT kernels only")
    ap.add_argument("--tc-min-class", type=int, default=None, help="first row-length class solved by the tensor-core kernel (default: library's)")
    ap.add_argument("--exchange", default=os.environ.get("BFL_EXCHANGE", "p2p"), choices=["p2p", "allgather"],
                    help="multi-GPU: fused peer stores from the solve kernel (default) or an NCCL all-gather per half-epoch")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the factors of the last step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl ours")
    if args.algo != "als":
        sys.path.insert(0, os.path.join(ROOT, "benchmarks"))
        import sgd_bench
        args.workload = args.workload or ("c3" if args.algo == "bpr" else "c4")
        assert args.workload in sgd_bench.SGD_WORKLOADS and sgd_bench.SGD_WORKLOADS[args.workload]["algo"] == args.algo
        return sgd_bench.main(args)
    args.workload = args.workload or "c2"
    assert args.workload in WORKLOADS, "unknown ALS workload %s" % args.workload
    assert args.warmup >= 3 or args.workload != "c2" or args.impl == "reference", "timing rules: warmup >= 3"

    import torch
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    w = WORKLOADS[args.workload]
    d = w["d"]
    opt = dict(ALS_OPT, d=d, _b200_kernel_mode=args.kernel_mode)
    if args.tc_min_class is not None:
        opt["_b200_tc_min_class"] = args.tc_min_class
    cores, tinfo = host_threads()

    if args.impl == "reference":
        if rank != 0:
            return 0
        return reference_arm(args, w, opt, cores, tinfo)

    assert torch.cuda.is_available(), "bench.py (our arm) needs a GPU: there is no CPU fallback"
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    from buffalo_b200 import _cabi, backend

    t_setup = time.perf_counter()
    wl = make_workload(w, device)
    U, I, nnz = wl["U"], wl["I"], wl["nnz"]
    P = init_factors_t(U, d, device, 7)
    Q = init_factors_t(I, d, device, 8)
    if rank == 0:
        log("workload built in %.1fs: U=%d I=%d nnz=%d d=%d" % (time.perf_counter() - t_setup, U, I, nnz, d))

    if world > 1 and args.exchange == "p2p":
        from buffalo_b200.parallel.dist import exportable_like
        P, Q = exportable_like(P), exportable_like(Q)
    obj = backend.CuALS()
    assert obj.init(opt), obj.last_error
    obj.bind_factors(P, Q)
    obj.bind_csr(0, wl["r_indptr"], wl["r_keys"], wl["vals"])
    obj.bind_csr(1, wl["c_indptr"], wl["c_keys"], wl["vals"])
    # contiguous row shards per rank + one in-place all-gather per half-epoch (buffalo_b200/parallel/dist.py)
    from buffalo_b200.parallel.dist import ShardedALS
    drv = ShardedALS(obj.precompute_device, obj.update_device, P, Q, rank, world, dist if world > 1 else None,
                     exchange=args.exchange, backend=obj, indptrs=(wl["r_indptr"], wl["c_indptr"]))
    (u0, u1, _), (i0, i1, _) = drv.ranges
    stream = torch.cuda.current_stream()
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    solve_events = []
    pending = {}

    def on_update(axis, when):
        e = ev()
        e.record(stream)
        if when == "begin":
            pending[axis] = e
        else:
            solve_events.append((axis, pending.pop(axis), e))

    def step(record=False):
        drv.iteration(on_update if record else None)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = _cabi.lib().bfl_kernel_launch_count()
    t0e, t1e = ev(), ev()
    barrier()
    t0e.record(stream)
    for _ in range(args.steps):
        step(record=True)
    t1e.record(stream)
    barrier()
    launches = _cabi.lib().bfl_kernel_launch_count() - launches0
    ms = t0e.elapsed_time(t1e)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"P": P, "Q": Q})   # every rank holds the full factors after the exchange
    if world > 1:
        t = torch.tensor([ms], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = nnz * args.steps / (ms / 1e3)

    # dominant kernel: the row-solve launches (one per half-epoch and rank)
    per_axis_ms = {0: [], 1: []}
    for axis, e0, e1 in solve_events:
        per_axis_ms[axis].append(e0.elapsed_time(e1))
    peak, peak_src = measured_peak()
    my_nnz = [int(wl["r_indptr"][u1 - 1].item() - (wl["r_indptr"][u0 - 1].item() if u0 else 0)),
              int(wl["c_indptr"][i1 - 1].item() - (wl["c_indptr"][i0 - 1].item() if i0 else 0))]
    my_rows = [u1 - u0, i1 - i0]
    alg_bytes = [algorithmic_bytes(my_nnz[a], my_rows[a], d) for a in (0, 1)]
    t_solve = sum(np.mean(per_axis_ms[a]) for a in (0, 1)) / 1e3
    achieved = sum(alg_bytes) / t_solve / 1e9
    # DRAM traffic of the same launches from the committed ncu capture (profiles/run_ncu.sh); single-GPU C2 only
    traffic, traffic_src = None, None
    tpath = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "traffic_c2.json")
    if world == 1 and args.workload == "c2" and os.path.isfile(tpath):
        tj = json.load(open(tpath))
        traffic, traffic_src = tj["user_pass"] + tj["item_pass"], tj["source"]
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "kernel": "ALS row-solve (user + item launches of one iteration)",
                "algorithmic_bytes_per_launch": {"user_pass": alg_bytes[0], "item_pass": alg_bytes[1]},
                "launch_ms": {"user_pass": float(np.mean(per_axis_ms[0])), "item_pass": float(np.mean(per_axis_ms[1]))},
                "share_of_step": t_solve * 1e3 * args.steps / ms}

    out = {"metric": "interactions/sec (nnz/s) ALS d=%d" % d, "value": value, "unit": "nnz/s", "n_gpus": world,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
           "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": w["desc"], "users": U, "items": I, "nnz": nnz, "d": d, "optimizer": "ialspp (d>=128)",
                      "parallelism": ("row-sharded x%d, updated factor rows pushed to the peer replicas from inside the solve "
                                      "kernel (P2P stores over NVLink) + 1-element all-reduce as barrier" % world)
                      if (world > 1 and args.exchange == "p2p") else
                      ("row-sharded x%d, NCCL all-gather of the updated factor shard per half-epoch" % world) if world > 1
                      else "single GPU",
                      "l2_policy": "inputs (>= 16 GB) larger than L2; no explicit flush"},
           "gpu_launches": int(launches), "roofline": roofline, "clocks": clocks}

    if world == 1 and not args.no_e2e:
        out["e2e"] = e2e_host_path(args, wl, opt, d, device, P, Q)
    elif world > 1 and not args.no_e2e:
        out["e2e"] = e2e_sharded(args, wl, drv, d, device, P, Q, rank, world, dist)
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            out["cpu_baseline"] = cpu_baseline(args, wl, P, Q, opt, cores, tinfo)
        except Exception as e:  # the oracle is test infrastructure; never fail the bench on it
            out["cpu_baseline"] = {"value": None, "error": str(e)}
    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()   # nobody tears down (peer mappings, NCCL) before rank 0 has printed
        dist.destroy_process_group()
    return 0


def e2e_sharded(args, wl, drv, d, device, P, Q, rank, world, dist):
    """N > 1: the same sharded iteration fed from HOST memory.  Every step each rank copies its shard of the CSR
    (keys + values of both orientations) from pinned host memory into the device arrays, solves, exchanges, and
    copies its freshly updated rows back to pinned host memory -- all inside the timed region (device time, max over
    ranks).  (The reference's plugin ABI is single-GPU; at N = 1 `e2e` goes through that ABI instead.)"""
    import torch
    (u0, u1, _), (i0, i1, _) = drv.ranges
    span = lambda ind, lo, hi: ((int(ind[lo - 1].item()) if lo else 0), int(ind[hi - 1].item()) if hi > lo else 0)  # noqa: E731
    ra, rb = span(wl["r_indptr"], u0, u1)
    ca, cb = span(wl["c_indptr"], i0, i1)
    rb, cb = max(rb, ra), max(cb, ca)
    pin = lambda t: t.cpu().pin_memory()  # noqa: E731
    host = {0: (pin(wl["r_keys"][ra:rb]), pin(wl["vals"][ra:rb]), ra, rb, wl["r_keys"]),
            1: (pin(wl["c_keys"][ca:cb]), pin(wl["vals"][ca:cb]), ca, cb, wl["c_keys"])}
    out_host = {0: torch.empty((u1 - u0, d), dtype=torch.float32).pin_memory(),
                1: torch.empty((i1 - i0, d), dtype=torch.float32).pin_memory()}
    # values are shared by both orientations in the synthetic workload (all ones): stage them in a scratch buffer so the
    # H2D copy is real but the resident array stays valid for the other orientation
    scratch = torch.empty(max(rb - ra, cb - ca, 1), dtype=torch.float32, device=device)

    # three streams: the H2D copy of the NEXT half-epoch's CSR shard and the D2H copy of the PREVIOUS half-epoch's rows
    # run beside the current solve (the shard being copied is not the one being read)
    cur = torch.cuda.current_stream()
    s_h2d, s_d2h = torch.cuda.Stream(), torch.cuda.Stream()
    h2d_done = {0: torch.cuda.Event(), 1: torch.cuda.Event()}
    solved = {0: torch.cuda.Event(), 1: torch.cuda.Event()}
    d2h_done = {0: torch.cuda.Event(), 1: torch.cuda.Event()}
    rows_of = {0: (u0, u1), 1: (i0, i1)}

    def issue_h2d(axis):
        hk, hv, a, b, dkeys = host[axis]
        s_h2d.wait_event(solved[axis])          # the previous solve of this orientation is done reading the shard
        with torch.cuda.stream(s_h2d):
            dkeys[a:b].copy_(hk, non_blocking=True)
            scratch[: b - a].copy_(hv, non_blocking=True)
            h2d_done[axis].record(s_h2d)

    for ax in (0, 1):
        solved[ax].record(cur)
        d2h_done[ax].record(cur)
    issue_h2d(0)

    def step():
        for axis in (0, 1):
            cur.wait_event(h2d_done[axis])
            cur.wait_event(d2h_done[axis])      # the rows about to be overwritten have reached the host
            issue_h2d(1 - axis)                 # next half-epoch's inputs fly behind this solve
            drv.half_epoch(axis)
            solved[axis].record(cur)
            lo, hi = rows_of[axis]
            F = P if axis == 0 else Q
            s_d2h.wait_event(solved[axis])
            with torch.cuda.stream(s_d2h):
                out_host[axis].copy_(F[lo:hi], non_blocking=True)
                d2h_done[axis].record(s_d2h)

    def barrier():
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
    step()
    cur.wait_stream(s_d2h)
    cur.wait_stream(s_h2d)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    cur.wait_stream(s_d2h)      # the last rows have reached the host
    cur.wait_stream(s_h2d)      # (one look-ahead copy of the next step's first shard is in the timed region too)
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    h2d = torch.tensor([8.0 * ((rb - ra) + (cb - ca))], device=device, dtype=torch.float64)
    d2h = torch.tensor([4.0 * d * ((u1 - u0) + (i1 - i0))], device=device, dtype=torch.float64)
    dist.all_reduce(h2d)
    dist.all_reduce(d2h)
    return {"value": wl["nnz"] * args.steps / (ms / 1e3), "unit": "nnz/s", "h2d_bytes_per_step": int(h2d.item()),
            "d2h_bytes_per_step": int(d2h.item()), "ms_per_step": ms / args.steps,
            "api": "sharded device iteration fed from pinned host CSR shards (H2D, copied beside the other orientation's solve) with D2H of the updated rows, all ranks"}


def e2e_host_path(args, wl, opt, d, device, Pd, Qd):
    """The same ALS iteration through the reference-facing C ABI with HOST buffers
    (init / initialize_model / set_placeholder / precompute / partial_update per chunk), pinned memory,
    H2D of every chunk's keys+vals and D2H of the updated rows inside the timed region."""
    import torch
    from buffalo_b200 import backend
    U, I, nnz = wl["U"], wl["I"], wl["nnz"]
    pin = lambda t: t.cpu().pin_memory()  # noqa: E731
    t0 = time.perf_counter()
    h = {"r_indptr": wl["r_indptr"].cpu().numpy(), "c_indptr": wl["c_indptr"].cpu().numpy(),
         "r_keys": pin(wl["r_keys"]), "c_keys": pin(wl["c_keys"]), "vals": pin(wl["vals"])}
    P = Pd.cpu().pin_memory()
    Q = Qd.cpu().pin_memory()
    obj = backend.CuALS()
    assert obj.init(opt)
    obj.initialize_model(P.numpy(), Q.numpy())
    # BufferedDataMatrix semantics: row-aligned chunks of <= limit nnz (buffered_data.py:47-118), batch_mb=4098
    limit = int(4098 * 1024 * 1024 / 16 / 2)
    obj.set_placeholder(h["r_indptr"], h["c_indptr"], limit)
    log("e2e host staging %.1fs" % (time.perf_counter() - t0))

    def chunks(indptr):
        out, start, rows = [], 0, len(indptr)
        while start < rows:
            beg = 0 if start == 0 else int(indptr[start - 1])
            nxt = int(np.searchsorted(indptr, beg + limit, side="right"))
            nxt = min(max(nxt, start + 1), rows)
            out.append((start, nxt, beg, int(indptr[nxt - 1])))
            start = nxt
        return out
    plan = [(0, chunks(h["r_indptr"]), h["r_indptr"], h["r_keys"].numpy()),
            (1, chunks(h["c_indptr"]), h["c_indptr"], h["c_keys"].numpy())]
    vals = h["vals"].numpy()

    def step():
        for axis, cks, indptr, keys in plan:
            obj.precompute(axis)
            for (a, b, beg, end) in cks:
                obj.partial_update(a, b, indptr, keys[beg:end], vals[beg:end], axis)
    step()  # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return {"value": nnz * args.steps / dt, "unit": "nnz/s", "h2d_bytes_per_step": int(2 * nnz * 8),
            "d2h_bytes_per_step": int((U + I) * d * 4), "ms_per_step": dt * 1e3 / args.steps,
            "api": "bfl_als_partial_update (host CSR chunks, pinned)", "chunks_per_step": len(plan[0][1]) + len(plan[1][1])}


def cpu_baseline(args, wl, P, Q, opt, threads, tinfo):
    import oracle
    oracle.build()
    Ph, Qh = P.cpu().numpy(), Q.cpu().numpy()
    frac, sample = size_cpu_sample(wl, Ph, Qh, opt, threads, args.cpu_seconds)
    r = cpu_run(sample, opt, threads)
    return cpu_report(r, wl["nnz"], threads, tinfo, frac)[1]


def reference_arm(args, w, opt, threads, tinfo):
    """CPU arm: the restated reference path (oracle port; oracle/_ref cannot be built, DESIGN.md) on the host threads
    this process may use, each step a bounded random sample of the same workload, extrapolated to the full job."""
    import torch
    import oracle
    oracle.build()
    device = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
    if device.type == "cpu":
        w = dict(w)
        log("no GPU for workload generation: CPU generation of a 1/50 slice of the workload")
        scale = 50
        w.update(users=w["users"] // scale, nnz=w["nnz"] // scale)
    wl = make_workload(w, device) if device.type == "cuda" else make_workload_cpu(w)
    d = w["d"]
    P = init_factors_t(wl["U"], d, device, 7)
    Q = init_factors_t(wl["I"], d, device, 8)
    Ph, Qh = P.cpu().numpy(), Q.cpu().numpy()
    frac, sample = size_cpu_sample(wl, Ph, Qh, opt, threads, args.cpu_seconds)
    total_nnz = wl["nnz"]
    del wl
    for _ in range(args.warmup):
        cpu_run(sample, opt, threads)
    acc = None
    for _ in range(args.steps):
        r = cpu_run(sample, opt, threads)
        if acc is None:
            acc = dict(r)
        else:
            for k in ("t_gram_s", "t_solve_s", "t_full_s"):
                acc[k] += r[k]
    for k in ("t_gram_s", "t_solve_s", "t_full_s"):
        acc[k] /= args.steps
    v, cb = cpu_report(acc, total_nnz, threads, tinfo, frac)
    out = {"impl": "reference", "metric": "interactions/sec (nnz/s) ALS d=%d" % d, "value": v, "unit": "nnz/s",
           "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": acc["t_full_s"] * 1e3, "ms_per_step_measured_sample": (acc["t_gram_s"] + acc["t_solve_s"]) * 1e3,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": w["desc"], "users": w["users"], "items": w["items"], "nnz": w["nnz"], "d": d,
                      "optimizer": "ialspp (d>=128)", "sampled": cb["sample"]},
           "cpu_baseline": cb,
           "e2e": {"value": v, "unit": "nnz/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)
    return 0


def make_workload_cpu(w, seed=2024):
    import torch
    rng = np.random.default_rng(seed)
    U, I, nnz = w["users"], w["items"], w["nnz"]
    deg = np.minimum(np.exp(rng.normal(np.log(nnz / U) - 0.5, 1.0, U)), 10000)
    deg = np.maximum((deg * nnz / deg.sum()).round().astype(np.int64), 0)
    nnz = int(deg.sum())
    rows = np.repeat(np.arange(U), deg)
    cols = rng.integers(0, I, nnz)
    key = np.sort(rows * I + cols)
    r_keys = (key % I).astype(np.int32)
    rows = key // I
    key2 = np.sort(r_keys.astype(np.int64) * U + rows)
    t = torch.from_numpy
    return dict(U=U, I=I, nnz=nnz, r_indptr=t(np.cumsum(deg)), r_keys=t(r_keys),
                c_indptr=t(np.cumsum(np.bincount(key2 // U, minlength=I))), c_keys=t((key2 % U).astype(np.int32)),
                vals=torch.ones(nnz))


if __name__ == "__main__":
    sys.exit(main())
