#!/usr/bin/env python
"""bench.py -- TF-IDF + LSI(k=50) throughput on synthetic sparse ATAC (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--scaling weak|strong] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" is one pass of the hot path -- mu.atac.pp.tfidf + mu.atac.tl.lsi -- over the whole synthetic matrix.
Default workload = BASELINE.json configs[1]: 1M cells x 200k peaks, 3 % nnz per GPU (weak scaling: every rank owns
1M cells; peak-space objects are replicated, one allreduce of column sums, one of A^T Y per Lanczos step, one of
the b x b Gram per QR).  ``--scaling strong`` splits --cells over the ranks instead.

Prints ONE JSON line (rank 0):
  value        cells/s with the counts already resident in HBM (CUDA events, max over ranks)
  e2e          the same calls on HOST scipy matrices (H2D of indices/values, D2H of the TF-IDF values and the
               factors inside the timed region), with a host-side breakdown
  roofline     the dominant kernel (CSR SpMM) measured live with CUDA events
  cpu_baseline the scipy oracle on a bounded row-sample + the GPU on that SAME sample (same_matrix_speedup)
  mofa         BASELINE configs[2]: mu.tl.mofa, RNA + ATAC, k=30, 15 iterations, cells sharded like the main leg
  strong       (N > 1) the main step with --cells TOTAL split over the ranks
  cfg3         (N = 8, or --cfg3 1) BASELINE configs[3]: LSI k=100 on 4M x 500k over 8 GPUs
``--impl reference`` times the CPU oracle (scipy restatement of the reference, oracle/) on the host cores; it never
loads the CUDA library.

``--dump-outputs DIR`` writes, after the timed steps, what the last main-leg step returned (TF-IDF values, LSI
embedding, loadings and standard deviations) as DIR/<slot>.npy.  The synthetic matrix depends only on the arguments,
so two builds run with the same arguments can be compared array for array (``dump_outputs``).
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "cells/sec for TF-IDF+LSI(k=50) on 1Mx200k sparse ATAC"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--cells", type=int, default=1_000_000, help="cells per GPU (weak) or in total (strong)")
    ap.add_argument("--peaks", type=int, default=200_000)
    ap.add_argument("--density", type=float, default=0.03)
    ap.add_argument("--k", type=int, default=50)
    ap.add_argument("--topics", type=int, default=0,
                    help="planted topics of the synthetic matrix (0: max(64, k+14), so that the k wanted components "
                         "are separated from the noise bulk, SURVEY App. E)")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--tol", type=float, default=1e-5)
    ap.add_argument("--sample-cells", type=int, default=10_000,
                    help="rows of the CPU-baseline sample (first rows of the benchmark matrix)")
    ap.add_argument("--e2e-cells", type=int, default=-1,
                    help="cells per GPU for the e2e legs (-1: same as the main leg, reduced only if host RAM cannot hold "
                         "every rank's host matrices; the limit is stated in the JSON)")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-mofa", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--cfg3", type=int, default=-1, help="run the configs[3] leg (-1: only when 8 ranks)")
    ap.add_argument("--mofa-cells", type=int, default=-1, help="cells per GPU of the MOFA leg (-1: as the main leg)")
    ap.add_argument("--mofa-iters", type=int, default=15)
    ap.add_argument("--mofa-k", type=int, default=30)
    ap.add_argument("--breakdown", action="store_true", help="one extra, synchronising step with phase timers")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned to its caller as DIR/<slot>.npy "
                         "(fixed samples of the large arrays, under 64 MB in all; rank 0's cell shard when N > 1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 9 for n, v in zip(names, r[5:9]) if v.lower() == "active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def onchip_roofline(nnz, P, ms_per_pass, sm_mhz, n_sms=148, operand_bytes=4.0):
    """Second roofline of the SpMM kernel: every non-zero moves P operand elements plus its 8-byte {index, value}
    entry through the SM's L1/LSU data path (128 B/clk/SM, shared with shared-memory traffic).  Reported next to
    the HBM figure because this, not DRAM, is what the kernel saturates (DESIGN.md section 4)."""
    if not sm_mhz or not ms_per_pass or ms_per_pass != ms_per_pass:
        return None
    bytes_per_pass = float(nnz) * (operand_bytes * P + 8.0)
    peak = n_sms * 128.0 * sm_mhz * 1e6 / 1e12                     # TB/s
    ach = bytes_per_pass / (ms_per_pass * 1e-3) / 1e12
    return {"bound": "l1-lsu data path (128 B/clk/SM)", "achieved": ach, "peak": peak, "unit": "TB/s",
            "frac": ach / peak, "bytes_per_nnz": operand_bytes * P + 8.0, "sm_mhz": sm_mhz, "sms": n_sms}


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ------------------------------------------------------------------------------------------------
def cpu_oracle_step(X, k):
    """The reference's CPU path (scipy restatement of preproc.py:92-119 + svds + tools.py:56-65)."""
    from oracle.lsi_ref import lsi_ref
    from oracle.tfidf_ref import tfidf_ref
    t0 = time.perf_counter()
    Y = tfidf_ref(X)
    t1 = time.perf_counter()
    lsi_ref(Y, k)
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1


def run_reference(args, rank):
    """--impl reference: the oracle (kind 'port': import muon is impossible here, SURVEY 8c) timed on the host cores
    on a bounded row-sample of the same workload.  Rank 0 only.  Does not load libmuon_b200.so: the sample comes from
    the numpy twin of the generator (bit-identical to the device generator, tests/test_gpu_kernels.py)."""
    if rank != 0:
        return
    from muon_b200._synth import generate_host, make_tables
    S = args.sample_cells
    tb = make_tables(args.peaks, args.density, args.topics, args.seed)
    t0 = time.perf_counter()
    X = generate_host(S, args.peaks, args.density, tables=tb, row0=0)
    t_gen = time.perf_counter() - t0
    # warm-up steps touch every code path (scipy, ARPACK, BLAS thread pools) on the first S/8 rows: a CPU has no
    # clocks or caches to warm for minutes, and W full-size steps would triple the wall time of this arm
    Xw = X[: max(S // 8, min(S, 256))]
    for _ in range(args.warmup):
        cpu_oracle_step(Xw, min(args.k, min(Xw.shape) - 1))
    t0 = time.perf_counter()
    parts = [cpu_oracle_step(X, args.k) for _ in range(args.steps)]
    dt = time.perf_counter() - t0
    v = S * args.steps / dt
    sample = (f"first {S} cells x {args.peaks} peaks ({X.nnz} nnz) of the synthetic matrix (numpy generator, {t_gen:.0f} s, "
              f"untimed); per step tfidf {np.mean([p[0] for p in parts]):.2f} s + svds {np.mean([p[1] for p in parts]):.2f} s; "
              f"warm-up steps on the first {Xw.shape[0]} cells")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "cells/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"TF-IDF + LSI k={args.k} on {args.cells}x{args.peaks} ATAC ({args.density:.0%} nnz) per GPU",
                   "sample": sample},
        "cpu_baseline": {"value": v, "unit": "cells/s", "cores": host_threads(), "kind": "port", "sample": sample,
                         "note": "scipy's sparse kernels (csr_matvec inside ARPACK, SMMP matmul in tfidf) are "
                                 "single-threaded; BLAS in the svds tail uses all cores"},
        "e2e": {"value": v, "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ------------------------------------------------------------------------------------------------
class Ctx:
    pass


def timed_steps(ctx, step, steps, warmup, sample_clocks=False):
    """W untimed + K timed steps, barrier + synchronize on both sides, CUDA events, max over ranks.
    Returns (ms_total, per-kernel event times, launches, last step result, clocks)."""
    import torch
    from muon_b200 import _lib
    res = None
    for _ in range(warmup):
        res = step()
    sampler = ClockSampler(ctx.local) if (sample_clocks and ctx.rank == 0) else None
    if sampler:
        sampler.start()
    ctx.barrier()
    _lib.PROFILE = {}
    launches0 = _lib.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        res = step()
    e1.record()
    ctx.barrier()
    prof, _lib.PROFILE = _lib.PROFILE, None
    launches = _lib.LAUNCHES - launches0
    clocks = sampler.stop() if sampler else None
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if ctx.world > 1:
        import torch.distributed as dist
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    kern = {name: [a.elapsed_time(b) for a, b in evs] for name, evs in prof.items()}
    return float(ms[0]), kern, launches, res, clocks


def lsi_step_fn(ctx, A, k, tol):
    import pandas as pd

    import muon_b200 as mu
    obs0 = pd.DataFrame(index=pd.RangeIndex(A.shape[0]).astype(str))
    var0 = pd.DataFrame(index=pd.RangeIndex(A.shape[1]).astype(str))

    def step(keep=None):
        """``keep``: a dict that receives the step's AnnData (the caller's view of the result) as keep["ad"]."""
        if keep is not None:
            keep.clear()                              # the previous step's result goes before this step allocates
        ad = mu.SimpleAnnData(A, obs=obs0, var=var0)  # counts stay untouched: tfidf writes a new matrix
        mu.atac.pp.tfidf(ad)
        info = mu.atac.tl.lsi(ad, n_comps=k, tol=tol, return_info=True)
        # leading singular values (stdev * sqrt(n-1), tools.py:65): the same global matrix must give the same
        # values on any number of GPUs (strong leg at N ranks vs main leg at 1 rank)
        info.sigma_head = [float(x) * float(np.sqrt(max(A.n_total - 1, 1))) for x in ad.uns["lsi"]["stdev"][:4]]
        if keep is not None:
            keep["ad"] = ad
        return info
    return step


DUMP_BYTES = 16 << 20      # per dumped array: the four arrays of dump_outputs stay under 64 MB


def dump_outputs(out_dir, ad):
    """Write the slots one step of the main leg leaves for its caller, so that two builds can be compared output for
    output.  Arrays up to DUMP_BYTES are written whole.  Of a larger one, a fixed sample of rows (seed 0, ascending
    order) is written, so every run with the same arguments writes the same positions.
      uns_lsi_stdev   uns["lsi"]["stdev"]                          (k,)
      obsm_X_lsi      rows of obsm["X_lsi"]                         (cells, k)
      varm_LSI        rows of varm["LSI"]                           (peaks, k)
      X_data          stored TF-IDF values of X (kept in HBM)       (entries,)
    The sign of each LSI component is arbitrary and can differ from run to run, so embedding and loading columns are
    flipped together to make the largest-magnitude entry of each full loading column positive (the loadings are the
    same on every rank).  Returns {name: shape}."""
    import torch
    rng = np.random.default_rng(0)

    def rows(n, row_bytes):
        m = max(1, DUMP_BYTES // row_bytes)
        return np.arange(n) if n <= m else np.sort(rng.choice(n, m, replace=False))

    X, emb, load = ad.X, ad.obsm["X_lsi"], ad.varm["LSI"]
    sgn = np.where(load[np.abs(load).argmax(0), np.arange(load.shape[1])] < 0, -1, 1).astype(load.dtype)
    pos = torch.from_numpy(rows(X.nnz, X.data.element_size())).to(X.device)
    out = {"uns_lsi_stdev": ad.uns["lsi"]["stdev"],
           "obsm_X_lsi": emb[rows(emb.shape[0], emb.itemsize * emb.shape[1])] * sgn,
           "varm_LSI": load[rows(load.shape[0], load.itemsize * load.shape[1])] * sgn,
           "X_data": X.data[pos].cpu().numpy()}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
    return {name: list(a.shape) for name, a in out.items()}


def spmm_roofline(ctx, kern, info, steps, nnz, n_local, D, k, clocks):
    """roofline block of the dominant kernel from the CUDA-event times of its launches inside the timed region."""
    import muon_b200 as mu
    f32_ms = kern.get("mub_spmm_csr_f32", []) + kern.get("mub_spmm_csrp_f32", [])
    h16_ms = kern.get("mub_spmm_csr_h16", []) + kern.get("mub_spmm_csrp_h16", [])
    P = mu._device.pad_width(min(k + 8, 128))
    # one "pass" = one product with A or A^T over all nnz of the shard (A^T runs as several row-panel launches).
    # Algorithmic bytes per pass (SURVEY 8d): 8 B/nnz + the dense operands once (fp32 by the SURVEY's model,
    # also for the half-operand passes: the same algorithmic work done with fewer bytes moved).
    pass_bytes = 8.0 * nnz + 4.0 * P * (n_local + D)
    n_pass = info.passes * steps
    n_lowp = getattr(info, "lowp_passes", 0) * steps
    total = float(np.sum(f32_ms) + np.sum(h16_ms)) if (f32_ms or h16_ms) else float("nan")
    pk, pk_kind = peaks()
    hbm = float(pk.get("hbm_gbs", 6650.0))
    ach = n_pass * pass_bytes / (total * 1e-3) / 1e9 if total == total else None
    r = {"bound": "hbm",
         "kernel": f"spmm_csr_rowwarp_kernel<{P},*> + spmm_csr_rowwarp_h_kernel<{P},*> (A*V on CSR arrays, A^T*U on pair-layout panels)",
         "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": (ach / hbm) if ach else None, "traffic": None,
         "peak_kind": pk_kind, "launches": len(f32_ms) + len(h16_ms), "passes": n_pass, "passes_half_operand": n_lowp,
         "ms_per_pass": total / max(n_pass, 1), "bytes_per_pass": pass_bytes,
         "ms_per_pass_f32": float(np.sum(f32_ms)) / max(n_pass - n_lowp, 1) if f32_ms else None,
         "ms_per_pass_h16": float(np.sum(h16_ms)) / max(n_lowp, 1) if h16_ms else None,
         "note": "algorithmic bytes = 8 B/nnz + 4*P*(n+D) per pass; every nnz also gathers P operand elements "
                 "through L2->L1 (4 B each in the fp32 kernel, 2 B in the half-operand kernel), which is the practical "
                 "limiter (DESIGN.md section 4)"}
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        key = f"spmm_rowwarp{P}_n{n_local}_d{D}"
        if key in tr:
            r["traffic"] = tr[key]["dram_bytes_per_pass"]
            r["traffic_source"] = tr[key]["source"]
    except Exception:
        pass
    if ctx.rank == 0 and clocks and total == total:
        import torch
        sms = torch.cuda.get_device_properties(ctx.local).multi_processor_count
        if f32_ms:
            r["onchip"] = onchip_roofline(nnz, P, r["ms_per_pass_f32"], clocks.get("sm_mhz"), sms, 4.0)
        if h16_ms:
            r["onchip_h16"] = onchip_roofline(nnz, P, r["ms_per_pass_h16"], clocks.get("sm_mhz"), sms, 2.0)
    return r


def host_ram_limit(ctx, bytes_per_cell, n_want):
    """Largest cells-per-GPU for the e2e legs such that every rank's host matrices fit the host's available RAM."""
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        return n_want, None
    budget = 0.6 * avail / max(ctx.local_world, 1)
    n_fit = int(budget // bytes_per_cell)
    return min(n_want, max(n_fit, 1000)), avail


def main():
    args = parse()
    if args.topics <= 0:
        args.topics = max(64, args.k + 14)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist

    import muon_b200 as mu
    from muon_b200 import _device, _lib
    from muon_b200._synth import generate_device, make_tables

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback in the product path)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def note(tag, obj):
        """progress on stderr (rank 0): a failing side leg must not cost the numbers of the legs before it"""
        if rank == 0:
            print(f"[bench] {tag}: {json.dumps(obj, default=str)[:1500]}", file=sys.stderr, flush=True)

    ctx = Ctx()
    ctx.world, ctx.rank, ctx.local = world, rank, local
    ctx.local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    ctx.barrier = barrier

    def free():
        gc.collect()
        torch.cuda.empty_cache()

    D, k = args.peaks, args.k
    n_local = args.cells if args.scaling == "weak" else -(-args.cells // world)
    n_total = n_local * world
    tb = make_tables(D, args.density, args.topics, args.seed)
    A = generate_device(n_local, D, args.density, tables=tb, row0=rank * n_local, n_total=n_total)
    nnz = A.nnz
    torch.cuda.synchronize()

    # ---- main leg: device-resident counts -> tfidf -> lsi ------------------------------------------------------
    step = lsi_step_fn(ctx, A, k, args.tol)
    last = {} if args.dump_outputs else None
    ms_total, kern, launches, info, clocks = timed_steps(ctx, lambda: step(last), args.steps, args.warmup,
                                                         sample_clocks=True)
    if last is not None:
        if rank == 0:
            note("dump_outputs", {"dir": args.dump_outputs, "arrays": dump_outputs(args.dump_outputs, last["ad"])})
        last.clear()
    value = n_total * args.steps / (ms_total / 1e3)
    roofline = spmm_roofline(ctx, kern, info, args.steps, nnz, n_local, D, k, clocks)
    pk, _ = peaks()
    hbm = float(pk.get("hbm_gbs", 6650.0))
    tf_red = kern.get("mub_tfidf_reduce_f32", []) + kern.get("mub_tfidf_reduce_tiled_f32", [])
    tf_app = kern.get("mub_tfidf_apply_f32", [])
    if tf_red and tf_app:
        t = float(np.mean(tf_red) + np.mean(tf_app))
        roofline["tfidf"] = {"achieved": 20.0 * nnz / (t * 1e-3) / 1e9, "unit": "GB/s", "ms": t,
                             "ms_reduce": float(np.mean(tf_red)), "ms_apply": float(np.mean(tf_app)),
                             "frac": 20.0 * nnz / (t * 1e-3) / 1e9 / hbm,
                             "kernels": "tfidf_reduce_tiled_kernel (8 B/nnz) + tfidf_apply_kernel (12 B/nnz)"
                             if "mub_tfidf_reduce_tiled_f32" in kern else "tfidf_reduce_kernel + tfidf_apply_kernel"}
    phase_ms = {name: float(np.sum(v)) / args.steps for name, v in kern.items()}
    note("main", {"value": value, "ms_per_step": ms_total / args.steps, "passes": info.passes,
                  "lowp": getattr(info, "lowp_passes", 0), "history": info.history, "roofline": roofline, "phase_ms": phase_ms})

    breakdown = None
    if args.breakdown:
        _lib.PHASES = {}
        with _lib.phase("total"):
            step()
        breakdown = {kk: round(1e3 * v, 2) for kk, v in _lib.PHASES.items()}
        _lib.PHASES = None

    # ---- strong-scaling leg (N > 1): the same step with --cells TOTAL split over the ranks ------------------------
    strong = None
    if world > 1 and args.scaling == "weak" and not args.no_strong:
        ns = -(-args.cells // world)
        As = generate_device(ns, D, args.density, tables=tb, row0=rank * ns, n_total=ns * world)
        ms_s, kern_s, _, info_s, _ = timed_steps(ctx, lsi_step_fn(ctx, As, k, args.tol), args.steps, max(args.warmup, 1))
        note("strong", {"ms_per_step": ms_s / args.steps})
        strong = {"cells_total": ns * world, "cells_per_gpu": ns, "ms_per_step": ms_s / args.steps,
                  "sigma_head": getattr(info_s, "sigma_head", None),
                  "value": ns * world * args.steps / (ms_s / 1e3), "unit": "cells/s", "passes": info_s.passes,
                  "spmm_ms_per_step": float(np.sum([np.sum(v) for n_, v in kern_s.items() if "spmm" in n_])) / args.steps}
        del As
        free()

    # ---- same-matrix leg: the GPU on exactly the rows the CPU baseline is timed on (BASELINE.md 4.5) ---------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        S = min(args.sample_cells, n_local)
        Asmp = generate_device(S, D, args.density, tables=tb, row0=0, n_total=S)
        Xs = Asmp.get()
        ms_smp, _, _, info_smp, _ = timed_steps(ctx, lsi_step_fn(ctx, Asmp, k, args.tol), 3, 2)
        del Asmp
        t_tfidf, t_lsi = cpu_oracle_step(Xs, k)
        cpu = {"value": S / (t_tfidf + t_lsi), "unit": "cells/s", "cores": host_threads(), "kind": "port",
               "sample": f"first {S} cells x {D} peaks ({Xs.nnz} nnz); tfidf {t_tfidf:.2f}s + svds {t_lsi:.2f}s; "
                         "scipy sparse kernels are single-threaded, BLAS tail uses all cores",
               "tfidf_nnz_per_s": Xs.nnz / t_tfidf,
               "gpu_same_matrix_ms": ms_smp / 3, "gpu_same_matrix_passes": info_smp.passes,
               "same_matrix_speedup": (t_tfidf + t_lsi) / (ms_smp / 3e3)}
        del Xs
        note("cpu_baseline", cpu)

    # ---- e2e: same public calls on HOST matrices -------------------------------------------------------------------
    e2e, X, Xt = None, None, None
    want_mofa = not args.no_mofa
    if not args.no_e2e:
        import pandas as pd
        ne_want = n_local if args.e2e_cells < 0 else min(args.e2e_cells, n_local)
        # host bytes per cell while the leg runs: int64 indices + f32 counts + f32 tf-idf values (+ RNA for the MOFA leg)
        bpc = args.density * D * (8 + 4 + 4) + (0.07 * 30_000 * 12 if want_mofa else 0) + 1024
        ne, avail = host_ram_limit(ctx, bpc, ne_want)
        if world > 1:
            t_ne = torch.tensor([ne], dtype=torch.int64, device="cuda")
            dist.all_reduce(t_ne, op=dist.ReduceOp.MIN)
            ne = int(t_ne[0])
        Ae = A if ne == n_local else generate_device(ne, D, args.density, tables=tb, row0=rank * ne, n_total=ne * world)
        X = Ae.get()                                    # host scipy CSR (int64 indices when nnz >= 2^31)
        h2d = X.indptr.nbytes + 4 * X.nnz + X.data.nbytes    # int64 host indices are narrowed to int32 while staging
        d2h = X.data.nbytes + 4 * (ne * k + D * k + k)
        if Ae is not A:
            del Ae
        obs_df = pd.DataFrame(index=pd.RangeIndex(ne).astype(str))
        var_df = pd.DataFrame(index=pd.RangeIndex(D).astype(str))
        last = {}

        def step_host():
            last.clear()                                       # drops the previous step's result (and its device twin)
            ad = mu.SimpleAnnData(X, obs=obs_df, var=var_df)   # tfidf rebinds ad.X; X itself is never modified
            t0 = time.perf_counter()
            mu.atac.pp.tfidf(ad)
            t1 = time.perf_counter()
            mu.atac.tl.lsi(ad, n_comps=k, tol=args.tol)
            t2 = time.perf_counter()
            last["tfidf_s"], last["lsi_s"], last["X"] = t1 - t0, t2 - t1, ad.X
            return float(ad.uns["lsi"]["stdev"][0])

        step_host()
        barrier()
        _device.HOST_TIMES = {}
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            step_host()
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        ht, _device.HOST_TIMES = _device.HOST_TIMES, None
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        per = float(dt[0]) / args.e2e_steps
        if "h2d_bytes" in ht:       # bytes the staging engine actually put on the bus (counts cross as uint8), + indptr
            h2d = int(ht.pop("h2d_bytes") / args.e2e_steps) + X.indptr.nbytes
        if "d2h_bytes" in ht:
            d2h = int(ht.pop("d2h_bytes") / args.e2e_steps) + 4 * k + (0 if ne * k * 4 > (8 << 20) else 4 * ne * k) + (0 if D * k * 4 > (8 << 20) else 4 * D * k)
        bd = {kk: v / args.e2e_steps for kk, v in ht.items()}
        bd.update({"tfidf_call_s": last["tfidf_s"], "lsi_call_s": last["lsi_s"],
                   "host_other_s": max(0.0, per - last["tfidf_s"] - last["lsi_s"])})
        e2e = {"value": ne * world / per, "unit": "cells/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "cells_per_gpu": ne, "steps": args.e2e_steps,
               "ms_per_step": 1e3 * per, "breakdown_s": {kk: round(v, 3) for kk, v in bd.items()},
               "copy_threads": _device.copy_threads(), "host_ram_available_gb": round(avail / 2**30, 1) if avail else None,
               "cells_limited_by_host_ram": ne < ne_want,
               "path": "scipy csr on host -> mu.atac.pp.tfidf -> mu.atac.tl.lsi -> numpy slots (breakdown: host wall "
                       "seconds; h2d_s/d2h_s = time inside the staging engine, fingerprint_s = twin validation)"}
        note("e2e", e2e)
        Xt = last.pop("X") if want_mofa else None          # host TF-IDF matrix: the ATAC view of the MOFA e2e leg
        last.clear()
        _device.release_all_resident()
        if Xt is not None:
            _device.release_resident(Xt)
        if not want_mofa:
            del X
            X = None

    # ---- configs[2]: mu.tl.mofa (RNA + ATAC, k=30, 15 iterations), cells sharded like the main leg ------------------
    mofa = None
    box = {"A": A, "Xt": Xt}                                    # ownership moves to the leg (it frees as it goes)
    del A, X, Xt
    if want_mofa:
        try:
            mofa = mofa_leg(ctx, args, box, tb, n_local, n_total, free)
        except Exception as e:                                  # the headline must survive a failure of a side leg
            mofa = {"error": f"{type(e).__name__}: {e}"[:400]}
    box.clear()
    free()

    # ---- configs[3]: LSI k=100 on 4M x 500k over 8 GPUs -------------------------------------------------------------
    cfg3 = None
    if args.cfg3 == 1 or (args.cfg3 < 0 and world == 8):
        try:
            cfg3 = cfg3_leg(ctx, args, free)
        except Exception as e:
            cfg3 = {"error": f"{type(e).__name__}: {e}"[:400]}

    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": "cells/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"TF-IDF + LSI k={k} on {n_local}x{D} ATAC ({args.density:.0%} nnz) per GPU",
                       "cells_total": n_total, "nnz_per_gpu": nnz, "parallelism": f"cells-sharded x{world}",
                       "l2": "inputs (8 B/nnz CSR stream) exceed L2 by >100x; no flush needed",
                       "lsi": {"block": info.block, "iterations": info.iterations, "passes": info.passes,
                               "passes_half_operand": getattr(info, "lowp_passes", 0),
                               "tol": args.tol, "converged": info.converged, "stalled": info.stalled,
                               "sigma_head": getattr(info, "sigma_head", None),
                               "sampled_stop": getattr(info, "sampled_stop", False),
                               "replica_repairs": getattr(info, "replica_repairs", 0),
                               "max_rel_residual": max(info.residuals),
                               "residual_history": [float("%.3g" % h) for h in info.history]}},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
            "phase_ms_per_step": phase_ms, "breakdown_ms": breakdown, "strong": strong, "mofa": mofa, "cfg3": cfg3,
        }
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
def mofa_leg(ctx, args, box, tb, n_local, n_total, free):
    """BASELINE configs[2].  A (device counts) is TF-IDF'd IN PLACE here (the LSI legs are over), the RNA view is
    generated next to it with non-integer (log-normalised) values, so both views are gaussian."""
    import torch

    import muon_b200 as mu
    from muon_b200 import _device
    from muon_b200._mofa import run_mofa_device
    from muon_b200._synth import generate_device, make_tables
    world, rank = ctx.world, ctx.rank
    K, iters = args.mofa_k, args.mofa_iters
    A, Xt_host = box.pop("A"), box.pop("Xt")
    nm = n_local if args.mofa_cells < 0 else min(args.mofa_cells, n_local)
    Nm = nm * world
    D_rna, dens_rna = 30_000, 0.07
    if nm != n_local:
        del A
        free()
        A = generate_device(nm, args.peaks, args.density, tables=tb, row0=rank * nm, n_total=Nm)
    atac = _device.tfidf_csr(A, inplace_values=True)
    tb_r = make_tables(D_rna, dens_rna, 64, 2)
    rna = _device.tfidf_csr(generate_device(nm, D_rna, dens_rna, tables=tb_r, row0=rank * nm, n_total=Nm), inplace_values=True)
    views = [rna, atac]
    nnzs = [v.nnz for v in views]
    Z0 = torch.from_numpy(np.random.RandomState(1).normal(size=(Nm, K))[rank * nm:(rank + 1) * nm])

    def step():
        return run_mofa_device(views, K, iters, Nm, Z0, check_convergence=False)
    ms, kern, launches, res, _ = timed_steps(ctx, step, 2, 1)
    ms_fit = ms / 2
    P = _device.pad_width(K)
    spmm_ms = float(np.sum(kern.get("mub_spmm_csr_f32", [])) + np.sum(kern.get("mub_spmm_csrp_f32", []))) / 2
    # SURVEY 8d: per iteration and view two sparse passes of 8 B/nnz + the dense operands once
    spmm_bytes = sum(2 * (8.0 * z + 4.0 * P * (nm + v.shape[1])) for z, v in zip(nnzs, views)) * iters
    pk, pk_kind = peaks()
    hbm = float(pk.get("hbm_gbs", 6650.0))
    ach = spmm_bytes / (spmm_ms * 1e-3) / 1e9 if spmm_ms > 0 else None
    out = {"metric": f"cells/sec for mu.tl.mofa (RNA {D_rna} genes + ATAC {args.peaks} peaks, k={K}, {iters} iterations)",
           "value": Nm / (ms_fit / 1e3), "unit": "cells/s", "ms_per_fit": ms_fit, "ms_per_iteration": ms_fit / iters,
           "cells_per_gpu": nm, "cells_total": Nm, "nnz_per_gpu": nnzs, "steps": 2, "warmup": 1, "gpu_launches": launches // 2,
           "roofline": {"bound": "hbm", "kernel": f"spmm_csr_rowwarp_kernel<{P},*>", "achieved": ach, "peak": hbm,
                        "unit": "GB/s", "frac": ach / hbm if ach else None, "peak_kind": pk_kind,
                        "ms_spmm_per_fit": spmm_ms, "bytes_per_fit": spmm_bytes},
           "elbo_first_last": [res["elbo"][0], res["elbo"][-1]],
           "elbo_monotone": bool(all(b >= a - 1e-9 * abs(a) for a, b in zip(res["elbo"], res["elbo"][1:]))),
           "kernel_ms_per_fit": {kk: float(np.sum(v)) / 2 for kk, v in kern.items()}}
    del res

    # e2e: mu.tl.mofa on a MuData of HOST scipy matrices (uploads inside the timed region, factors/loadings back)
    if Xt_host is not None and Xt_host.shape[0] == nm:
        import pandas as pd
        rna_h = rna.get()
        for v in views:
            v._tp = None                      # drop the cached transposes of the device leg: the e2e call builds its own
        del views, rna, atac, A
        free()
        obs = pd.DataFrame(index=pd.RangeIndex(nm).astype(str))
        md = mu.SimpleMuData({"rna": mu.SimpleAnnData(rna_h, obs=obs), "atac": mu.SimpleAnnData(Xt_host, obs=obs)})
        _device.release_all_resident()
        ctx.barrier()
        t0 = time.perf_counter()
        mu.tl.mofa(md, n_factors=K, n_iterations=iters, likelihoods="gaussian", use_var=None, convergence_mode="slow",
                   seed=1, quiet=True)
        ctx.barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        h2d = sum(m.indptr.nbytes + 4 * m.nnz + m.data.nbytes for m in (rna_h, Xt_host))
        d2h = 8 * (nm * K + (D_rna + args.peaks) * K)
        out["e2e"] = {"value": Nm / float(dt[0]), "unit": "cells/s", "ms_per_fit": 1e3 * float(dt[0]),
                      "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": 1,
                      "iterations_run": int(md.uns["mofa"]["_b200"]["iterations"]),
                      "path": "MuData of host scipy csr -> mu.tl.mofa -> obsm/varm/uns"}
        del md, rna_h
    # CPU baseline: the float64 oracle (oracle/mofa_ref.py; mofapy2 is not installable) on a bounded slice
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            from oracle.mofa_ref import mofa_ref
            from muon_b200._synth import generate_host
            from oracle.tfidf_ref import tfidf_ref
            Sc, Dr, Da = 2000, 3000, 20_000
            Y1 = tfidf_ref(generate_host(Sc, Dr, dens_rna, n_topics=64, seed=2)).toarray().astype(np.float64)
            Y2 = tfidf_ref(generate_host(Sc, Da, args.density, n_topics=64, seed=1)).toarray().astype(np.float64)
            Zs = np.random.RandomState(1).normal(size=(Sc, K))
            t0 = time.perf_counter()
            mofa_ref([Y1, Y2], K, iters, Z0=Zs, check_convergence=False)
            dtc = time.perf_counter() - t0
            out["cpu_baseline"] = {"value": Sc / dtc, "unit": "cells/s", "cores": host_threads(), "kind": "port",
                                   "sample": f"{Sc} cells x ({Dr} + {Da}) features dense float64 (oracle/mofa_ref.py, numpy/BLAS); "
                                             f"{dtc:.1f} s for {iters} iterations; cost per cell grows with the feature count, the "
                                             "benchmark has 10x more features",
                                   "cell_feature_products_per_s": Sc * (Dr + Da) * iters / dtc}
        except Exception as e:
            out["cpu_baseline"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    return out


def cfg3_leg(ctx, args, free):
    """BASELINE configs[3]: LSI k=100 on 4M cells x 500k peaks, 8 GPUs (500k cells per rank), 2 % nnz, 128 planted
    topics (T >= k+14, SURVEY App. E); Gram / A^T U allreduces over NVLink."""
    import torch
    from muon_b200._synth import generate_device, make_tables
    world, rank = ctx.world, ctx.rank
    n, D, k, dens, topics = 4_000_000 // max(world, 1) if world >= 8 else 500_000, 500_000, 100, 0.02, 128
    tb = make_tables(D, dens, topics, 3)
    A = generate_device(n, D, dens, tables=tb, row0=rank * n, n_total=n * world)
    ms, kern, launches, info, _ = timed_steps(ctx, lsi_step_fn(ctx, A, k, args.tol), 2, 1)
    spmm_ms = float(np.sum([np.sum(v) for n_, v in kern.items() if "spmm" in n_])) / 2
    out = {"workload": f"TF-IDF + LSI k={k} on {n * world}x{D} ATAC ({dens:.0%} nnz), {world} GPUs, {topics} topics",
           "value": n * world * 2 / (ms / 1e3), "unit": "cells/s", "ms_per_step": ms / 2, "steps": 2, "warmup": 1,
           "cells_per_gpu": n, "nnz_per_gpu": A.nnz, "passes": info.passes, "passes_half_operand": getattr(info, "lowp_passes", 0),
           "block": info.block, "converged": info.converged, "stalled": info.stalled,
           "residual_history": [float("%.3g" % h) for h in info.history], "spmm_ms_per_step": spmm_ms,
           "gpu_launches": launches // 2}
    del A
    free()
    return out


if __name__ == "__main__":
    main()
