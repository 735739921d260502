#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native DP fill (see BASELINE.json / SURVEY.md §8d).

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR

--dump-outputs writes what the timed path computed in its last step as DIR/<name>.npy (float32, or float64 where
float32 would round), so that two builds can be compared output for output on the same seeded inputs.

A "step" is one pass of the hot path over one batch: forward + reverse fill with packed
traceback and the near-optimal cell set for the C3 workload (100k synthetic protein pairs,
lengths 100-500, BLOSUM62, gi=12 ge=1, semi_local; seed 1003+rank).  Metric: GCUPS =
cell updates (Lq*Lt per direction, fwd+rev = 2 per matrix cell) / second / 1e9, whole job.

Legs of the default arm:
  value  device-timed (CUDA events), inputs already resident in HBM
  e2e    aadp_fill_batch through the C ABI from pinned HOST buffers, H2D + D2H inside the timing
  roofline / issue_roofline   dominant kernel, timed live with CUDA events on its stream
  cpu_baseline   the reference's own DPMatrix fill (oracle/_ref) on the host cores, bounded sample
The reference arm (--impl reference) times only the reference CPU implementation.
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
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GI, GE = 12.0, 1.0
DELTA = 0.01
METRIC = "GCUPS fwd+rev DP fill (near-optimal cell set + packed traceback)"


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.samples = []
        self.proc = None
        self.t = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.t = threading.Thread(target=self._read, daemon=True)
        self.t.start()

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1, _widened=False):
        sm, mx, reasons = [], 0.0, set()
        for ts, line in self.samples:
            if ts < t0 - 0.05 or ts > t1 + 0.05:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm and not _widened:
            # a timed region shorter than the sampling interval: take the samples of the second around it
            out = self.summary(t0 - 0.5, t1 + 0.5, True)
            out["note"] = "timed region shorter than the sampling interval: samples within 0.5 s of it"
            return out
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": mx or None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirname, rank, arrays):
    """Write each array as <dirname>/<name>.npy (rank > 0: <name>.rank<r>.npy).  Integers become float32 when every
    value is exact in float32, float64 otherwise."""
    conv = {}
    for name, arr in arrays.items():
        arr = np.asarray(arr)
        if arr.dtype == np.float32 or arr.dtype == np.uint8:
            arr = arr.astype(np.float32)
        elif arr.dtype.kind in "iu" and (arr.size == 0 or int(np.abs(arr).max()) < (1 << 24)):
            arr = arr.astype(np.float32)
        else:
            arr = arr.astype(np.float64)
        conv[name] = arr
    total = sum(a.nbytes for a in conv.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("--dump-outputs: %d bytes, more than the %d allowed" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(dirname, exist_ok=True)
    suffix = "" if rank == 0 else ".rank%d" % rank
    for name, arr in conv.items():
        np.save(os.path.join(dirname, name + suffix + ".npy"), arr)


def batch_outputs(ctx, a, what, d_f, d_r, d_t, d_c, seqs=None, pq=None, pt=None, sample_pairs=0):
    """What a caller of aadp_run_batch receives: the per-pair arrays it asked for and, for a fixed seeded sample of
    pairs, the resident matrices it can fetch with aadp_batch_fetch_pair (flattened and concatenated in sample order)."""
    out = {}
    if what & a.W_FWD:
        out["fwd_score"] = d_f.cpu().numpy()
    if what & a.W_REV:
        out["rev_score"] = d_r.cpu().numpy()
    if what & a.W_MASK:
        out["threshold"] = d_t.cpu().numpy()
        out["nearopt_count"] = d_c.cpu().numpy()
    if sample_pairs and (what & a.W_TB):
        n = len(pq)
        ids = np.sort(np.random.default_rng(0).choice(n, min(sample_pairs, n), replace=False))
        parts = {}
        for p in ids:
            Lq, Lt = len(seqs[pq[p]]), len(seqs[pt[p]])
            # without W_SCORES the reverse score matrix is never materialised: reverse traceback only
            got = ctx.fetch_pair(int(p), Lq, Lt, fwd=True, rev=False, mask=bool(what & a.W_MASK))
            got.update({k: v for k, v in ctx.fetch_pair(int(p), Lq, Lt, fwd=False, rev=True, scores=False).items()
                        if v is not None})
            for k, v in got.items():
                if v is not None:
                    parts.setdefault(k, []).append(v.ravel())
        out["sample_pair_ids"] = ids
        for k, v in parts.items():
            out["sample_" + k] = np.concatenate(v)
    return out


def make_workload(rank, npairs):
    from alignment_algos_b200 import synth
    return synth.pair_workload(1003 + rank, npairs, 100, 500)


def reference_timer(seqs, pq, pt, budget_s, nthreads, what=3):
    """Time the reference's own DPMatrix fill (oracle/_ref when present, else the C port) on a
    bounded sample of the workload.  Returns dict(value GCUPS, cores, kind, sample, seconds)."""
    from oracle import pyoracle as po
    import alignment_algos_b200 as a
    alpha, M = a.blosum62()
    have_ref = os.path.exists(po.LIB_REF)
    ncell = lambda idx: float(sum(len(seqs[pq[p]]) * len(seqs[pt[p]]) for p in idx))
    if have_ref:
        R = po.Reference(alpha, M, GI, GE, po.SEMI_LOCAL)
        run = lambda idx: R.time_fills(seqs, [pq[p] for p in idx], [pt[p] for p in idx], what, nthreads)[0]
        kind = "reference"
    else:
        O = po.Oracle(M, GI, GE, po.SEMI_LOCAL)
        nthreads = 1

        def run(idx):
            t0 = time.perf_counter()
            for p in idx:
                O.fill(seqs[pq[p]], seqs[pt[p]], po.FWD)
                if what & 2:
                    O.fill(seqs[pq[p]], seqs[pt[p]], po.REV)
            return time.perf_counter() - t0
        kind = "port"
    # calibrate on one pair per thread, then size the sample to the budget
    cal = list(range(min(nthreads, len(pq))))
    t_cal = max(run(cal), 1e-3)
    per_pair = t_cal  # seconds per "round" of nthreads pairs
    rounds = max(1, int(budget_s / per_pair))
    n = min(len(pq), rounds * nthreads)
    idx = list(range(n))
    sec = run(idx)
    cells = ncell(idx)
    ndir = 2 if (what & 2) else 1
    return {"value": cells * ndir / sec / 1e9, "unit": "GCUPS", "cores": nthreads, "kind": kind,
            "sample": "first %d pairs of the workload (%.3g cell updates x%d directions) in %.2f s" % (n, cells, ndir, sec),
            "seconds": sec, "pairs": n}


def fair_cpu_timer(seqs, pq, pt, budget_s, what=3):
    """The O(mn) three-state restatement of the same recurrence (oracle/aadp_oracle.c, `fast` fill: scores + traceback,
    both directions) on ONE host thread and on ALL host cores, over a bounded sample of the workload: the CPU baseline
    with the reference's O(n) algorithmic handicap removed (BASELINE.md §3)."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import pyoracle as po
    import alignment_algos_b200 as a
    alpha, M = a.blosum62()
    O = po.Oracle(M, GI, GE, po.SEMI_LOCAL)
    ndir = 2 if (what & 2) else 1

    def one(p):
        O.fill(seqs[pq[p]], seqs[pt[p]], po.FWD, True, fast=True)
        if what & 2:
            O.fill(seqs[pq[p]], seqs[pt[p]], po.REV, True, fast=True)
        return float(len(seqs[pq[p]])) * float(len(seqs[pt[p]]))

    t0 = time.perf_counter()
    one(0)
    per = max(time.perf_counter() - t0, 1e-4)
    n1 = int(max(8, min(len(pq), budget_s / per)))
    t0 = time.perf_counter()
    cells1 = sum(one(p) for p in range(n1))
    s1 = time.perf_counter() - t0
    ncores = os.cpu_count() or 1
    nall = int(min(len(pq), n1 * ncores))
    t0 = time.perf_counter()
    with ThreadPoolExecutor(ncores) as ex:  # the C fill releases the GIL (ctypes)
        cellsN = sum(ex.map(one, range(nall), chunksize=max(1, nall // (ncores * 8))))
    sN = time.perf_counter() - t0
    return {"unit": "GCUPS", "kind": "port, O(mn) restatement (oracle fast fill: scores + traceback)",
            "value_1_thread": cells1 * ndir / s1 / 1e9, "value": cellsN * ndir / sN / 1e9, "cores": ncores,
            "sample": "first %d pairs on 1 thread in %.2f s; first %d pairs on %d threads in %.2f s" % (n1, s1, nall, ncores, sN)}


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    seqs, pq, pt = make_workload(0, 4096)
    ncores = os.cpu_count() or 1
    budget = 8.0
    vals = []
    for _ in range(args.warmup):
        reference_timer(seqs, pq, pt, 1.0, ncores)
    last = None
    t0 = time.perf_counter()
    for _ in range(args.steps):
        last = reference_timer(seqs, pq, pt, budget, ncores)
        vals.append(last["value"])
    wall = time.perf_counter() - t0
    v = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "GCUPS", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": wall / max(args.steps, 1) * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "c3: synthetic protein pairs L in [100,500], BLOSUM62 gi=12 ge=1 semi_local, fwd+rev "
                               "DPMatrix fill; bounded sample per step (the reference is O(n^3))"},
        "cpu_baseline": {"value": v, "unit": "GCUPS", "cores": last["cores"], "kind": last["kind"], "sample": last["sample"]},
        "e2e": {"value": v, "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_c4(args, rank, local_rank, world, barrier, max_over_ranks, sum_over_ranks, emit=True, steps=None, warmup=None):
    """C4: all-vs-all of N synthetic sequences (every unordered pair i<j, query=i, template=j), forward
    score only, through the cross-mode entry points.  The upper triangle is cut into rectangles
    (shard.triangle_rects) which are dealt over the ranks: STRONG scaling, no data-path collective."""
    import torch
    import alignment_algos_b200 as a
    from alignment_algos_b200 import shard, synth
    if steps is not None:
        args = argparse.Namespace(**dict(vars(args), steps=steps, warmup=warmup))
    alpha, M = a.blosum62()
    rng = np.random.default_rng(1004)
    seqs = synth.random_seqs(rng, args.seqs, 100, 500)
    lens = np.array([len(x) for x in seqs], np.int64)
    res, off = a.Context.pack(seqs)
    blk = shard.choose_block(args.seqs, world)
    rects = shard.shard_rects(shard.triangle_rects(args.seqs, blk, max(blk // 4, 1)), lens, world)[rank]
    # useful work of the whole job: sum over i<j of Li*Lj
    tot = float(lens.sum())
    useful_cu = (tot * tot - float((lens.astype(np.float64) ** 2).sum())) / 2.0
    n_pairs_job = args.seqs * (args.seqs - 1) // 2
    sizes = [(r[1] - r[0]) * (r[3] - r[2]) for r in rects]
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    d_scores = torch.empty(int(offs[-1]), dtype=torch.float32, device="cuda")
    h_scores = torch.empty(int(offs[-1]), dtype=torch.float32).pin_memory()
    res_p = torch.from_numpy(res.copy()).pin_memory()
    off_p = torch.from_numpy(off.copy()).pin_memory()
    ctx = a.Context(local_rank)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    ctx.set_scoring(M, GI, GE, a.SEMI_LOCAL)
    ids = np.arange(args.seqs, dtype=np.int32)
    ctx.upload_sequences(res_p.numpy(), off_p.numpy())
    computed_cu = [0.0]
    launches = [0]

    def step_resident():
        cu, ln = 0.0, 0
        for k, (q0, q1, t0, t1) in enumerate(rects):
            ctx.cross_run(ids[q0:q1], ids[t0:t1], d_scores.data_ptr() + 4 * int(offs[k]))
            cu += ctx.last_cross_cell_updates()
            ln += ctx.last_launch_count()
        computed_cu[0], launches[0] = cu, ln

    for _ in range(args.warmup):
        step_resident()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    ctx.set_profiling(True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.time()
    e0.record(stream)
    for _ in range(args.steps):
        step_resident()
    e1.record(stream)
    barrier()
    w1 = time.time()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    prof = ctx.profile()
    ctx.set_profiling(False)
    if emit and args.dump_outputs:
        # the score blocks of this rank's rectangles, concatenated: a fixed seeded sample of them
        n_sc = d_scores.numel()
        idx = np.unique(np.random.default_rng(0).integers(0, n_sc, 1 << 20)) if n_sc else np.zeros(0, np.int64)
        dump_outputs(args.dump_outputs, rank, {
            "scores_sample": d_scores[torch.from_numpy(idx).cuda()].cpu().numpy(), "scores_sample_index": idx})
    value = useful_cu * args.steps / (ms_total * 1e-3) / 1e9
    # ---- end to end: sequences from pinned host memory, every score block back to the host
    def step_e2e():
        ctx.upload_sequences(res_p.numpy(), off_p.numpy())
        step_resident()
        h_scores.copy_(d_scores, non_blocking=True)
        stream.synchronize()
    step_e2e()
    barrier()
    x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    x0.record(stream)
    for _ in range(args.steps):
        step_e2e()
    x1.record(stream)
    barrier()
    e2e_ms = max_over_ranks(x0.elapsed_time(x1))
    sampler.stop()
    clocks = sampler.summary(w0, w1)
    # spot check inside the bench: the two roles of a symmetric scoring scheme give the same optimum
    k = next((i for i, r in enumerate(rects) if shard.rect_is_diagonal(r)), None)
    if k is not None:
        q0, q1, t0, t1 = rects[k]
        blk = h_scores[int(offs[k]):int(offs[k + 1])].numpy().reshape(q1 - q0, t1 - t0)
        assert np.array_equal(blk, blk.T), "all-vs-all block is not symmetric"
    kms = sum(ms for _, ms, _ in prof)
    kcells = sum(c for _, _, c in prof)
    hbm_peak, peak_src, sm_max = load_peaks()
    props = torch.cuda.get_device_properties(local_rank)
    clk = (clocks["sm_mhz"] or sm_max) * 1e6
    i_alg = 7.0  # SURVEY.md §8d instruction model of a score-only cell update
    lane_peak = props.multi_processor_count * 128 * clk
    dom_gcups = kcells / max(kms * 1e-3, 1e-9) / 1e9
    # algorithmic HBM bytes: the residues of both sequences in, 4 bytes out, per pair
    bytes_per_cu = (2 * float(lens.mean()) + 4.0) / float(lens.mean()) ** 2
    line = {
        "metric": "GCUPS forward score-only DP fill, all-vs-all", "value": value, "unit": "GCUPS", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "i16", "data": "synthetic",
        "config": {"workload": "c4: all-vs-all of %d synthetic sequences (%d pairs i<j), L in [100,500], BLOSUM62 gi=12 ge=1 "
                               "semi_local, forward score-only, cross-mode packed kernel" % (args.seqs, n_pairs_job),
                   "rectangles_this_rank": len(rects), "cache": "each launch streams its own sequences; scores are written once",
                   "sharding": "upper-triangle rectangles dealt over ranks (LPT by cells), no collective on the data path",
                   "computed_over_useful": sum_over_ranks(computed_cu[0]) / useful_cu},
        "pairs_per_s": n_pairs_job * args.steps / (ms_total * 1e-3),
        "clocks": clocks,
        "e2e": {"value": useful_cu * args.steps / (e2e_ms * 1e-3) / 1e9, "unit": "GCUPS", "h2d_bytes_per_step": int(res.nbytes + off.nbytes),
                "d2h_bytes_per_step": int(h_scores.numel() * 4), "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": int(launches[0] * args.steps),
        "roofline": {"bound": "hbm", "kernel": "packed_kernel<TB=0,FST=0,MSK=0,XM=1>fwd", "achieved": dom_gcups * bytes_per_cu,
                     "peak": hbm_peak, "unit": "GB/s", "frac": dom_gcups * bytes_per_cu / hbm_peak, "traffic": None,
                     "peak_source": peak_src, "bytes_per_cell_update": bytes_per_cu,
                     "note": "score-only: HBM is not the binding roofline, see issue_roofline"},
        "issue_roofline": {"kernel": "packed_kernel<TB=0,FST=0,MSK=0,XM=1>fwd", "i_alg": i_alg, "lane_ops_per_s": lane_peak,
                           "ceiling_gcups": lane_peak / i_alg / 1e9, "achieved_gcups": dom_gcups,
                           "frac": dom_gcups / (lane_peak / i_alg / 1e9), "sm_mhz": clk / 1e6},
    }
    if rank == 0 and emit:
        print(json.dumps(line), flush=True)
    ctx.close()
    return line


def quick_pairlist(workload, args, rank, local_rank, world, barrier, max_over_ranks, sum_over_ranks, steps, warmup,
                   dump_dir=None):
    """Device-timed value of one of the pair-list workloads (inputs resident), for the `extra` keys of the default
    line: c2 (10k pairs forward score-only) and c5 (one 30k x 30k pair fwd+rev+traceback+mask, one replica per rank)."""
    import torch
    import alignment_algos_b200 as a
    from alignment_algos_b200 import synth
    alpha, M = a.blosum62()
    gi, ge = GI, GE
    if workload == "c2":
        seqs, pq, pt = synth.pair_workload(1002 + rank, 10_000, 100, 500)
        what = a.W_FWD
    elif workload == "c3f":
        # the C3 shape under the reference's DEFAULT penalties (alib.cpp:17-18): off the dyadic grid, so the exact fp32
        # general-gap path runs (record-list kernel, 0 ulp); scores + near-optimal counts, no resident traceback
        seqs, pq, pt = synth.pair_workload(1003 + rank, 20_000, 100, 500)
        what = a.W_FWD | a.W_REV | a.W_MASK
        gi, ge = 4.73, 0.34
    else:
        rng = np.random.default_rng(1005 + rank)
        seqs = [rng.integers(0, 20, args.long_len).astype(np.uint8) for _ in range(2)]
        pq, pt = np.array([0], np.int32), np.array([1], np.int32)
        what = a.W_FWD | a.W_REV | a.W_TB | a.W_MASK
    res, off = a.Context.pack(seqs)
    ctx = a.Context(local_rank)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    ctx.set_scoring(M, gi, ge, a.SEMI_LOCAL)
    n = len(pq)
    d_f = torch.empty(n, dtype=torch.float32, device="cuda")
    d_r = torch.empty(n, dtype=torch.float32, device="cuda")
    d_t = torch.empty(n, dtype=torch.float32, device="cuda")
    d_c = torch.empty(n, dtype=torch.int64, device="cuda")
    ctx.upload_batch(res, off, pq, pt, what)
    for _ in range(warmup):
        ctx.run_batch(what, DELTA, d_f.data_ptr(), d_r.data_ptr(), d_t.data_ptr(), d_c.data_ptr())
    torch.cuda.synchronize()
    cu_step = ctx.last_cell_updates()
    ctx.set_profiling(True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        ctx.run_batch(what, DELTA, d_f.data_ptr(), d_r.data_ptr(), d_t.data_ptr(), d_c.data_ptr())
    e1.record(stream)
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    prof = ctx.profile()
    ctx.set_profiling(False)
    if dump_dir:
        dump_outputs(dump_dir, rank, batch_outputs(ctx, a, what, d_f, d_r, d_t, d_c))
    if (what & a.W_REV) and workload != "c3f":  # (fp32 scoring: the two directions round differently)
        assert torch.equal(d_f, d_r), "forward and reverse optima differ"
    by = {}
    for name, kms, cells in prof:
        d = by.setdefault(name, [0.0, 0.0])
        d[0] += kms
        d[1] += cells
    out = {"value": sum_over_ranks(cu_step) * steps / (ms * 1e-3) / 1e9, "unit": "GCUPS", "ms_per_step": ms / steps,
           "steps": steps, "scaling": "weak (one replica per rank)" if workload == "c5" else "weak",
           "kernel_ms_per_step": {k: v[0] / steps for k, v in by.items()}}
    if workload == "c3f":
        out["pairs_per_s"] = sum_over_ranks(n) * steps / (ms * 1e-3)
        out["workload"] = "c3 shape (20000 pairs per GPU, L in [100,500]), BLOSUM62 with the reference's default gi=4.73 ge=0.34, semi_local: exact fp32 general-gap fill fwd+rev + near-optimal counts"
        out["dtype"] = "f32"
        ctx.close()
        return out
    dom = max(((k, v) for k, v in by.items() if v[1] > 0), key=lambda kv: kv[1][0], default=None)
    if dom:
        bpc = kernel_bytes_per_cu(dom[0], what)
        hbm_peak, peak_src, _ = load_peaks()
        gcups = dom[1][1] / (dom[1][0] * 1e-3) / 1e9
        out["roofline"] = {"bound": "hbm", "kernel": dom[0], "achieved": gcups * bpc, "peak": hbm_peak, "unit": "GB/s",
                           "frac": gcups * bpc / hbm_peak, "bytes_per_cell_update": bpc, "kernel_gcups": gcups}
    ctx.close()
    return out


def kernel_bytes_per_cu(kernel, what):
    """Algorithmic HBM bytes per cell update of a fill kernel (DESIGN.md §6; SURVEY.md §8d):
    packed forward + traceback + score spill: 0.5 B traceback + 2 B int16 score written            = 2.5
    packed reverse + traceback + fused mask:  0.5 B traceback + 2 B int16 score read + 1/8 B mask  = 2.625
    long-pair wavefront (int32 scores):       0.5 B traceback + 4 B score written                  = 4.5
    score-only kernels: residues in, one score out per pair."""
    import re
    if "wave" in kernel:
        return 4.5
    score_only = (2 * 300.0 + 4.0) / 300.0 ** 2
    m = re.search(r"packed_kernel<TB=(\d),FST=(\d),MSK=(\d)", kernel)
    if m:
        tb, fst, msk = (int(x) for x in m.groups())
        if msk:
            return 0.5 * tb + 2.0 + 0.125 + 2.0 * fst
        b = 0.5 * tb + 2.0 * fst
        return b if b > 0 else score_only
    m = re.search(r"fill_kernel<K=\d+,TB=(\d),ST=(\d)", kernel)
    if m:
        tb, st = int(m.group(1)), int(m.group(2))
        b = 0.5 * tb + 2.0 * st
        return b if b > 0 else score_only
    return score_only


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--pairs", type=int, default=100_000, help="pairs per GPU (C3 = 100000)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e-overlap", action="store_true", help="skip the three-context end-to-end leg")
    ap.add_argument("--seqs", type=int, default=20_000, help="sequences of the all-vs-all workload (C4 = 20000)")
    ap.add_argument("--workload", default="c3", choices=["c3", "c2", "c4", "c5", "c3f"],
                    help="c3 (default, the headline): 100k pairs fwd+rev+traceback+mask; c2: 10k pairs forward "
                         "score-only; c4: all-vs-all of --seqs sequences, forward score-only, strong scaling over ranks; "
                         "c5: one 30k x 30k pair fwd+rev+traceback+mask (multi-CTA wavefront)")
    ap.add_argument("--long-len", type=int, default=30000)
    ap.add_argument("--no-extras", action="store_true",
                    help="default (c3) run only: skip the `extra` keys (C2, C4 strong scaling, C5, alignments end to end)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step as DIR/<name>.npy (at most 64 MB; "
                         "larger outputs as a fixed seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs the GPU implementation")
    rank, local_rank, world = env_int("RANK", 0), env_int("LOCAL_RANK", 0), env_int("WORLD_SIZE", 1)
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import torch.distributed as dist
    import alignment_algos_b200 as a

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- workload (synthetic, seeded; every rank owns its own C3-sized shard: weak scaling)
    alpha, M = a.blosum62()
    if args.workload == "c4":
        run_c4(args, rank, local_rank, world, barrier, max_over_ranks, sum_over_ranks)
        if world > 1:
            dist.destroy_process_group()
        return
    if args.workload == "c3f":  # the C3 shape under the reference's default (non-dyadic) penalties: exact fp32 path
        r = quick_pairlist("c3f", args, rank, local_rank, world, barrier, max_over_ranks, sum_over_ranks, args.steps, 1,
                           args.dump_outputs)
        if rank == 0:
            print(json.dumps({"metric": "GCUPS fwd+rev exact fp32 general-gap fill + near-optimal counts", "n_gpus": world,
                              "higher_is_better": True, "data": "synthetic", "vs_baseline": None, **r}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return
    if args.workload == "c3":
        seqs, pq, pt = make_workload(rank, args.pairs)
        what = a.W_FWD | a.W_REV | a.W_TB | a.W_MASK
        wl_desc = ("c3: %d synthetic protein pairs per GPU, L in [100,500], BLOSUM62 gi=12 ge=1 semi_local, "
                   "fwd+rev fill + packed traceback + near-optimal cell set (delta=0.01)" % args.pairs)
    elif args.workload == "c2":
        from alignment_algos_b200 import synth
        npairs = args.pairs if args.pairs != 100_000 else 10_000
        seqs, pq, pt = synth.pair_workload(1002 + rank, npairs, 100, 500)
        what = a.W_FWD
        wl_desc = ("c2: %d synthetic protein pairs per GPU, L in [100,500], BLOSUM62 gi=12 ge=1 semi_local, "
                   "forward score-only fill" % npairs)
    else:
        rng = np.random.default_rng(1005 + rank)
        seqs = [rng.integers(0, 20, args.long_len).astype(np.uint8) for _ in range(2)]
        pq, pt = np.array([0], np.int32), np.array([1], np.int32)
        what = a.W_FWD | a.W_REV | a.W_TB | a.W_MASK
        wl_desc = ("c5: one synthetic pair %d x %d, BLOSUM62 gi=12 ge=1 semi_local, fwd+rev fill + packed traceback "
                   "+ near-optimal cell set, multi-CTA anti-diagonal wavefront" % (args.long_len, args.long_len))
    res, off = a.Context.pack(seqs)
    # pinned host staging buffers (numpy views of torch pinned tensors) for the end-to-end leg
    def pinned(arr):
        t = torch.from_numpy(arr.copy()).pin_memory()
        return t, t.numpy()
    keep = []
    hb = {}
    for name, arr in (("res", res), ("off", off), ("pq", pq), ("pt", pt)):
        t, v = pinned(arr)
        keep.append(t)
        hb[name] = v

    ctx = a.Context(local_rank)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    ctx.set_scoring(M, GI, GE, a.SEMI_LOCAL)
    n = len(pq)
    d_f = torch.empty(n, dtype=torch.float32, device="cuda")
    d_r = torch.empty(n, dtype=torch.float32, device="cuda")
    d_t = torch.empty(n, dtype=torch.float32, device="cuda")
    d_c = torch.empty(n, dtype=torch.int64, device="cuda")

    ctx.upload_batch(hb["res"], hb["off"], hb["pq"], hb["pt"], what)

    def step_resident():
        ctx.run_batch(what, DELTA, d_f.data_ptr(), d_r.data_ptr(), d_t.data_ptr(), d_c.data_ptr())

    for _ in range(args.warmup):
        step_resident()
    torch.cuda.synchronize()
    cu_step = ctx.last_cell_updates()  # fwd + rev cell updates of this rank's batch
    launches_step = ctx.last_launch_count()

    # ---- leg 1: device-timed, inputs resident
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    ctx.set_profiling(True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.time()
    e0.record(stream)
    for _ in range(args.steps):
        step_resident()
    e1.record(stream)
    barrier()
    w1 = time.time()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    prof = ctx.profile()
    ctx.set_profiling(False)
    total_cu = sum_over_ranks(cu_step)
    value = total_cu * args.steps / (ms_total * 1e-3) / 1e9
    ms_per_step = ms_total / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rank, batch_outputs(ctx, a, what, d_f, d_r, d_t, d_c, seqs, pq, pt,
                                                           8 if args.workload == "c3" else 0))

    # correctness guard inside the bench: the two directions must agree on every optimum
    if what & a.W_REV:
        assert torch.equal(d_f, d_r), "forward and reverse optima differ"

    # ---- leg 2: end to end through the C ABI with host buffers
    for _ in range(2):
        out = ctx.fill_batch(hb["res"], hb["off"], hb["pq"], hb["pt"], what, DELTA)
    barrier()
    x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    x0.record(stream)
    for _ in range(args.steps):
        out = ctx.fill_batch(hb["res"], hb["off"], hb["pq"], hb["pt"], what, DELTA)
    x1.record(stream)
    barrier()
    w2 = time.time()
    e2e_ms = max_over_ranks(x0.elapsed_time(x1))
    e2e_value = total_cu * args.steps / (e2e_ms * 1e-3) / 1e9
    h2d, d2h = ctx.last_transfer_bytes()  # counted by the library from the copies it issues
    if what & a.W_REV:
        assert np.array_equal(out["fwd_score"], out["rev_score"])
    e2e_serial_ms = e2e_ms
    e2e_mode = "one context, one aadp_fill_batch call after the other"

    # ---- leg 2a: the same call followed by the product a caller of this path actually reads (optimal.h:47-75): the
    # optimal alignment of EVERY pair, traced on the GPU over the packed traceback (aadp_batch_optimal_all) and copied to
    # pinned host memory -- inputs H2D, alignments D2H, all inside the timed region
    e2e_ali = None
    if (what & a.W_TB) and (what & a.W_FWD):
        cap_rows = int(sum(len(seqs[pq[p]]) + len(seqs[pt[p]]) + 2 for p in range(n)))
        pairs_t = torch.empty((cap_rows, 2), dtype=torch.int32).pin_memory()
        n_t = torch.empty(n, dtype=torch.int32).pin_memory()
        st_t = torch.empty(n, dtype=torch.int32).pin_memory()
        asteps = args.steps

        def step_ali():
            ctx.fill_batch(hb["res"], hb["off"], hb["pq"], hb["pt"], what, DELTA)
            return ctx.optimal_all_compact(a.FWD, n, pairs=pairs_t.numpy())

        step_ali()
        barrier()
        z0, z1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        z0.record(stream)
        for _ in range(asteps):
            ao, ap_, an, ast_ = step_ali()
        z1.record(stream)
        barrier()
        ali_ms = max_over_ranks(z0.elapsed_time(z1))
        assert int(ast_.max()) == 0 and int(an.min()) >= 2
        e2e_ali = {"value": total_cu * asteps / (ali_ms * 1e-3) / 1e9, "unit": "GCUPS", "ms_per_step": ali_ms / asteps,
                   "steps": asteps, "h2d_bytes_per_step": h2d,
                   "d2h_bytes_per_step": int(d2h + ctx.last_transfer_bytes()[1]),  # scalars + the alignment slots copied back
                   "aligned_pairs_per_step": int(an.astype(np.int64).sum()),
                   "what": "aadp_fill_batch + aadp_batch_optimal_all_compact(forward): every optimal alignment, packed, back in pinned host memory"}

    # ---- leg 2b: the same calls from THREE host threads over three contexts (independent contexts are thread-safe,
    # include/aadp.h), each on its own non-blocking stream: while the GPU fills the batch of one call, the other threads
    # schedule and upload theirs.  Every step still copies its own inputs H2D and its own results D2H inside the timed
    # region; the time is taken on the device (events on every stream, the latest one counts).
    if args.workload != "c5" and args.steps >= 3 and not args.no_e2e_overlap:
        import threading
        T = 3
        ctxs, streams = [], []
        for k in range(T):
            c = a.Context(local_rank)
            sk = torch.cuda.Stream()
            c.set_stream(sk.cuda_stream)
            c.set_scoring(M, GI, GE, a.SEMI_LOCAL)
            c.fill_batch(hb["res"], hb["off"], hb["pq"], hb["pt"], what, DELTA)
            ctxs.append(c)
            streams.append(sk)
        outs = [None] * T
        share = [args.steps // T + (1 if k < args.steps % T else 0) for k in range(T)]

        def worker(k):
            for _ in range(share[k]):
                outs[k] = ctxs[k].fill_batch(hb["res"], hb["off"], hb["pq"], hb["pt"], what, DELTA)

        torch.cuda.synchronize()
        barrier()
        y0 = torch.cuda.Event(enable_timing=True)
        y0.record(stream)
        for sk in streams:
            sk.wait_event(y0)
        th = [threading.Thread(target=worker, args=(k,)) for k in range(T)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        ends = []
        for sk in streams:
            e = torch.cuda.Event(enable_timing=True)
            e.record(sk)
            ends.append(e)
        torch.cuda.synchronize()
        barrier()
        ovl_ms = max_over_ranks(max(y0.elapsed_time(e) for e in ends))
        for k in range(T):
            assert np.array_equal(outs[k]["fwd_score"], out["fwd_score"])
            ctxs[k].close()
        if ovl_ms < e2e_ms:
            e2e_ms = ovl_ms
            e2e_value = total_cu * args.steps / (e2e_ms * 1e-3) / 1e9
            e2e_mode = "three contexts on three host threads, calls overlapped (each step with its own H2D and D2H)"
    # ---- leg 2c: the same overlap WITHOUT threads: one host thread drives two contexts through aadp_fill_batch_submit /
    # aadp_fill_batch_wait (include/aadp.h), results into pinned buffers; the host schedules batch k+1 while the GPU
    # fills batch k.  Reported as e2e.async_*; it becomes e2e.value when it is the best of the three modes.
    e2e_async = None
    if args.workload != "c5" and args.steps >= 4 and not args.no_e2e_overlap:
        T = int(os.environ.get("AADP_BENCH_ASYNC_CTX", "2"))
        actx, astreams, aouts = [], [], []
        for k in range(T):
            c = a.Context(local_rank)
            sk = torch.cuda.Stream()
            c.set_stream(sk.cuda_stream)
            c.set_scoring(M, GI, GE, a.SEMI_LOCAL)
            c.fill_batch(hb["res"], hb["off"], hb["pq"], hb["pt"], what, DELTA)
            o = {}
            for key, ty in (("fwd_score", torch.float32), ("rev_score", torch.float32), ("threshold", torch.float32), ("nearopt_count", torch.int64)):
                tpin = torch.zeros(n, dtype=ty).pin_memory()
                keep.append(tpin)
                o[key] = tpin.numpy()
            actx.append(c)
            astreams.append(sk)
            aouts.append(o)
        torch.cuda.synchronize()
        barrier()
        z0 = torch.cuda.Event(enable_timing=True)
        z0.record(stream)
        for sk in astreams:
            sk.wait_event(z0)
        inflight = [False] * T
        for it in range(args.steps):
            k = it % T
            if inflight[k]:
                actx[k].fill_batch_wait()
            actx[k].fill_batch_submit(hb["res"], hb["off"], hb["pq"], hb["pt"], what, DELTA, out=aouts[k])
            inflight[k] = True
        for k in range(T):
            if inflight[k]:
                actx[k].fill_batch_wait()
        ends = []
        for sk in astreams:
            e = torch.cuda.Event(enable_timing=True)
            e.record(sk)
            ends.append(e)
        torch.cuda.synchronize()
        barrier()
        async_ms = max_over_ranks(max(z0.elapsed_time(e) for e in ends))
        for k in range(T):
            assert np.array_equal(aouts[k]["fwd_score"], out["fwd_score"])
            actx[k].close()
        e2e_async = {"value": total_cu * args.steps / (async_ms * 1e-3) / 1e9, "ms_per_step": async_ms / args.steps,
                     "mode": "one host thread, %d contexts, aadp_fill_batch_submit / aadp_fill_batch_wait" % T}
        if async_ms < e2e_ms:
            e2e_ms = async_ms
            e2e_value = e2e_async["value"]
            e2e_mode = e2e_async["mode"] + " (each step with its own H2D and D2H)"
    sampler.stop()
    clocks = sampler.summary(w0, w1)

    # ---- dominant kernel + rooflines
    by = {}
    for name, ms, cells in prof:
        d = by.setdefault(name, [0.0, 0.0, 0])
        d[0] += ms
        d[1] += cells
        d[2] += 1
    fills = {k: v for k, v in by.items() if v[1] > 0}
    dom = max(fills.items(), key=lambda kv: kv[1][0]) if fills else ("none", [1.0, 0.0, 1])
    dom_ms = dom[1][0] / dom[1][2]
    dom_cells = dom[1][1] / dom[1][2]
    hbm_peak, peak_src, sm_max = load_peaks()
    # algorithmic bytes per cell update of the dominant fill kernel (DESIGN.md §6): per kernel, not one constant
    bytes_per_cu = kernel_bytes_per_cu(dom[0], what)
    achieved_gbs = dom_cells * bytes_per_cu / (dom_ms * 1e-3) / 1e9
    props = torch.cuda.get_device_properties(local_rank)
    clk = (clocks["sm_mhz"] or sm_max) * 1e6
    i_alg = 15.0 if (what & a.W_TB) else 7.0  # SURVEY.md §8d instruction model: with traceback / score-only
    lane_peak = props.multi_processor_count * 128 * clk
    dom_gcups = dom_cells / (dom_ms * 1e-3) / 1e9
    kernel_share = {k: v[0] / sum(x[0] for x in by.values()) for k, v in by.items()} if by else {}

    # measured DRAM traffic and executed instructions of that kernel: one `ncu --set full` capture of THIS build
    # (profiles/r02_kernel_counts.json, written by profiles/tools/ncu_counts.py from the .ncu-rep), scaled to this launch
    traffic, i_cell_sass, counts_src = None, None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_kernel_counts.json")))
        if dom[0] in tj["kernels"]:
            kc = tj["kernels"][dom[0]]
            traffic = kc["dram_bytes_per_cell_update"] * dom_cells
            i_cell_sass = kc["lane_ops_per_cell_update"]
            counts_src = tj.get("source")
    except Exception:
        pass
    line = {
        "metric": METRIC if args.workload != "c2" else "GCUPS forward score-only DP fill", "value": value, "unit": "GCUPS",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32" if args.workload == "c5" else "i16", "data": "synthetic",
        "config": {"workload": wl_desc,
                   "pairs_per_gpu": n, "cache": "outputs (%.1f GB/step) exceed L2; no flush needed" % (
                       (ctx.resident_bytes(a.W_TB) + ctx.resident_bytes(a.W_SCORES) + ctx.resident_bytes(a.W_MASK)) / 1e9),
                   "sharding": "independent pair shards per rank, no collective on the data path"},
        "pairs_per_s": sum_over_ranks(float(n)) * args.steps / (ms_total * 1e-3),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "GCUPS", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms / args.steps, "mode": e2e_mode,
                "serial_value": total_cu * args.steps / (e2e_serial_ms * 1e-3) / 1e9,
                "serial_ms_per_step": e2e_serial_ms / args.steps,
                **({"async_value": e2e_async["value"], "async_ms_per_step": e2e_async["ms_per_step"], "async_mode": e2e_async["mode"]}
                   if e2e_async else {})},
        "gpu_launches": int(launches_step * args.steps),
        "roofline": {"bound": "hbm", "kernel": dom[0], "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s",
                     "frac": achieved_gbs / hbm_peak, "traffic": traffic, "peak_source": peak_src,
                     "traffic_source": ("%s: ncu dram bytes per cell update x cell updates of this launch" % counts_src) if counts_src else None,
                     "bytes_per_cell_update": bytes_per_cu, "ms_per_launch": dom_ms,
                     "i_cell_sass": i_cell_sass},
        "issue_roofline": {"kernel": dom[0], "i_alg": i_alg, "lane_ops_per_s": lane_peak, "ceiling_gcups": lane_peak / i_alg / 1e9,
                           "achieved_gcups": dom_gcups, "frac": dom_gcups / (lane_peak / i_alg / 1e9), "sm_mhz": clk / 1e6},
        "kernel_share": kernel_share,
    }
    if e2e_ali:
        line["e2e_alignments"] = e2e_ali
    ctx.close()
    # ---- extra keys of the default (C3) line: the other headline configs, so that the driver's N = 1, 2, 4, 8 runs record
    # them too.  C2 and C5 run one replica per rank (weak); C4 is the all-vs-all job dealt over the ranks (STRONG scaling).
    if args.workload == "c3" and not args.no_extras:
        extra = {}
        try:
            extra["c2"] = quick_pairlist("c2", args, rank, local_rank, world, barrier, max_over_ranks, sum_over_ranks, 20, 5)
            extra["c5"] = quick_pairlist("c5", args, rank, local_rank, world, barrier, max_over_ranks, sum_over_ranks, 3, 2)
            extra["c3_float_default"] = quick_pairlist("c3f", args, rank, local_rank, world, barrier, max_over_ranks, sum_over_ranks, 2, 1)
            c4 = run_c4(args, rank, local_rank, world, barrier, max_over_ranks, sum_over_ranks, emit=False, steps=1, warmup=1)
            extra["c4"] = {k: c4[k] for k in ("metric", "value", "unit", "ms_per_step", "scaling", "pairs_per_s", "e2e", "issue_roofline")}
            extra["c4"]["workload"] = c4["config"]["workload"]
        except Exception as e:  # an extra must never take the headline line down
            extra["error"] = repr(e)
        line["extra"] = extra
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        if args.workload == "c5":  # the reference cannot run 30k x 30k (21.6 GB of DPCell, O(n^3)): C3-shaped sample
            seqs, pq, pt = make_workload(0, 2048)
        cb = reference_timer(seqs, pq, pt, 15.0, os.cpu_count() or 1, 3 if (what & a.W_REV) else 1)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        line["cpu_baseline_fair"] = fair_cpu_timer(seqs, pq, pt, 4.0, 3 if (what & a.W_REV) else 1)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
