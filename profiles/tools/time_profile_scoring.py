"""Position-specific template profiles (aadp_set_profile_scoring) against the substitution scoring they replace.

Two measurements in one run, both with IDENTITY profiles (prof[t][j-1, a] = BLOSUM62[a, t_j]), so that both scorings
compute the same numbers and the outputs are compared for equality:
  c3     C3-shaped batch: 100 k synthetic pairs, L in [100, 500], gi=12 ge=1 semi_local, fwd+rev+traceback+mask
         (aadp_fill_batch, host clock around the synchronous call), plus the per-kernel device times of one profiled run;
  cross  all-vs-all aadp_cross_run of 20 k synthetic sequences (forward scores into device memory, CUDA-synchronised).
The substitution and profile runs alternate, `--reps` times each after one warm-up.  No target is asserted.
usage: python profiles/tools/time_profile_scoring.py [--pairs 100000] [--seqs 20000] [--reps 3] [--out FILE.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np  # noqa: E402


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = q[0] if q else None
    except Exception as e:  # the measurement does not depend on it
        info["power_limit_and_max_sm_clock"] = "unavailable (%s)" % e
    return info


def kernel_ms(c, fn):
    c.set_profiling(True)
    fn()
    by = {}
    for name, ms, _ in c.profile():
        by[name] = by.get(name, 0.0) + ms
    c.set_profiling(False)
    return {k: round(v, 3) for k, v in sorted(by.items())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=100_000)
    ap.add_argument("--seqs", type=int, default=20_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import alignment_algos_b200 as a
    from alignment_algos_b200 import synth
    _, sub = a.blosum62()
    sub = np.asarray(sub, np.float32)
    A = sub.shape[0]
    out = {"config": vars(args), **gpu_info()}

    # ---- C3 shape
    seqs, pq, pt = synth.pair_workload(1003, args.pairs, 100, 500)
    res, off = a.Context.pack(seqs)
    cells = float(sum(len(seqs[q]) * len(seqs[t]) for q, t in zip(pq, pt)))
    what = a.W_FWD | a.W_REV | a.W_TB | a.W_MASK
    templates = set(pt.tolist())
    profiles = [np.ascontiguousarray(sub[:, s].T) if k in templates else None for k, s in enumerate(seqs)]
    ctx = {"sub": a.Context(0), "profile": a.Context(0)}
    ctx["sub"].set_scoring(sub, 12, 1, a.SEMI_LOCAL)
    t0 = time.perf_counter()
    ctx["profile"].set_profile_scoring(profiles, 12, 1, a.SEMI_LOCAL)
    out["c3_set_profile_scoring_s"] = round(time.perf_counter() - t0, 3)
    out["c3_profile_bytes_host_fp32"] = int(sum(p.nbytes for p in profiles if p is not None))
    times = {k: [] for k in ctx}
    results = {}
    for rep in range(args.reps + 1):
        for k, c in ctx.items():
            t0 = time.perf_counter()
            r = c.fill_batch(res, off, pq, pt, what, 0.01)
            dt = time.perf_counter() - t0
            if rep:
                times[k].append(dt)
            results[k] = r
    same = all(np.array_equal(results["sub"][f], results["profile"][f]) for f in ("fwd_score", "rev_score", "threshold",
                                                                                  "nearopt_count"))
    out["c3"] = {"pairs": args.pairs, "cells_per_direction": cells, "identical_outputs": bool(same)}
    for k in ctx:
        best = min(times[k])
        out["c3"][k] = {"wall_s": [round(x, 4) for x in times[k]], "best_s": round(best, 4),
                        "gcups_end_to_end": round(2 * cells / best / 1e9, 1),
                        "kernel_ms": kernel_ms(ctx[k], lambda: ctx[k].fill_batch(res, off, pq, pt, what, 0.01))}
    out["c3"]["profile_over_sub_wall"] = round(out["c3"]["profile"]["best_s"] / out["c3"]["sub"]["best_s"], 4)
    for c in ctx.values():
        c.close()
    del profiles, results

    # ---- 20 k all-vs-all cross
    rng = np.random.default_rng(1004)
    seqs = synth.random_seqs(rng, args.seqs, 100, 500)
    res, off = a.Context.pack(seqs)
    ids = np.arange(args.seqs, dtype=np.int32)
    profiles = [np.ascontiguousarray(sub[:, s].T) for s in seqs]
    ctx = {"sub": a.Context(0), "profile": a.Context(0)}
    ctx["sub"].set_scoring(sub, 12, 1, a.SEMI_LOCAL)
    ctx["profile"].set_profile_scoring(profiles, 12, 1, a.SEMI_LOCAL)
    dev = {k: torch.empty((args.seqs, args.seqs), dtype=torch.float32, device="cuda") for k in ctx}
    times = {k: [] for k in ctx}
    for k, c in ctx.items():
        c.upload_sequences(res, off)
    for rep in range(args.reps + 1):
        for k, c in ctx.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            c.cross_run(ids, ids, dev[k].data_ptr())
            c.synchronize()
            dt = time.perf_counter() - t0
            if rep:
                times[k].append(dt)
    xcells = ctx["sub"].last_cross_cell_updates()
    out["cross"] = {"seqs": args.seqs, "cells": xcells, "identical_outputs": bool(torch.equal(dev["sub"], dev["profile"]))}
    for k in ctx:
        best = min(times[k])
        out["cross"][k] = {"wall_s": [round(x, 4) for x in times[k]], "best_s": round(best, 4),
                           "gcups": round(xcells / best / 1e9, 1)}
    out["cross"]["profile_over_sub_wall"] = round(out["cross"]["profile"]["best_s"] / out["cross"]["sub"]["best_s"], 4)
    for c in ctx.values():
        c.close()
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
