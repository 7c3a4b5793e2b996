"""Near-duplicate audit on the B200: the triangle self-join (Engine.near_duplicates) next to the both-ends range search.

    python tools/audit_bench.py [--out FILE] [--rows 1000000] [--reps 3]
    torchrun --nproc-per-node W tools/audit_bench.py --dist [--rows N] [--check-rows 200000] [--out FILE]

One GPU: a 1M x 1024 cohort with 5 random folds and t = 0.999 (range_bench's audit).  Alternated in one process:
  * both-ends: the cohort in fold order, one K1 pass, _range_pairs(op, op, folds, folds, fold_sorted) and the a < b
    filter (cross_fold_pairs) -- the audit as it ran before the self-join existed;
  * self-join: near_duplicates(..., folds).
Filter and refine kernel times come from the library's timing ring, whole-call times from a host clock around calls
that end in a device synchronise; TFLOP/s count 2 D flops per admissible pair each path computes (ordered cross-fold
pairs for both-ends, unordered ones for the self-join).  The pair sets and scores must be equal.  With
``--unit-clock`` one more call of each path runs with EMR2A_TC_UNIT_CLOCK=1 and the per-pair busy time of the CTA-pair
kernel is summarised.
Under torchrun (--dist): near_duplicates(distributed=True) per call and each rank's filter time, and bit-equality
with one GPU at --check-rows.  Card name and power limit are read in the same run."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from emr2a_b200 import native, synth          # noqa: E402
from emr2a_b200.engine import _fold_order, cross_fold_pairs, get_engine   # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines() if r.returncode == 0 else ["nvidia-smi unavailable"]


def timed_ring(eng, fn):
    """fn() with the library's kernel timing on: (result, [filter ms, refine ms] of its range call, call s)."""
    native.check(eng.lib.emr2a_debug_tc_timing(1))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    call = time.perf_counter() - t0
    buf = (C.c_float * 64)()
    n = C.c_int(0)
    native.check(eng.lib.emr2a_debug_tc_elapsed(buf, 64, C.byref(n)))
    native.check(eng.lib.emr2a_debug_tc_timing(0))
    return out, [buf[i] for i in range(n.value - 2, n.value)], call


def both_ends(eng, x, folds, t):
    """The audit through the general range search: each pair from both ends, a < b kept afterwards."""
    perm = _fold_order(folds)
    xs, fs = (x, folds) if perm is None else (x.index_select(0, perm), folds.index_select(0, perm))
    op = eng.prepare(xs, None, 1.0, 1.0, native.NF_ROWNORM, "rescore")
    pairs = eng._range_pairs(op, op, t, fs, fs, True, 0, 1 << 27, first_per_query=2)
    return cross_fold_pairs(pairs, perm, fs)


def unit_clock_summary(eng, fn):
    """Per-pair busy time of the last CTA-pair launch made inside fn with EMR2A_TC_UNIT_CLOCK=1."""
    os.environ["EMR2A_TC_UNIT_CLOCK"] = "1"
    try:
        fn()
        torch.cuda.synchronize()
    finally:
        os.environ.pop("EMR2A_TC_UNIT_CLOCK")
    plan = (C.c_int64 * 8)()
    cap = 1 << 16
    clk = (C.c_uint64 * (2 * cap))()
    native.check(eng.lib.emr2a_debug_unit_clocks(clk, cap, plan))
    m_tiles, n_tiles, splits, tps, mg, sync_tiles, grid, units = (int(v) for v in plan)
    n_pairs = grid // 2
    start = [clk[2 * u] for u in range(units)]
    end = [clk[2 * u + 1] for u in range(units)]
    t0, t1 = min(start), max(end)
    busy = [sum(end[u] - start[u] for u in range(p, units, n_pairs)) for p in range(n_pairs)]
    last = [max(end[u] for u in range(p, units, n_pairs)) - t0 for p in range(n_pairs)]
    return {"plan": {"m_tiles": m_tiles, "n_tiles": n_tiles, "splits": splits, "tiles_per_split": tps, "mg": mg,
                     "sync_tiles": sync_tiles, "grid": grid, "units": units},
            "span_ms": (t1 - t0) / 1e6, "pair_busy_ms_mean": statistics.mean(busy) / 1e6,
            "pair_busy_ms_min": min(busy) / 1e6, "pair_busy_ms_max": max(busy) / 1e6,
            "pair_last_end_ms_min": min(last) / 1e6, "pair_last_end_ms_median": statistics.median(last) / 1e6}


def single(args, eng):
    dev = eng.device
    n, D, t = args.rows, 1024, 0.999
    x, _ = synth.device_block(0, n, D, 16, 53, dev)
    folds = torch.randint(0, 5, (n,), generator=torch.Generator().manual_seed(5), dtype=torch.uint8).to(dev)
    cnt = torch.bincount(folds.long(), minlength=5).double()
    cross_ordered = float(n) * n - float((cnt * cnt).sum())
    flops = {"both_ends": 2.0 * D * cross_ordered, "self_join": 2.0 * D * cross_ordered / 2}
    paths = {"both_ends": lambda: both_ends(eng, x, folds, t),
             "self_join": lambda: eng.near_duplicates([x], t, folds=folds)}
    rows = {name: {"filter_ms": [], "refine_ms": [], "call_s": []} for name in paths}
    outs = {}
    for name, fn in paths.items():                       # warm-up: module load, first allocations
        outs[name] = fn()
    torch.cuda.synchronize()
    for rep in range(args.reps):
        for name, fn in paths.items():
            out, (f_ms, r_ms), call = timed_ring(eng, fn)
            rows[name]["filter_ms"].append(round(f_ms, 3))
            rows[name]["refine_ms"].append(round(r_ms, 3))
            rows[name]["call_s"].append(round(call, 4))
            outs[name] = out
    a, b = outs["both_ends"], outs["self_join"]
    equal = all(torch.equal(a[k], b[k]) for k in ("i", "j", "score", "fold_i", "fold_j"))
    assert equal, "self-join and both-ends pair lists differ"
    res = {"rows": n, "dim": D, "folds": 5, "min_score": t, "pairs_found": int(b["i"].numel()), "equal": equal,
           "admissible_pairs": {"both_ends": cross_ordered, "self_join": cross_ordered / 2}}
    for name in paths:
        med = {k: statistics.median(v) for k, v in rows[name].items()}
        rows[name]["median"] = med
        rows[name]["filter_tflops"] = flops[name] / (med["filter_ms"] * 1e-3) / 1e12
    res["paths"] = rows
    res["filter_ratio_self_join_over_both_ends"] = (rows["self_join"]["median"]["filter_ms"]
                                                    / rows["both_ends"]["median"]["filter_ms"])
    res["call_ratio_self_join_over_both_ends"] = (rows["self_join"]["median"]["call_s"]
                                                  / rows["both_ends"]["median"]["call_s"])
    if args.unit_clock:
        res["unit_clocks"] = {name: unit_clock_summary(eng, fn) for name, fn in paths.items()}
    return res


def distributed(args, eng):
    import torch.distributed as dist
    dev = eng.device
    world, rank = dist.get_world_size(), dist.get_rank()
    res = {"world": world}

    def cohort(n):
        x, _ = synth.device_block(0, n, 1024, 16, 53, dev)
        folds = torch.randint(0, 5, (n,), generator=torch.Generator().manual_seed(5), dtype=torch.uint8).to(dev)
        return x, folds

    x, folds = cohort(args.check_rows)
    for name, f in (("no_folds", None), ("unsorted_folds", folds)):
        a = eng.near_duplicates([x], 0.999, folds=f, distributed=True)
        b = eng.near_duplicates([x], 0.999, folds=f, distributed=False)
        same = set(a) == set(b) and all(torch.equal(a[k], b[k]) for k in a)
        res[f"check_{name}"] = {"rows": args.check_rows, "pairs": int(a["i"].numel()), "equal_to_one_gpu": same}
    del x, folds
    torch.cuda.empty_cache()
    x, folds = cohort(args.rows)
    eng.near_duplicates([x], 0.999, folds=folds, distributed=True)       # warm-up
    calls, filt = [], []
    for rep in range(args.reps):
        dist.barrier()
        _, (f_ms, _r), call = timed_ring(eng, lambda: eng.near_duplicates([x], 0.999, folds=folds, distributed=True))
        calls.append(round(call, 4))
        filt.append(round(f_ms, 3))
    per_rank = [None] * world
    dist.all_gather_object(per_rank, {"rank": rank, "filter_ms": filt, "call_s": calls})
    res.update({"rows": args.rows, "dim": 1024, "folds": 5, "min_score": 0.999, "per_rank": per_rank,
                "call_s_median_rank0": statistics.median(calls)})
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--dist", action="store_true")
    ap.add_argument("--check-rows", type=int, default=200_000)
    ap.add_argument("--unit-clock", action="store_true")
    args = ap.parse_args()
    rank = 0
    if args.dist:
        import torch.distributed as dist
        lr = int(os.environ["LOCAL_RANK"])
        torch.cuda.set_device(lr)
        dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
        rank = dist.get_rank()
    eng = get_engine()
    res = {"device": card()}
    res.update(distributed(args, eng) if args.dist else single(args, eng))
    if rank == 0:
        text = json.dumps(res, indent=1)
        print(text, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as fh:
                fh.write(text + "\n")
    if args.dist:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
