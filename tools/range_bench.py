"""Range search on one B200: per-stage CUDA-event times next to the rescore arm's Top-K on the same inputs.

    python tools/range_bench.py [--out FILE] [--reps 5] [--audit-rows 1000000]

C2 shape (1M x 1024 database, 10k queries, fp32 in, deferred database rows as the pipelines use them), thresholds for
about 1, 20 and 200 rows per query: filter kernel time (events around the launch inside the library) and its share of
the bf16 tensor peak, refine kernel time and its gathered bytes over the HBM peak, candidates and results per query,
and, alternated with it in the same process, topk_filter and topk_search(rescore, K=10).  Then the cross-fold
near-duplicate audit of a 1M-case cohort (1024-d, 5 folds, t = 0.999) next to cv_search_and_vote at K = 5 on the same
rows.  Card name and power limit are read in the same run.  Peaks: MEASURED_PEAKS.json as bench.py reads it."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from bench import peaks, tensor_peak          # noqa: E402
from emr2a_b200 import native, synth          # noqa: E402
from emr2a_b200.engine import csr_from_pairs, get_engine   # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "nvidia-smi unavailable"


def timed_ring(eng, fn, n_entries):
    """Run fn with the library's kernel timing on; returns (fn result, last n_entries kernel times in ms, call ms)."""
    native.check(eng.lib.emr2a_debug_tc_timing(1))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    import ctypes as C
    buf = (C.c_float * 64)()
    n = C.c_int(0)
    native.check(eng.lib.emr2a_debug_tc_elapsed(buf, 64, C.byref(n)))
    native.check(eng.lib.emr2a_debug_tc_timing(0))
    return out, [buf[i] for i in range(n.value - n_entries, n.value)], e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--audit-rows", type=int, default=1_000_000)
    args = ap.parse_args()
    eng = get_engine()
    dev = eng.device
    pk = peaks()
    res = {"device": card(), "peaks": pk, "c2": [], "audit": None}
    N, Q, D = 1_000_000, 10_000, 1024
    db_raw = synth.device_block(0, N, D, 16, 41, dev)[0]
    q_raw = synth.device_block(N, Q, D, 16, 41, dev)[0]
    db = eng.prepare(db_raw, None, 1.0, 1.0, native.NF_ROWNORM, "rescore", defer_f32=eng.defer_default(D))
    qs = eng.prepare(q_raw, None, 1.0, 1.0, native.NF_ROWNORM, "rescore")
    # thresholds from fp32 scores of 64 sampled queries (plain torch here: only the measurement is sized by them)
    qn = q_raw[:64] / (q_raw[:64].norm(dim=1, keepdim=True) + 1e-8)
    s = torch.cat([qn @ (c / (c.norm(dim=1, keepdim=True) + 1e-8)).T for c in db_raw.split(1 << 17)], dim=1)
    top = torch.topk(s, 200, dim=1).values
    del s
    flops = 2.0 * D * Q * N
    for per_q in (1, 20, 200):
        t = float(top[:, per_q - 1].median())
        rows = {"rows_per_query_target": per_q, "min_score": t, "range_filter_ms": [], "range_refine_ms": [],
                "range_call_ms": [], "csr_ms": [], "topk_filter_kernel_ms": [], "topk_filter_call_ms": [],
                "topk_rescore_call_ms": [], "topk_rescore_filter_kernel_ms": []}
        for rep in range(args.reps + 1):                 # rep 0 warms every shape up and is not recorded
            pairs, (f_ms, r_ms), call_ms = timed_ring(
                eng, lambda: eng._range_pairs(qs, db, t, None, None, False, 0, 1 << 26), 2)
            c0 = time.perf_counter()
            csr = csr_from_pairs(pairs, Q)
            torch.cuda.synchronize()
            csr_ms = (time.perf_counter() - c0) * 1e3
            _, (tf_ms,), tf_call = timed_ring(eng, lambda: eng.topk_filter(qs, db, 10), 1)
            _, (tr_ms,), tr_call = timed_ring(eng, lambda: eng.topk_search(qs, db, 10, "rescore"), 1)
            eng.consume_status()
            if rep:
                for k, v in (("range_filter_ms", f_ms), ("range_refine_ms", r_ms), ("range_call_ms", call_ms),
                             ("csr_ms", csr_ms), ("topk_filter_kernel_ms", tf_ms), ("topk_filter_call_ms", tf_call),
                             ("topk_rescore_call_ms", tr_call), ("topk_rescore_filter_kernel_ms", tr_ms)):
                    rows[k].append(round(v, 4))
        n_res = int(csr["offsets"][-1])
        # candidate count of the last call: the filter's counter, read through a call with zero capacities
        counts = torch.zeros(2, dtype=torch.int64, device=dev)
        ws_bytes = int(eng.lib.emr2a_range_search_workspace_bytes(Q, N, D))
        ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=dev)
        from emr2a_b200.engine import _lazy_arg, _ld, _round_up
        lazy_arg, _keep = _lazy_arg(db) if db.f32 is None else (None, None)
        native.check(eng.lib.emr2a_range_search(
            qs.f32.data_ptr(), _ld(qs.f32), qs.hi.data_ptr(), _ld(qs.hi), native.ptr(db.f32),
            _ld(db.f32) if db.f32 is not None else 0, db.hi.data_ptr(), _ld(db.hi), Q, N, D, None, None, 0, 0, t,
            qs.stats.data_ptr(), db.stats.data_ptr(), None, 0, None, 0, counts.data_ptr(), _round_up(ws.data_ptr(), 256),
            ws_bytes, lazy_arg, eng._stream()))
        n_cand = int(counts[0])
        med = {k: statistics.median(v) for k, v in rows.items() if isinstance(v, list)}
        peak, peak_kind = tensor_peak(pk, med["range_filter_ms"] * 1e-3 * args.reps)
        gathered = n_cand * D * 4.0 + n_cand * 16.0              # one fp32 (raw) database row + the candidate per candidate
        rows.update({
            "candidates_per_query": n_cand / Q, "results_per_query": n_res / Q,
            "median_ms": med,
            "range_filter_tflops": flops / (med["range_filter_ms"] * 1e-3) / 1e12,
            "range_filter_frac_of_tensor_peak": flops / (med["range_filter_ms"] * 1e-3) / 1e12 / peak,
            "tensor_peak": peak_kind,
            "range_filter_over_topk_filter_kernel": med["range_filter_ms"] / med["topk_filter_kernel_ms"],
            "refine_gathered_bytes": gathered,
            "refine_frac_of_hbm_peak": gathered / (med["range_refine_ms"] * 1e-3) / (pk["hbm_gbs"] * 1e9),
        })
        res["c2"].append(rows)
        print(json.dumps({k: rows[k] for k in ("rows_per_query_target", "candidates_per_query", "results_per_query",
                                               "median_ms", "range_filter_over_topk_filter_kernel",
                                               "range_filter_frac_of_tensor_peak", "refine_frac_of_hbm_peak")}), flush=True)
    del db, qs, db_raw, q_raw, top
    torch.cuda.empty_cache()

    n = args.audit_rows
    x, labels = synth.device_block(0, n, D, 16, 53, dev)
    folds = torch.randint(0, 5, (n,), generator=torch.Generator().manual_seed(5), dtype=torch.uint8).to(dev)
    audit = {"rows": n, "dim": D, "folds": 5, "min_score": 0.999}
    for name, fn in (("cross_fold_duplicates_s", lambda: eng.cross_fold_duplicates([x], folds, 0.999)),
                     ("cv_search_and_vote_k5_s", lambda: eng.cv_search_and_vote([x], labels, folds, 16, 5))):
        times = []
        for rep in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = fn()
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        audit[name] = [round(v, 4) for v in times[1:]]
        if name.startswith("cross"):
            audit["pairs_found"] = int(out["i"].numel())
    audit["note"] = "first call of each excluded (module load); host clock around calls that end in a device synchronise"
    res["audit"] = audit
    print(json.dumps(audit), flush=True)
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    else:
        print(text)


if __name__ == "__main__":
    main()
