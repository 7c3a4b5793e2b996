"""Near-duplicate groups on the B200: the union-find kernels alone, duplicate_groups next to near_duplicates, and a
cohort whose pair list does not fit max_results.

    python tools/groups_bench.py [--out profiles/r05_duplicate_groups.json] [--rows 1000000] [--reps 3]

(a) emr2a_components_union + emr2a_components_finish (CUDA events, median of --reps, parent reset between reps) on a
    10M-vertex graph with 1e8 uniform random edges and on a 1M-vertex path given in descending and in shuffled order.
    The byte bound is the edge bytes read once (16 B per edge) over the 7.7 TB/s HBM data-sheet peak; the kernels do
    random 8-byte accesses to parent[], so they are bound by access latency, far from that bound.  Beside it: the same
    graph through scipy.sparse.csgraph.connected_components on the host (one run), plus the device-to-host copy of the
    edges it would need.  Labels are checked against scipy (smallest vertex of each component).
(b) duplicate_groups against near_duplicates on audit_bench's 1M x 1024 cohort at t = 0.999, alternated, host clock
    around calls that end in a device synchronise.
(c) the same cohort with one planted cluster of 12k identical rows (7.2e7 pairs): near_duplicates with its default
    max_results raises; duplicate_groups completes.  Bands, overflowed passes and time are reported.
Card name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tools"))
from audit_bench import card                      # noqa: E402
from emr2a_b200 import synth                      # noqa: E402
from emr2a_b200.engine import get_engine          # noqa: E402

HBM_PEAK = 7.7e12                                 # B/s, HGX B200 data sheet, one GPU


def min_labels_host(n, edges_host):
    import scipy.sparse as sp
    from scipy.sparse.csgraph import connected_components
    t0 = time.perf_counter()
    g = sp.coo_matrix((np.ones(edges_host.shape[0], dtype=np.int8), (edges_host[:, 0], edges_host[:, 1])),
                      shape=(n, n)).tocsr()
    _, lab = connected_components(g, directed=False)
    sec = time.perf_counter() - t0
    smallest = np.full(lab.max() + 1, n, dtype=np.int64)
    np.minimum.at(smallest, lab, np.arange(n))
    return smallest[lab], sec


def union_find(eng, name, n, edges, reps):
    """Kernel times of union and finish on one graph, the scipy comparison and the D2H copy of the edges."""
    dev = eng.device
    start = torch.arange(n, dtype=torch.int64, device=dev)
    parent = torch.empty_like(start)
    bad = torch.zeros(1, dtype=torch.int64, device=dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    u_ms, f_ms = [], []
    for rep in range(reps + 1):                                   # rep 0 warms up
        parent.copy_(start)
        torch.cuda.synchronize()
        ev[0].record()
        eng._components_union(parent, edges, bad)
        ev[1].record()
        eng._components_finish(parent)
        ev[2].record()
        torch.cuda.synchronize()
        if rep:
            u_ms.append(ev[0].elapsed_time(ev[1]))
            f_ms.append(ev[1].elapsed_time(ev[2]))
    assert int(bad.item()) == 0
    m = int(edges.shape[0])
    host = torch.empty((m, 2), dtype=torch.int64, pin_memory=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    host.copy_(edges)
    torch.cuda.synchronize()
    d2h = time.perf_counter() - t0
    want, scipy_s = min_labels_host(n, host.numpy())
    same = bool(np.array_equal(parent.cpu().numpy(), want))
    assert same, f"{name}: labels differ from scipy"
    um, fm = statistics.median(u_ms), statistics.median(f_ms)
    bound_ms = m * 16 / HBM_PEAK * 1e3
    return {"vertices": n, "edges": m, "union_ms": [round(x, 3) for x in u_ms], "finish_ms": [round(x, 3) for x in f_ms],
            "union_ms_median": round(um, 3), "finish_ms_median": round(fm, 3),
            "edges_per_s": m / ((um + fm) * 1e-3), "edge_read_bound_ms": round(bound_ms, 3),
            "union_share_of_byte_bound": bound_ms / um, "scipy_host_s": round(scipy_s, 3),
            "d2h_edges_s": round(d2h, 4), "labels_equal_scipy": same,
            "components": int(np.count_nonzero(want == np.arange(n)))}


def part_a(eng, reps):
    dev = eng.device
    g = torch.Generator(device=dev).manual_seed(7)
    out = {}
    n = 10_000_000
    edges = torch.randint(0, n, (100_000_000, 2), generator=g, device=dev, dtype=torch.int64)
    out["random_10M_1e8"] = union_find(eng, "random", n, edges, reps)
    del edges
    n = 1_000_000
    path = torch.stack([torch.arange(n - 1, device=dev), torch.arange(1, n, device=dev)], dim=1)
    out["path_1M_descending"] = union_find(eng, "path_desc", n, path.flip(0).contiguous(), reps)
    perm = torch.randperm(n - 1, generator=g, device=dev)
    out["path_1M_shuffled"] = union_find(eng, "path_shuffled", n, path[perm].contiguous(), reps)
    return out


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def part_b(eng, x, reps):
    t = 0.999
    paths = {"near_duplicates": lambda: eng.near_duplicates([x], t),
             "duplicate_groups": lambda: eng.duplicate_groups([x], t)}
    outs = {name: fn() for name, fn in paths.items()}               # warm-up
    secs = {name: [] for name in paths}
    for _ in range(reps):
        for name, fn in paths.items():
            outs[name], s = timed(fn)
            secs[name].append(round(s, 4))
    nd, dg = outs["near_duplicates"], outs["duplicate_groups"]
    assert dg["n_pairs"] == int(nd["i"].numel())
    med = {name: statistics.median(v) for name, v in secs.items()}
    return {"rows": int(x.shape[0]), "dim": int(x.shape[1]), "min_score": t, "pairs": dg["n_pairs"],
            "groups": dg["n_groups"], "bands": dg["n_bands"], "call_s": secs, "call_s_median": med,
            "overhead_groups_over_pairs": med["duplicate_groups"] / med["near_duplicates"] - 1.0}


def part_c(eng, x, cluster_rows):
    t = 0.999
    n = int(x.shape[0])
    rows = torch.randperm(n, generator=torch.Generator().manual_seed(11))[:cluster_rows].sort().values.to(x.device)
    x = x.clone()
    x[rows] = x[rows[0]].clone()
    res = {"rows": n, "dim": int(x.shape[1]), "min_score": t, "cluster_rows": cluster_rows,
           "cluster_pairs": cluster_rows * (cluster_rows - 1) // 2}
    try:
        eng.near_duplicates([x], t)
        res["near_duplicates"] = "completed"
    except ValueError as e:
        res["near_duplicates"] = f"ValueError: {e}"
    torch.cuda.empty_cache()
    eng.duplicate_groups([x], t)                                    # warm-up of the shapes the split passes use
    dg, s = timed(lambda: eng.duplicate_groups([x], t))
    group = dg["group"]
    assert bool((group[rows] == rows[0]).all()), "the planted cluster is not one group"
    res.update({"duplicate_groups_s": round(s, 3), "pairs": dg["n_pairs"], "groups": dg["n_groups"],
                "bands": dg["n_bands"], "overflowed_passes": dg["n_overflows"],
                "cluster_is_one_group": True})
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cluster-rows", type=int, default=12_000)
    args = ap.parse_args()
    eng = get_engine()
    res = {"device": card(), "hbm_peak_bytes_per_s": HBM_PEAK}
    res["a_union_find"] = part_a(eng, args.reps)
    torch.cuda.empty_cache()
    x, _ = synth.device_block(0, args.rows, 1024, 16, 53, eng.device)
    res["b_groups_vs_pairs"] = part_b(eng, x, args.reps)
    torch.cuda.empty_cache()
    res["c_planted_cluster"] = part_c(eng, x, args.cluster_rows)
    text = json.dumps(res, indent=1)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
