"""Run under torchrun: sharded search at world_size W must give bit-identical keys to a
single-GPU search of the whole database (global-index tie rule)."""
import os, sys
import torch, torch.distributed as dist
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from emr2a_b200 import native, synth
from emr2a_b200.dist import fold_balanced_ranges, ranges_to_rows, shard_range, sharded_cv_search_and_vote, sharded_search_and_vote
from emr2a_b200.engine import get_engine

rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr); dev = torch.device("cuda", lr)
dist.init_process_group("nccl", device_id=dev)
eng = get_engine(dev)
n, d, q, k, c = 300_000, 256, 3000, 10, 3
flags = native.NF_SEGNORM | native.NF_ROWNORM
labels = synth.device_labels(0, n, c, 11, dev)
qi, ql = synth.device_block(50_003_968, q, d, c, 11, dev, label_seed=11)
qt, _ = synth.device_block(50_003_968, q, d, c, 12, dev, label_seed=11)
ok = True
for prec in ("rescore", "rescore-selfcontained", "bf16x3", "fp32"):
    coop = prec == "rescore"                      # cooperative shards (staged K2, two collectives) vs self-contained ones
    name, prec = prec, prec.split("-")[0]
    lo, hi = shard_range(n, rank, world)
    di, _ = synth.device_block(lo, hi - lo, d, c, 11, dev, label_seed=11)
    dt, _ = synth.device_block(lo, hi - lo, d, c, 12, dev, label_seed=11)
    r = sharded_search_and_vote(eng, (di, dt), (qi, qt), labels, ql, c, k, lo, flags, flags, precision=prec, cooperative=coop)
    fi, _ = synth.device_block(0, n, d, c, 11, dev, label_seed=11)
    ft, _ = synth.device_block(0, n, d, c, 12, dev, label_seed=11)
    full = eng.search_and_vote((fi, ft), (qi, qt), labels, ql, c, k, db_flags=flags, q_flags=flags, precision=prec)
    same = torch.equal(r["keys"], full["keys"]) and torch.equal(r["pred_vote"], full["pred_vote"]) and torch.equal(r["confusion"], full["confusion"])
    print(f"rank {rank}/{world} {name}: sharded == single-GPU: {same} (unverified {r.get('unverified')})", flush=True)
    ok = ok and same
# near-duplicate neighbourhoods spread over all shards: the bound cannot verify the queries that fall into them, so the
# cooperative path has to REPAIR them (exact re-scan on every shard, seeded with the merged lists, second all-gather)
def plant(block, first_row, every=997, count=300):
    rows = torch.arange(first_row, first_row + block.shape[0], device=dev)
    hit = (rows % every == 0) & (rows // every < count)
    cols = torch.arange(block.shape[1], device=dev, dtype=torch.float32)
    base = torch.cos(cols * 0.7311) + 0.25 * torch.sin(cols * 2.113)
    wiggle = 1e-4 * torch.sin(rows[hit, None].float() * 0.37 + cols[None, :] * 1.3)
    block = block.clone()
    block[hit] = base[None, :] + wiggle
    return block

lo, hi = shard_range(n, rank, world)
di = plant(synth.device_block(lo, hi - lo, d, c, 11, dev, label_seed=11)[0], lo)
dt = plant(synth.device_block(lo, hi - lo, d, c, 12, dev, label_seed=11)[0], lo)
fi = plant(synth.device_block(0, n, d, c, 11, dev, label_seed=11)[0], 0)
ft = plant(synth.device_block(0, n, d, c, 12, dev, label_seed=11)[0], 0)
qi2, qt2 = qi.clone(), qt.clone()
qi2[:8] = plant(qi[:8], 0, every=1, count=8)
qt2[:8] = plant(qt[:8], 0, every=1, count=8)
for coop in (True, False):
    r = sharded_search_and_vote(eng, (di, dt), (qi2, qt2), labels, ql, c, k, lo, flags, flags, precision="rescore", cooperative=coop)
    full = eng.search_and_vote((fi, ft), (qi2, qt2), labels, ql, c, k, db_flags=flags, q_flags=flags, precision="rescore")
    same = torch.equal(r["keys"], full["keys"]) and torch.equal(r["pred_vote"], full["pred_vote"]) and torch.equal(r["confusion"], full["confusion"])
    print(f"rank {rank}/{world} rescore with near-duplicates ({'cooperative' if coop else 'self-contained'}): sharded == single-GPU: {same} "
          f"(unverified {r.get('unverified')}, single GPU {full.get('unverified')})", flush=True)
    ok = ok and same and (not coop or world == 1 or r.get("unverified", 0) > 0)
del di, dt, fi, ft
# all-queries CV over the sharded cohort == the single-GPU one-pass CV
n_cv, n_folds = 200_000, 5
lo, hi = shard_range(n_cv, rank, world)
xi, _ = synth.device_block(lo, hi - lo, d, c, 19, dev, label_seed=19)
xt, _ = synth.device_block(lo, hi - lo, d, c, 20, dev, label_seed=19)
lab = synth.device_labels(0, n_cv, c, 19, dev)
fold = (torch.arange(n_cv, device=dev, dtype=torch.int64) * n_folds // n_cv).to(torch.uint8)
fi, _ = synth.device_block(0, n_cv, d, c, 19, dev, label_seed=19)
ft, _ = synth.device_block(0, n_cv, d, c, 20, dev, label_seed=19)
for prec in ("rescore", "bf16x3"):
    r = sharded_cv_search_and_vote(eng, (xi, xt), lab, fold, c, 5, lo, flags, k_list=[1, 3, 5], precision=prec,
                                   n_folds=n_folds, q_block=65536, want_lists=True)
    full = eng.cv_search_and_vote((fi, ft), lab, fold, c, 5, flags=flags, k_list=[1, 3, 5], precision=prec, n_folds=n_folds,
                                  distributed=False)
    names = ("hit_counts", "vote_counts", "confusion", "group_sizes", "top_idx", "top_scores", "pred_vote", "pred_weighted")
    same = all(torch.equal(r[key], full[key]) for key in names)
    print(f"rank {rank}/{world} cv {prec}: sharded == single-GPU: {same} (unverified {r['unverified']})", flush=True)
    ok = ok and same
    # fold-balanced shards (a slice of every fold per rank; the C5 layout of bench.py), rows generated per range
    ranges = fold_balanced_ranges([int((fold == f).sum()) for f in range(n_folds)], rank, world)
    bi = torch.cat([synth.device_block(g0, cnt, d, c, 19, dev, label_seed=19)[0] for g0, cnt in ranges])
    bt = torch.cat([synth.device_block(g0, cnt, d, c, 20, dev, label_seed=19)[0] for g0, cnt in ranges])
    r = sharded_cv_search_and_vote(eng, (bi, bt), lab, fold, c, 5, 0, flags, k_list=[1, 3, 5], precision=prec,
                                   n_folds=n_folds, q_block=16384, want_lists=True, row_ids=ranges_to_rows(ranges, dev))
    same = all(torch.equal(r[key], full[key]) for key in names)
    print(f"rank {rank}/{world} cv {prec}: fold-balanced shards == single-GPU: {same}", flush=True)
    ok = ok and same
    # the engine call itself goes multi-GPU under torchrun (every rank passes the same arrays), here with UNSORTED folds
    mixed = ((torch.arange(n_cv, device=dev, dtype=torch.int64) * 7919) % n_folds).to(torch.uint8)
    auto = eng.cv_search_and_vote((fi, ft), lab, mixed, c, 5, flags=flags, k_list=[1, 3, 5], precision=prec, n_folds=n_folds,
                                  distributed=True)
    single = eng.cv_search_and_vote((fi, ft), lab, mixed, c, 5, flags=flags, k_list=[1, 3, 5], precision=prec, n_folds=n_folds,
                                    distributed=False)
    same = all(torch.equal(auto[key], single[key]) for key in names)
    print(f"rank {rank}/{world} cv {prec}: engine auto-distributed == single-GPU: {same}", flush=True)
    ok = ok and same
# the multi-GPU near-duplicate self-join: each rank joins its band of query rows, pair lists all-gathered
n_sj = 120_000
xs, _ = synth.device_block(0, n_sj, d, c, 23, dev)
xs[n_sj // 2:n_sj // 2 + 500] = xs[:500] + 1e-3 * xs[500:1000]          # planted near-duplicates across the cohort
sj_folds = ((torch.arange(n_sj, device=dev, dtype=torch.int64) * 7919) % 5).to(torch.uint8)
for name, f in (("no folds", None), ("unsorted folds", sj_folds)):
    a = eng.near_duplicates([xs], 0.999, folds=f, distributed=True)
    b = eng.near_duplicates([xs], 0.999, folds=f, distributed=False)
    same = set(a) == set(b) and all(torch.equal(a[key], b[key]) for key in a)
    print(f"rank {rank}/{world} near_duplicates {name}: distributed == single-GPU: {same} ({int(b['i'].numel())} pairs)",
          flush=True)
    ok = ok and same and int(b["i"].numel()) > 0
# near-duplicate groups: each rank folds its band into a forest of its own, the forests are merged on every rank;
# a chain through both halves of the cohort joins rows of different ranks' bands, a tiny budget splits the bands
xs[n_sj - 700:n_sj - 200] = xs[n_sj // 2:n_sj // 2 + 500] + 1e-3 * xs[1000:1500]
for budget in (1 << 26, 600):
    a = eng.duplicate_groups([xs], 0.999, pair_budget=budget, distributed=True)
    b = eng.duplicate_groups([xs], 0.999, distributed=False)
    same = all(torch.equal(a[key], b[key]) for key in ("group", "keep", "group_size")) and \
        (a["n_groups"], a["n_pairs"]) == (b["n_groups"], b["n_pairs"])
    print(f"rank {rank}/{world} duplicate_groups pair_budget={budget}: distributed == single-GPU: {same} "
          f"({b['n_groups']} groups, {b['n_pairs']} pairs, {a['n_bands']} bands)", flush=True)
    ok = ok and same and b["n_groups"] < n_sj
a = eng.leak_free_folds([xs], sj_folds, 0.999, distributed=True)
b = eng.leak_free_folds([xs], sj_folds, 0.999, distributed=False)
same = all(torch.equal(a[key], b[key]) for key in b)
clean = int(eng.cross_fold_duplicates([xs], a["folds"], 0.999)["i"].numel()) == 0
print(f"rank {rank}/{world} leak_free_folds: distributed == single-GPU: {same}, no cross-fold pair left: {clean} "
      f"({int(a['moved'].numel())} rows moved)", flush=True)
ok = ok and same and clean
dist.barrier(); dist.destroy_process_group()
sys.exit(0 if ok else 1)
