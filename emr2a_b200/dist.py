"""Row-sharded database across GPUs: one process per GPU, ``torch.distributed`` (NCCL over NVLink/NVSwitch) for the
exchange steps of the path.  Global row indices travel inside the packed keys, ties break on the global index and
every arm returns exact fp32 scores, so results are bit-identical for any GPU count and any sharding (SURVEY.md §8e).

* ``sharded_search_and_vote``     queries against a row-sharded database.  Cooperative shards: an all-reduce (MAX) of
                                  the shards' K-th best filter score, exact re-scoring of what can reach the global
                                  Top-K, ONE all-gather of exact keys + bounds, verification of the merged lists.
* ``sharded_cv_search_and_vote``  every case a query (5-fold CV rule) over fold-balanced shards; query blocks of prepared
                                  rows are broadcast from their owner over NVLink, double-buffered.
* ``self_join_ranges``             query bands of the multi-GPU self-join (``Engine.near_duplicates``,
                                  ``Engine.duplicate_groups``): equal admissible tensor-core tiles per rank under the
                                  triangle and fold skips; also the sub-bands of a band whose pairs overflow.
* host-resident databases         ``spread_device`` (ranks spread over the host bridges), ``h2d_rates`` +
                                  ``weighted_ranges`` (shards sized by each rank's host link), ``gather_host_rows``
                                  (replicated query rows copied once per node, all-gathered over NVLink).
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist

from .engine import Operand


def shard_range(n_rows: int, rank: int, world: int, align: int = 256) -> Tuple[int, int]:
    """Contiguous, tile-aligned row range [lo, hi) of ``rank``; the last rank takes the tail."""
    per = (n_rows + world - 1) // world
    per = (per + align - 1) // align * align
    lo = min(rank * per, n_rows)
    hi = min(lo + per, n_rows)
    return lo, hi


def spread_device(local_rank: int, local_world: int, visible: Optional[int] = None) -> int:
    """Device index for a rank when FEWER ranks than visible GPUs run on the node: the ranks are spread evenly over the
    devices (4 ranks on an 8-GPU box -> 0, 2, 4, 6) instead of packed onto the first ones.  GPUs are enumerated in PCI
    order, so neighbours hang off the same host bridge / socket and share its host-memory bandwidth; measured on this
    pool's 8-GPU boxes (tools/h2d_probe.py, profiles/r02_h2d_topology.md): GPUs 0-3 together get 93 GB/s from host
    memory, GPUs 4-7 together 142 GB/s, any single GPU 55.6 GB/s -- so {0, 1, 2, 3} move a host-resident database at
    half the rate of {0, 2, 4, 6}.  NVLink/NVSwitch bandwidth between any two GPUs is the same, so nothing is lost.
    ``EMR2A_SPREAD_DEVICES=0`` keeps device = local rank."""
    if visible is None:
        visible = torch.cuda.device_count()
    if os.environ.get("EMR2A_SPREAD_DEVICES", "1") == "0" or local_world <= 0 or visible <= local_world or visible % local_world:
        return local_rank
    return local_rank * (visible // local_world)


_H2D_RATES: Optional[List[float]] = None


def h2d_rates(device, mbytes: int = 256, reps: int = 3) -> List[float]:
    """Host->device rate (GB/s) of EVERY rank while all ranks copy at once (pinned memory, CUDA events), all-gathered:
    what each rank's link to host memory delivers under the load of a host-resident multi-GPU search.  Cached."""
    global _H2D_RATES
    if _H2D_RATES is not None:
        return _H2D_RATES
    world = dist.get_world_size() if dist.is_initialized() else 1
    n = (mbytes << 20) // 4
    host = torch.empty(n, dtype=torch.float32).pin_memory()
    buf = torch.empty(n, dtype=torch.float32, device=device)
    buf.copy_(host, non_blocking=True)
    torch.cuda.synchronize(device)
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        buf.copy_(host, non_blocking=True)
    e1.record()
    torch.cuda.synchronize(device)
    mine = torch.tensor([reps * n * 4 / (e0.elapsed_time(e1) / 1e3) / 1e9], dtype=torch.float64, device=device)
    if world > 1:
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        _H2D_RATES = [float(t) for t in allr]
    else:
        _H2D_RATES = [float(mine)]
    return _H2D_RATES


def weighted_ranges(n_rows: int, weights: Sequence[float], align: int = 256) -> List[Tuple[int, int]]:
    """Contiguous, ``align``-row-aligned row ranges [lo, hi) whose sizes are proportional to ``weights`` (one per
    rank).  For HOST-resident databases the step is bound by the copy to the device, so a rank whose link to host
    memory is slower takes proportionally fewer rows (``h2d_rates``) and all ranks finish their copies together."""
    w = [max(float(x), 0.0) for x in weights]
    total = sum(w)
    if total <= 0:
        w, total = [1.0] * len(w), float(len(w))
    out, lo, acc = [], 0, 0.0
    for r, x in enumerate(w):
        acc += x
        hi = n_rows if r == len(w) - 1 else min(n_rows, int(round(n_rows * acc / total / align)) * align)
        hi = max(hi, lo)
        out.append((lo, hi))
        lo = hi
    return out


def gather_host_rows(host_mats: Sequence[torch.Tensor], device) -> Tuple[List[torch.Tensor], int]:
    """Every rank holds the same HOST matrices (the queries of a host-resident search).  Each rank copies only its
    1/world slice of the rows to ``device`` and the slices are all-gathered (NCCL over NVLink; gloo for CPU tensors in
    the tests).  Returns (device matrices with all rows, bytes this rank copied from the host)."""
    world = dist.get_world_size() if dist.is_initialized() else 1
    rank = dist.get_rank() if dist.is_initialized() else 0
    out, copied = [], 0
    for m in host_mats:
        n = int(m.shape[0])
        per = (n + world - 1) // world
        lo, hi = min(rank * per, n), min(rank * per + per, n)
        mine = torch.zeros((per,) + tuple(m.shape[1:]), dtype=m.dtype, device=device)
        if hi > lo:
            mine[:hi - lo].copy_(m[lo:hi], non_blocking=True)
            copied += (hi - lo) * int(m[0].numel()) * m.element_size()
        out.append(gather_keys(mine).reshape((world * per,) + tuple(m.shape[1:]))[:n])
    return out, copied


def gather_keys(local_keys: torch.Tensor, group=None) -> torch.Tensor:
    """All-gather [Q, K] packed keys -> [world, Q, K].  Works for CUDA tensors (NCCL) and for
    CPU tensors (gloo; used by the CPU tests of this plumbing)."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return local_keys.unsqueeze(0)
    local_keys = local_keys.contiguous()
    out = torch.empty((world,) + tuple(local_keys.shape), dtype=local_keys.dtype, device=local_keys.device)
    if local_keys.is_cuda:
        dist.all_gather_into_tensor(out.view(-1), local_keys.view(-1), group=group)
    else:
        parts = [out[r] for r in range(world)]
        dist.all_gather(parts, local_keys, group=group)
    return out


def sharded_search_and_vote(eng, db_segs_local: Sequence, q_segs: Sequence, db_labels_global, q_labels,
                            n_classes: int, k: int, row_offset: int, db_flags: int, q_flags: int,
                            q_weights=(1.0, 1.0), k_list=(1, 3, 5), precision: str = "auto",
                            q_fold=None, db_fold_local=None, q_group=None, n_groups: int = 1,
                            want_lists: bool = True, timers: Optional[dict] = None,
                            defer_status: bool = False, cooperative: bool = True) -> Dict[str, torch.Tensor]:
    """Each rank: K1 on its database shard and on the (replicated) queries, local K2 with
    ``idx_base = row_offset``; all-gather keys; K3 merge; K4 vote on the merged lists.

    With the ``rescore`` arithmetic the shards work COOPERATIVELY (``_cooperative_search_and_vote``): they exchange
    their K-th best filter score before re-scoring, so a shard only re-scores the candidates that can still reach the
    global Top-K, and the verification is made once on the merged lists -- the per-rank cost of the exact stage shrinks
    with the shard instead of staying at 64 candidates per query.  ``cooperative=False`` (or ``EMR2A_COOP_SHARDS=0``)
    keeps every shard's search self-contained; both give bit-identical results."""
    n_q = int(q_segs[0].shape[0])
    n_db = int(db_segs_local[0].shape[0])
    dim = sum(int(s.shape[1]) for s in db_segs_local if s is not None)
    world = dist.get_world_size() if dist.is_initialized() else 1
    prec = eng.pick_precision(n_q, max(n_db, 1) * world, dim, k, precision)
    db = eng.prepare(db_segs_local[0], db_segs_local[1] if len(db_segs_local) > 1 else None, 1.0, 1.0, db_flags, prec,
                     defer_f32=eng.defer_default(dim))
    qs = eng.prepare(q_segs[0], q_segs[1] if len(q_segs) > 1 else None, q_weights[0], q_weights[1], q_flags, prec)
    if prec == "rescore" and world > 1 and cooperative and os.environ.get("EMR2A_COOP_SHARDS", "1") != "0":
        return _cooperative_search_and_vote(eng, qs, db, db_labels_global, q_labels, n_classes, k, row_offset, k_list,
                                            q_fold, db_fold_local, q_group, n_groups, want_lists, timers, defer_status)
    if timers is not None:
        timers["k2_start"].record()
    keys = eng.topk_search(qs, db, k, prec, q_fold=q_fold, db_fold=db_fold_local, idx_base=row_offset)
    if timers is not None:
        timers["k2_end"].record()
    # optimistic execution: the rescore status (did any rank overflow its exact re-scan list?) travels
    # with the keys in the same all-gather and is only looked at after the vote, so the step has a
    # single host synchronisation at its very end
    status = eng.pop_status_tensor() if prec == "rescore" else None
    if world > 1:
        payload = keys.reshape(-1)
        if status is not None:
            payload = torch.cat([payload, status.to(torch.int64)])
        allp = gather_keys(payload.unsqueeze(0)).squeeze(1)              # [world, Q*K (+4)]
        allk = allp[:, :keys.numel()].reshape(world, *keys.shape)
        if status is not None:
            status = allp[:, keys.numel():].to(torch.int32).max(dim=0).values
        keys = eng.topk_merge(allk, k)
    res = eng.vote_metrics(keys, db_labels_global, q_labels, n_classes, k_list=k_list, q_group=q_group,
                           n_groups=n_groups, want_lists=want_lists)
    res["keys"] = keys
    res["precision"] = prec
    if status is not None and defer_status:
        res["status"] = status          # device int32[4]: the caller checks [1] == 0 (see Engine.check_deferred)
    elif status is not None:
        st = status.cpu()
        if int(st[1]):            # some rank could not verify within its re-scan capacity: redo with the 3-pass arm
            return sharded_search_and_vote(eng, db_segs_local, q_segs, db_labels_global, q_labels, n_classes, k,
                                           row_offset, db_flags, q_flags, q_weights, k_list, "bf16x3", q_fold,
                                           db_fold_local, q_group, n_groups, want_lists, timers)
        res["unverified"] = int(st[0])
    return res


def _cooperative_search_and_vote(eng, qs, db, db_labels_global, q_labels, n_classes, k, row_offset, k_list, q_fold,
                                 db_fold_local, q_group, n_groups, want_lists, timers, defer_status):
    """The staged K2 of include/emr2a.h ("cooperative row shards") around two collectives:
        filter (tensor cores)  ->  all-reduce MAX of the local K-th best filter score (4*Q bytes)
        ->  exact re-scoring of the candidates above the global cut  ->  all-gather of exact keys + bounds
        ->  K3 merge  ->  verification of the MERGED selection  ->  K4 vote.
    Queries the merged lists cannot verify (rare: the global K-th best clears a shard's bound far more easily than a
    shard's own K-th best does) are re-searched exactly on every shard after the vote and patched in."""
    n_q = qs.n
    if timers is not None:
        timers["k2_start"].record()
    cand, tau, kth = eng.topk_filter(qs, db, k, q_fold=q_fold, db_fold=db_fold_local, idx_base=row_offset)
    if timers is not None:
        timers["k2_end"].record()                  # the dominant kernel: tensor-core filter + merge of its partial lists
    dist.all_reduce(kth, op=dist.ReduceOp.MAX)
    payload = eng.rescore_candidates(cand, tau, kth, qs, db, k, idx_base=row_offset)
    allp = gather_keys(payload.unsqueeze(0)).squeeze(1)                  # [world, Q*K + ceil(Q/2)]
    keys = eng.merge_payload(allp, n_q, k)
    flags, status = eng.verify_merged(keys, allp, k)

    def vote(kk):
        return eng.vote_metrics(kk, db_labels_global, q_labels, n_classes, k_list=k_list, q_group=q_group,
                                n_groups=n_groups, want_lists=want_lists)

    res = vote(keys)
    res["precision"] = "rescore"
    res["keys"] = keys
    if defer_status:
        res["status"] = status          # [1] != 0: some query needs the repair below -- the caller must not use the step
        return res
    n_flagged = int(status.cpu()[0])    # the step's only host synchronisation; identical on every rank
    if n_flagged:
        idx = torch.nonzero(flags).squeeze(1).to(torch.int32)
        comp = eng.exact_rescan(qs, db, idx, k, idx_base=row_offset, q_fold=q_fold, db_fold=db_fold_local,
                                seed_keys=keys.index_select(0, idx.long()))
        keys.index_copy_(0, idx.long(), eng.topk_merge(gather_keys(comp), k))
        res = vote(keys)
        res["precision"] = "rescore"
        res["keys"] = keys
    res["unverified"] = n_flagged
    return res


def fold_balanced_ranges(fold_counts: Sequence[int], rank: int, world: int, align: int = 256) -> List[Tuple[int, int]]:
    """Rows of ``rank`` in a FOLD-BALANCED sharding of a fold-ordered cohort (SURVEY.md §8e: "each shard holds
    ~N/(5G) rows of every fold so fold-skipping stays balanced"): every fold's row range is cut into ``world``
    contiguous, ``align``-row-aligned pieces and rank r takes piece r of every fold.  Returns [(first global row,
    count)] per fold, ascending.  With such shards every rank has the same amount of admissible work for ANY query
    block (it skips its piece of the block's own fold), so the per-block exchange of query rows costs no waiting."""
    out, start = [], 0
    for n_f in fold_counts:
        n_f = int(n_f)
        per = (n_f + world - 1) // world
        per = (per + align - 1) // align * align
        lo = min(rank * per, n_f)
        hi = min(lo + per, n_f)
        out.append((start + lo, hi - lo))
        start += n_f
    return out


def self_join_ranges(n_rows: int, fold_counts: Optional[Sequence[int]], world: int, tile: int = 256,
                     q_begin: int = 0, q_end: Optional[int] = None) -> List[Tuple[int, int]]:
    """Query bands [q0, q1) of the ranks in a multi-GPU self-join (``Engine.near_duplicates``) of ``n_rows`` rows,
    fold-ordered with ``fold_counts`` rows per fold (None: no folds).  The bands cover [0, n_rows), are cut at
    ``tile``-row boundaries and hold equal numbers of ADMISSIBLE tiles, counted as the tensor-core filter counts them
    with ``tile``-row query and database tiles: database tile b is computed for query tile a iff b >= a (triangle) and
    not both tiles lie inside the same fold.  A band of early rows is short, one of late rows long.  Ranks past the
    number of tiles get empty bands.
    ``q_begin`` (a multiple of ``tile``) and ``q_end`` cut the sub-range [q_begin, q_end) into ``world`` such bands
    instead: the sub-bands of one query band whose pairs overflow (``Engine.duplicate_groups``)."""
    q_end = n_rows if q_end is None else int(q_end)
    if q_begin % tile or not 0 <= q_begin <= q_end <= n_rows:
        raise ValueError(f"self_join_ranges: need a {tile}-aligned 0 <= q_begin <= q_end <= n_rows, "
                         f"got {q_begin}, {q_end}, {n_rows}")
    n_t = (n_rows + tile - 1) // tile
    t0, t1 = q_begin // tile, (q_end + tile - 1) // tile
    if t1 == t0:
        return [(q_begin, q_end)] * world
    a = np.arange(n_t, dtype=np.int64)
    cost = (n_t - a).astype(np.float64)                       # database tiles b >= a
    if fold_counts is not None:
        ends = np.cumsum(np.asarray([int(c) for c in fold_counts], dtype=np.int64))
        first, last = a * tile, np.minimum(a * tile + tile, n_rows) - 1
        f_lo = np.searchsorted(ends, first, side="right")      # fold of a tile's first / last row
        f_hi = np.searchsorted(ends, last, side="right")
        single = f_lo == f_hi
        # single-fold tiles of one fold are consecutive: those at or after tile a are skipped for a single-fold tile a
        for f in np.unique(f_lo[single]):
            idx = np.nonzero(single & (f_lo == f))[0]
            cost[idx] -= len(idx) - np.arange(len(idx))
    cum = np.concatenate([[0.0], np.cumsum(cost[t0:t1])])
    n_sub = t1 - t0
    cuts = [0] + [int(np.searchsorted(cum, cum[-1] * r / world, side="left")) for r in range(1, world)] + [n_sub]
    cuts = np.maximum.accumulate(np.minimum(cuts, n_sub)) + t0
    return [(min(int(cuts[r]) * tile, q_end), min(int(cuts[r + 1]) * tile, q_end)) for r in range(world)]


def ranges_to_rows(ranges: Sequence[Tuple[int, int]], device) -> torch.Tensor:
    parts = [torch.arange(g0, g0 + cnt, dtype=torch.int32, device=device) for g0, cnt in ranges if cnt > 0]
    return torch.cat(parts) if parts else torch.empty((0,), dtype=torch.int32, device=device)


def _gather_varlen(t: torch.Tensor, world: int) -> List[torch.Tensor]:
    """All-gather 1-D / 2-D tensors whose first dimension differs per rank."""
    if world == 1:
        return [t]
    n = torch.tensor([t.shape[0]], dtype=torch.int64, device=t.device)
    sizes = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(sizes, n)
    sizes = [int(x.item()) for x in sizes]
    cap = max(max(sizes), 1)
    pad = torch.zeros((cap,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    pad[:t.shape[0]] = t
    out = torch.empty((world, cap) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    if t.is_cuda:
        dist.all_gather_into_tensor(out.view(-1), pad.view(-1))
    else:
        dist.all_gather([out[r] for r in range(world)], pad)
    return [out[r, :sizes[r]] for r in range(world)]


def sharded_cv_search_and_vote(eng, segs_local: Sequence, labels_global, folds_global, n_classes: int, k: int,
                               row_offset: int, flags: int, q_weights=(1.0, 1.0), k_list=(1, 3, 5),
                               precision: str = "auto", n_folds: Optional[int] = None, q_block: int = 262144,
                               fold_sorted: bool = True, want_lists: bool = False,
                               full_segs: Optional[Sequence] = None, row_ids=None) -> Dict[str, torch.Tensor]:
    """The whole CV loop over a row-sharded cohort: EVERY case is a query against the cases of the OTHER folds
    (utils/cv_evaluator.py:349-376 builds exactly these train/test pairs, one fold at a time).  The rows are sharded
    over the ranks: ``segs_local`` = this rank's rows of every modality, ``row_ids`` (int32, ascending) their global
    indices -- or the contiguous range ``[row_offset, row_offset + n_local)`` when ``row_ids`` is None.  Shards that
    hold an equal slice of every fold (``fold_balanced_ranges``) keep all ranks equally busy on every query block.

    Data movement (queries ARE database rows, so nothing is prepared twice and nothing is replicated):
      1. every rank runs K1 ONCE on its own shard (fp32 rows and/or bf16 planes, as the precision arm needs);
      2. query blocks are walked owner by owner; the owner's PREPARED rows of the block are broadcast to the other
         ranks over NVLink (NCCL broadcast, double-buffered: block b+1 travels while block b is searched), so a rank
         holds its shard plus two query blocks -- never the cohort;
      3. each rank searches the block against its shard (fold rule: own-fold tiles skipped / masked), global row ids
         go into the keys (``emr2a_keys_map_rows``);
      4. the local Top-K keys are all-gathered, merged by K3, and K4 votes with per-fold counters.
    ``fold_sorted`` promises ``folds_global`` is non-decreasing (rows in fold order) so whole tiles of a single fold
    are skipped; pass False for arbitrary fold vectors (per-element mask only).  ``full_segs`` is accepted for
    backward compatibility and ignored.

    Returns per-fold counters (``hit_counts [F, nk]``, ``vote_counts [F, 3]``, ``confusion [F, 2, C, C]``,
    ``group_sizes [F]``), ``unverified`` and, with ``want_lists``, the per-query outputs of all N cases in global row
    order (identical on every rank).  Results are bit-identical for every GPU count and every sharding."""
    world = dist.get_world_size() if dist.is_initialized() else 1
    rank = dist.get_rank() if dist.is_initialized() else 0
    dev = eng.device
    mats = [eng._embedding(x)[0] for x in segs_local if x is not None]
    n_local = int(mats[0].shape[0])
    labels = eng.to_device(labels_global, torch.int32)
    folds = eng.to_device(folds_global, torch.uint8)
    n = int(labels.shape[0])
    if n_folds is None:
        n_folds = int(folds.max().item()) + 1 if n else 1
    dim = sum(int(m.shape[1]) for m in mats)
    prec = eng.pick_precision(n, n, dim, k, precision)
    contiguous = row_ids is None
    if contiguous:
        my_rows = torch.arange(row_offset, row_offset + n_local, dtype=torch.int32, device=dev)
    else:
        my_rows = eng.to_device(row_ids, torch.int32)
        if int(my_rows.shape[0]) != n_local:
            raise ValueError(f"sharded_cv_search_and_vote: {int(my_rows.shape[0])} row ids for {n_local} local rows")
    rows_of = _gather_varlen(my_rows, world)                   # every rank's global row ids
    # (1) K1 once per rank
    seg1 = mats[1] if len(mats) > 1 else None
    db = eng.prepare(mats[0], seg1, 1.0, 1.0, flags, prec)
    same_q = float(q_weights[0]) == 1.0 and float(q_weights[1]) == 1.0
    qsrc = db if same_q else eng.prepare(mats[0], seg1, q_weights[0], q_weights[1], flags, prec)
    planes = [nm for nm in ("f32", "hi", "lo") if getattr(db, nm) is not None]
    q_stats = None
    if qsrc.stats is not None:                                 # the owner's maxima are valid clamps for its rows
        q_stats = torch.stack(_gather_varlen(qsrc.stats.reshape(1, 2), world)).reshape(world, 2) if world > 1 \
            else qsrc.stats.reshape(1, 2)
    db_fold = folds[my_rows.long()]
    db_ids = None if contiguous else my_rows
    blocks = [(r, b0, min(b0 + q_block, int(rows_of[r].shape[0])))
              for r in range(world) for b0 in range(0, int(rows_of[r].shape[0]), q_block)]
    bufs = [None, None]
    if world > 1:
        cap = min(q_block, max(int(x.shape[0]) for x in rows_of))
        bufs = [{nm: torch.empty((cap, int(getattr(db, nm).shape[1])), dtype=getattr(db, nm).dtype, device=dev)
                 for nm in planes} for _ in range(2)]

    def post(i):
        """Start the broadcast of block i's prepared rows from its owner (asynchronous, NCCL's own stream)."""
        r, b0, b1 = blocks[i]
        if world == 1:
            return []
        works = []
        for nm in planes:
            t = getattr(qsrc, nm)[b0:b1] if r == rank else bufs[i % 2][nm][:b1 - b0]
            if t.dtype == torch.int16:                 # bf16 planes are stored as int16; NCCL has no 16-bit integer type
                t = t.view(torch.uint8)
            works.append(dist.broadcast(t, src=r, async_op=True))
        return works

    # (2)+(3) local searches, block b+1 in flight while block b is searched
    local = []
    pending = post(0) if blocks else []
    for i, (r, b0, b1) in enumerate(blocks):
        nxt = post(i + 1) if i + 1 < len(blocks) else []
        for w in pending:
            w.wait()
        pending = nxt
        src = qsrc if r == rank else None
        qs = Operand(n=b1 - b0, dim=dim,
                     f32=(src.f32[b0:b1] if src is not None else bufs[i % 2]["f32"][:b1 - b0]) if "f32" in planes else None,
                     hi=(src.hi[b0:b1] if src is not None else bufs[i % 2]["hi"][:b1 - b0]) if "hi" in planes else None,
                     lo=(src.lo[b0:b1] if src is not None else bufs[i % 2]["lo"][:b1 - b0]) if "lo" in planes else None,
                     stats=None if q_stats is None else q_stats[r])
        q_rows = rows_of[r][b0:b1].long()
        local.append(eng.topk_search(qs, db, k, prec, q_fold=folds[q_rows], db_fold=db_fold, fold_sorted=fold_sorted,
                                     idx_base=row_offset if contiguous else 0, row_ids=db_ids))
    # (4) exchange + merge + vote
    outs = []
    for i, (r, b0, b1) in enumerate(blocks):
        keys = local[i]
        if world > 1:
            keys = eng.topk_merge(gather_keys(keys), k)
        q_rows = rows_of[r][b0:b1].long()
        outs.append(eng.vote_metrics(keys, labels, labels[q_rows], n_classes, k_list=k_list, q_group=folds[q_rows],
                                     n_groups=n_folds, per_query=want_lists, want_lists=want_lists))
        local[i] = None
    unverified = 0
    if prec == "rescore" and blocks:
        st = eng.pop_status_tensor()
        if world > 1:
            st = st.to(torch.int64)
            dist.all_reduce(st, op=dist.ReduceOp.MAX)          # every rank must take the same branch below
        st = st.cpu()
        if int(st[1]):
            return sharded_cv_search_and_vote(eng, segs_local, labels_global, folds_global, n_classes, k, row_offset,
                                              flags, q_weights, k_list, "bf16x3", n_folds, q_block, fold_sorted, want_lists,
                                              None, row_ids)
        unverified = int(st[0])
    res: Dict[str, torch.Tensor] = {}
    for name in ("hit_counts", "vote_counts", "confusion", "group_sizes"):
        res[name] = torch.stack([o[name] for o in outs]).sum(dim=0) if outs else None
    if want_lists and outs:
        order = torch.cat([rows_of[r][b0:b1] for r, b0, b1 in blocks]).long()      # global row of every block position
        for name in ("top_idx", "top_scores", "top_labels", "pred_top1", "pred_vote", "pred_weighted"):
            cat = torch.cat([o[name] for o in outs])
            out = torch.empty_like(cat)
            out[order] = cat
            res[name] = out
    res["precision"] = prec
    res["unverified"] = unverified          # this rank's count (max over ranks when sharded)
    return res
