"""The self-join (emr2a_self_join, Engine.near_duplicates) without a GPU: the tile-skip and diagonal-mask predicates of
the tensor-core filter restated in numpy, the multi-GPU band planner, the host-side post-processing, and a gloo
world-2 run of the distributed plumbing with a numpy stand-in for the kernel call."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

from emr2a_b200.dist import self_join_ranges          # noqa: E402
from emr2a_b200.engine import Engine, Operand, self_join_result   # noqa: E402

TBN = 256


def _pack(score, idx):
    b = np.asarray(score, dtype=np.float32).view(np.uint32).astype(np.uint64)
    o = np.where(b & np.uint64(0x80000000), ~b & np.uint64(0xFFFFFFFF), b ^ np.uint64(0x80000000))
    return ((o << np.uint64(32)) | (np.uint64(0xFFFFFFFF) - np.asarray(idx, dtype=np.uint64))).view(np.int64)


def _tile_computed(q0, q1, n, fold, bm):
    """[Q, N] bool: the pair (local query row, local database row) of a call for the band [q0, q1) lies in a tile the
    filter computes (tc_common.cuh: tri_skipped, unit_fold / tile_skipped with fold-sorted rows)."""
    Q, N = q1 - q0, n - q0
    qf, df = fold[q0:q1], fold[q0:]
    out = np.zeros((Q, N), dtype=bool)
    for mt in range((Q + bm - 1) // bm):
        a, b = mt * bm, min(mt * bm + bm, Q) - 1
        ufold = qf[a] if qf[a] == qf[b] else -1
        for t in range((N + TBN - 1) // TBN):
            c, d = t * TBN, min(t * TBN + TBN, N) - 1
            tri = q0 + d <= q0 + mt * bm                          # db_row0 + last <= q_row0 + first query of the tile
            fsk = ufold >= 0 and df[c] == ufold and df[d] == ufold
            out[a:b + 1, c:d + 1] = not (tri or fsk)
    return out


def _diag_masked(q0, q1, n):
    """[Q, N] bool: scores set to -inf by the diagonal mask of scan_tile (per 32-column chunk: c <= lim)."""
    Q, N = q1 - q0, n - q0
    out = np.zeros((Q, N), dtype=bool)
    for q in range(Q):
        for c0 in range(0, N, 32):
            lim = q0 + q - q0 - c0                                # q_row0 + q - db_row0 - c0
            c = np.arange(min(32, N - c0))
            out[q, c0 + c] = (lim >= 0) & (c <= lim)
    return out


def test_tile_skip_and_diagonal_mask_against_brute_force():
    rng = np.random.default_rng(1)
    for trial in range(60):
        n = int(rng.integers(1, 1400))
        q0 = int(rng.integers(0, n + 1))
        q1 = int(rng.integers(q0, n + 1))
        if q1 == q0:
            continue
        fold = np.sort(rng.integers(0, int(rng.integers(1, 6)), n)).astype(np.uint8)
        i = np.arange(q0, q1)[:, None]
        j = np.arange(q0, n)[None, :]
        admissible = (j > i) & (fold[i] != fold[j])
        for bm in (128, 256):
            computed = _tile_computed(q0, q1, n, fold, bm)
            assert not (admissible & ~computed).any(), (trial, bm)      # no admissible pair in a skipped tile
        masked = _diag_masked(q0, q1, n)
        assert np.array_equal(masked, j <= i), trial                   # exactly j <= i, the diagonal included
        # every pair the filter can emit is admissible, and every admissible pair of the band is emitted
        emitted = _tile_computed(q0, q1, n, fold, 256) & ~masked & (fold[i] != fold[j])
        assert np.array_equal(emitted, admissible), trial


def test_triangle_skips_tiles_below_the_diagonal():
    n, fold = 4096, np.zeros(4096, dtype=np.uint8)
    fold[2048:] = 1
    comp = _tile_computed(0, n, n, fold, 256)
    tiles = comp[::256, ::256]
    assert not tiles[np.tril_indices(16, -1)].any()                   # strictly below: skipped
    assert tiles[np.diag_indices(16)].sum() == 0                      # diagonal tiles lie in one fold here
    assert tiles[:8, 8:].all()                                        # cross-fold tiles above the diagonal


def _band_cost(n, counts, q0, q1, tile=256):
    if q1 <= q0:
        return 0
    ends = np.cumsum(counts) if counts is not None else None
    fold = np.zeros(n, dtype=np.int64) if ends is None else np.searchsorted(ends, np.arange(n), side="right")
    cost = 0
    for a in range(q0 // tile, (q1 + tile - 1) // tile):
        fa0, fa1 = fold[a * tile], fold[min(a * tile + tile, n) - 1]
        for b in range(a, (n + tile - 1) // tile):
            fb0, fb1 = fold[b * tile], fold[min(b * tile + tile, n) - 1]
            if not (counts is not None and fa0 == fa1 == fb0 == fb1):
                cost += 1
    return cost


def test_self_join_ranges_cover_align_balance():
    rng = np.random.default_rng(2)
    cases = [(1000, None), (100_000, None), (100_000, [20_000] * 5), (77_777, [10_000, 30_000, 0, 37_777]),
             (300, None), (0, None)]
    for _ in range(4):
        n = int(rng.integers(3000, 60_000))
        cuts = np.sort(rng.integers(0, n, 4))
        cases.append((n, list(np.diff(np.concatenate([[0], cuts, [n]])))))
    for n, counts in cases:
        for world in (1, 2, 3, 8):
            bands = self_join_ranges(n, counts, world)
            assert len(bands) == world
            assert bands[0][0] == 0 and bands[-1][1] == n
            for (a, b), (c, d) in zip(bands, bands[1:]):
                assert b == c and a <= b
            assert all(lo % 256 == 0 or lo == n for lo, _ in bands)
            if n and n < 40_000:
                costs = [_band_cost(n, counts, a, b) for a, b in bands]
                total = _band_cost(n, counts, 0, n)
                assert sum(costs) == total
                per_tile = (n + 255) // 256                            # the most one query tile can cost
                assert max(costs) - min(costs) <= per_tile, (n, counts, world, costs)
    # more ranks than tiles: the surplus ranks get empty bands
    bands = self_join_ranges(300, None, 8)
    assert sum(1 for a, b in bands if b > a) == 2 and bands[-1] == (300, 300)


def test_balance_is_by_admissible_tiles_not_rows():
    bands = self_join_ranges(1 << 20, None, 8)
    sizes = [b - a for a, b in bands]
    assert sizes[0] < sizes[-1]                                       # early query rows have more partners
    assert bands == sorted(bands)


def test_self_join_result_maps_normalises_and_sorts():
    rng = np.random.default_rng(3)
    n = 500
    perm = rng.permutation(n)
    fold_sorted = np.sort(rng.integers(0, 4, n)).astype(np.uint8)
    # pairs a < b in the joined order with random scores, emitted in random order
    a = rng.integers(0, n - 1, 2000)
    b = a + 1 + rng.integers(0, n - 1 - a)
    keep = np.unique(a * n + b, return_index=True)[1]
    a, b = a[keep], b[keep]
    s = rng.uniform(0.5, 1.0, a.shape).astype(np.float32)
    order = rng.permutation(a.shape[0])
    pairs = torch.from_numpy(np.stack([a[order], _pack(s[order], b[order])], axis=1))
    res = self_join_result(pairs, torch.from_numpy(perm), torch.from_numpy(fold_sorted), n)
    ci, cj = perm[a], perm[b]
    lo, hi = np.minimum(ci, cj), np.maximum(ci, cj)
    o = np.lexsort((hi, lo))
    assert np.array_equal(res["i"].numpy(), lo[o]) and np.array_equal(res["j"].numpy(), hi[o])
    assert (res["i"] < res["j"]).all()
    assert np.array_equal(res["score"].numpy(), s[o])
    caller_fold = np.empty(n, dtype=np.int64)
    caller_fold[perm] = fold_sorted
    assert np.array_equal(res["fold_i"].numpy(), caller_fold[lo[o]])
    assert np.array_equal(res["fold_j"].numpy(), caller_fold[hi[o]])
    plain = self_join_result(pairs, None, None, n)
    assert set(plain) == {"i", "j", "score"}
    assert np.array_equal(plain["i"].numpy(), np.sort(a)) and (plain["i"] < plain["j"]).all()


# ---------------------------------------------------------------------------------------------------------------
# Engine.near_duplicates(distributed=True) under gloo, with a numpy stand-in for the emr2a_self_join call: checks the
# cohort guard, the band plan, the gather and the post-processing, against distributed=False in the same process.
class _StubEngine(Engine):
    def __init__(self):
        self.device = torch.device("cpu")
        self.launches = 0

    def _embedding(self, x):
        return torch.as_tensor(np.asarray(x), dtype=torch.float32), 0

    def to_device(self, x, dtype=None):
        t = torch.as_tensor(np.asarray(x))
        return (t.to(dtype) if dtype is not None else t).contiguous()

    def prepare(self, seg0, seg1=None, w0=1.0, w1=1.0, flags=0, precision="rescore", defer_f32=False):
        x = seg0 if seg1 is None else torch.cat([seg0, seg1], dim=1)
        x = x / x.norm(dim=1, keepdim=True)
        return Operand(n=int(x.shape[0]), dim=int(x.shape[1]), f32=x)

    def self_join_prepared(self, op, min_score, folds=None, q_begin=0, q_end=None, max_results=1 << 26):
        x = op.f32.numpy()
        q_end = op.n if q_end is None else q_end
        s = x[q_begin:q_end] @ x.T
        i, j = np.nonzero(s >= min_score)
        i = i + q_begin
        keep = j > i
        if folds is not None:
            f = folds.numpy()
            keep &= f[i] != f[j]
        i, j = i[keep], j[keep]
        if i.shape[0] > max_results:
            raise ValueError(f"range_search: {i.shape[0]} results exceed max_results = {max_results}")
        return torch.from_numpy(np.stack([i, _pack(s[i - q_begin, j], j)], axis=1).astype(np.int64))


def _sj_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rng = np.random.default_rng(5)                         # same cohort on every rank
    n = 1500
    x = rng.standard_normal((n, 24)).astype(np.float32)
    x[700:760] = x[:60] + 0.01 * rng.standard_normal((60, 24)).astype(np.float32)
    x[1400] = x[3]
    folds = rng.integers(0, 5, n).astype(np.uint8)         # unsorted: the cohort goes into fold order
    eng = _StubEngine()
    out = {}
    for name, f in (("plain", None), ("folds", folds)):
        got = eng.near_duplicates([x[:, :10], x[:, 10:]], 0.9, folds=f, distributed=True)
        want = eng.near_duplicates([x[:, :10], x[:, 10:]], 0.9, folds=f, distributed=False)
        out[name] = (set(got) == set(want) and all(torch.equal(got[k], want[k]) for k in want), int(want["i"].shape[0]))
    # a rank handed a different cohort is refused on every rank
    bad = x.copy()
    if rank == 1:
        bad[0, 0] += 1.0
    try:
        eng.near_duplicates([bad], 0.9, distributed=True)
        out["guard"] = False
    except ValueError:
        out["guard"] = True
    # an overflow on one rank's band raises on every rank (no rank is left waiting in a collective)
    try:
        eng.near_duplicates([x], -1.0, distributed=True, max_results=1000)
        out["overflow"] = False
    except ValueError:
        out["overflow"] = True
    q.put((rank, out))
    dist.destroy_process_group()


def test_distributed_near_duplicates_world2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + os.getpid() % 2000
    procs = [ctx.Process(target=_sj_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = sorted((q.get(timeout=180) for _ in procs), key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
    for _, r in out:
        assert r["plain"][0] and r["folds"][0], r
        assert r["plain"][1] >= 61 and r["folds"][1] > 0, r          # planted pairs were found
        assert r["guard"] and r["overflow"], r
