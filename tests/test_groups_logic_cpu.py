"""Near-duplicate groups (Engine.connected_components, duplicate_groups, leak_free_folds) without a GPU: the sub-band
planner, the band loop that splits on overflow, the leak-free fold rule, the merge of per-rank forests, and a gloo
world-2 run of the distributed path -- with numpy stand-ins for the self-join and the union-find kernels."""
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from scipy.sparse.csgraph import connected_components as scipy_cc

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

from emr2a_b200.dist import self_join_ranges          # noqa: E402
from emr2a_b200.engine import Engine, Operand, PairOverflow, range_retry_caps   # noqa: E402


def _pack(score, idx):
    b = np.asarray(score, dtype=np.float32).view(np.uint32).astype(np.uint64)
    o = np.where(b & np.uint64(0x80000000), ~b & np.uint64(0xFFFFFFFF), b ^ np.uint64(0x80000000))
    return ((o << np.uint64(32)) | (np.uint64(0xFFFFFFFF) - np.asarray(idx, dtype=np.uint64))).view(np.int64)


def _min_labels(n, edges):
    """Components of scipy, each labelled with its smallest vertex."""
    edges = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
    g = sp.coo_matrix((np.ones(edges.shape[0]), (edges[:, 0], edges[:, 1])), shape=(n, n))
    _, lab = scipy_cc(g, directed=False)
    smallest = np.full(lab.max() + 1 if n else 0, n, dtype=np.int64)
    np.minimum.at(smallest, lab, np.arange(n))
    return smallest[lab]


class _StubEngine(Engine):
    """The host logic of Engine with numpy stand-ins for the kernels: the self-join scores the rows in float32 and
    raises PairOverflow past ``max_results`` as the real retry rule does; the union-find is a sequential one."""

    def __init__(self):
        self.device = torch.device("cpu")
        self.launches = 0
        self.joins = []                                    # (q_begin, q_end, pairs, completed)

    def _embedding(self, x):
        return torch.as_tensor(np.asarray(x), dtype=torch.float32), 0

    def to_device(self, x, dtype=None):
        t = torch.as_tensor(np.asarray(x)) if not isinstance(x, torch.Tensor) else x
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
        self.joins.append((q_begin, q_end, int(i.shape[0]), i.shape[0] <= max_results))
        if i.shape[0] > max_results:
            range_retry_caps(4 * i.shape[0], i.shape[0], 4 * max_results, max_results, max_results)
        return torch.from_numpy(np.stack([i, _pack(s[i - q_begin, j], j)], axis=1).astype(np.int64))

    @staticmethod
    def _find(p, v):
        while p[v] != v:
            p[v] = p[p[v]]
            v = p[v]
        return v

    def _components_union(self, parent, edges, bad):
        p, n = parent.numpy(), int(parent.shape[0])
        for a, b in edges.tolist():
            if not (0 <= a < n and 0 <= b < n):
                bad += 1
                continue
            ra, rb = self._find(p, a), self._find(p, b)
            if ra != rb:
                p[max(ra, rb)] = min(ra, rb)

    def _components_finish(self, parent):
        p = parent.numpy()
        for v in range(p.shape[0]):
            p[v] = self._find(p, v)


def _band_cost(n, q0, q1, tile=256):
    """Admissible 256 x 256 tiles of the query band [q0, q1) under the triangle skip (no folds)."""
    if q1 <= q0:
        return 0
    n_t = (n + tile - 1) // tile
    return sum(n_t - a for a in range(q0 // tile, (q1 + tile - 1) // tile))


def test_sub_band_planner_cover_align_balance():
    rng = np.random.default_rng(11)
    cases = [(100_000, 0, 100_000), (100_000, 25_600, 100_000), (100_000, 0, 51_200), (77_777, 51_200, 77_777),
             (3000, 2816, 3000), (1000, 256, 512)]
    for _ in range(6):
        n = int(rng.integers(2000, 50_000))
        q0 = int(rng.integers(0, n // 256)) * 256
        q1 = int(rng.integers(q0 + 1, n + 1))
        cases.append((n, q0, q1))
    for n, q0, q1 in cases:
        for parts in (1, 2, 3, 7, 40):
            bands = self_join_ranges(n, None, parts, q_begin=q0, q_end=q1)
            assert len(bands) == parts
            assert bands[0][0] == q0 and bands[-1][1] == q1
            for (a, b), (c, d) in zip(bands, bands[1:]):
                assert b == c and a <= b
            assert all(lo % 256 == 0 for lo, hi in bands if hi > lo)
            costs = [_band_cost(n, a, b) for a, b in bands]
            assert sum(costs) == _band_cost(n, q0, q1)
            # each cut is off the ideal by less than one query tile, which costs at most n / 256 tiles
            assert max(costs) - min(costs) <= 2 * ((n + 255) // 256), (n, q0, q1, parts, costs)
    # the whole range is the plan of the multi-GPU self-join
    assert self_join_ranges(50_000, None, 4, q_begin=0, q_end=50_000) == self_join_ranges(50_000, None, 4)
    with pytest.raises(ValueError):
        self_join_ranges(1000, None, 2, q_begin=100, q_end=1000)


def test_pair_overflow_keeps_the_value_error_and_its_text():
    with pytest.raises(ValueError, match=r"range_search: 9 results exceed max_results = 8") as e:
        range_retry_caps(9, 9, 100, 100, 8)
    assert isinstance(e.value, PairOverflow) and e.value.pairs == 9
    with pytest.raises(PairOverflow, match=r"filter candidates exceed 4 x max_results = 32") as e:
        range_retry_caps(41, 0, 100, 100, 8)
    assert e.value.pairs == 11


def _cluster_cohort(n, dim, clusters, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, dim)).astype(np.float32)
    for rows in clusters:
        x[rows] = x[rows[0]]
    return x


def test_band_loop_splits_from_the_counts_and_equals_one_shot():
    n = 3000
    x = _cluster_cohort(n, 16, [np.arange(1000, 3000, 8), np.arange(2205, 2405, 2)], 12)   # 31125 + 4950 pairs
    eng = _StubEngine()
    want = eng.duplicate_groups([x], 0.95)
    assert want["n_bands"] == 1 and want["n_overflows"] == 0 and want["n_pairs"] == 31125 + 4950
    budget = 10_000
    eng.joins = []
    got = eng.duplicate_groups([x], 0.95, pair_budget=budget)
    for k in ("group", "keep", "group_size"):
        assert torch.equal(got[k], want[k]), k
    assert got["n_pairs"] == want["n_pairs"] and got["n_groups"] == want["n_groups"] == n - 249 - 99
    # the first pass takes the whole range and overflows; each overflowing pass is cut into sub-bands planned from
    # its count, and every pass that completed stays within the budget
    assert eng.joins[0] == (0, n, want["n_pairs"], False)
    calls = [j[:2] for j in eng.joins]
    for q0, q1, c, ok in eng.joins:
        if not ok:
            parts = min(-(-2 * c // budget), -(-(q1 - q0) // 256))              # capped at the band's tiles
            plan = [b for b in self_join_ranges(n, None, parts, q_begin=q0, q_end=q1) if b[1] > b[0]]
            assert len(plan) >= 2 and set(plan) <= set(calls), (q0, q1, plan)
    done = sorted((j[0], j[1]) for j in eng.joins if j[3])
    assert done[0][0] == 0 and done[-1][1] == n and all(b == c for (_, b), (c, _) in zip(done, done[1:]))
    assert all(j[2] <= budget for j in eng.joins if j[3])
    assert got["n_bands"] == len(done) >= 4
    assert got["n_overflows"] == sum(not j[3] for j in eng.joins) >= 2                # a sub-band was cut again
    # a single 256-row band above the budget cannot be split: the error names the count
    with pytest.raises(ValueError, match=r"cannot be split further and has \d+ pairs"):
        eng.duplicate_groups([x], 0.95, pair_budget=1000)


def test_connected_components_wrapper_on_random_graphs():
    rng = np.random.default_rng(13)
    eng = _StubEngine()
    for trial in range(20):
        n = int(rng.integers(1, 400))
        m = int(rng.integers(0, 2 * n))
        edges = rng.integers(0, n, (m, 2))
        lab = eng.connected_components(edges, n).numpy()
        assert np.array_equal(lab, _min_labels(n, edges)), trial
    with pytest.raises(ValueError, match="2 edges have an end outside"):
        eng.connected_components(np.array([[0, 1], [3, 5], [-1, 0]]), 5)
    with pytest.raises(ValueError, match="shape"):
        eng.connected_components(np.zeros((4, 3), dtype=np.int64), 5)


def test_new_folds_leave_no_cross_fold_edge():
    """new = folds[group] on random graphs: no edge joins two folds, and singletons keep their fold."""
    rng = np.random.default_rng(14)
    for trial in range(30):
        n = int(rng.integers(2, 600))
        m = int(rng.integers(0, n))
        edges = rng.integers(0, n, (m, 2))
        folds = rng.integers(0, 5, n).astype(np.uint8)
        group = _min_labels(n, edges)
        new = folds[group]
        assert (new[edges[:, 0]] == new[edges[:, 1]]).all(), trial
        size = np.bincount(group, minlength=n)[group]
        assert np.array_equal(new[size == 1], folds[size == 1])
        assert np.array_equal(new[group == np.arange(n)], folds[group == np.arange(n)])   # a group's smallest row


def test_leak_free_folds_removes_every_cross_fold_pair():
    rng = np.random.default_rng(15)
    n = 1200
    x = rng.standard_normal((n, 12)).astype(np.float32)
    src = rng.integers(0, n, 150)
    dst = rng.integers(0, n, 150)
    x[dst] = x[src] + 0.02 * rng.standard_normal((150, 12)).astype(np.float32)
    folds = rng.integers(0, 5, n).astype(np.uint8)
    eng = _StubEngine()
    before = eng.cross_fold_duplicates([x[:, :5], x[:, 5:]], folds, 0.99)
    assert before["i"].shape[0] > 20
    res = eng.leak_free_folds([x[:, :5], x[:, 5:]], folds, 0.99)
    new = res["folds"]
    assert new.dtype == torch.uint8
    assert eng.cross_fold_duplicates([x[:, :5], x[:, 5:]], new, 0.99)["i"].shape[0] == 0
    g = eng.duplicate_groups([x[:, :5], x[:, 5:]], 0.99)
    assert torch.equal(res["group"], g["group"])
    alone = (g["group_size"] == 1).numpy()
    assert np.array_equal(new.numpy()[alone], folds[alone])
    assert np.array_equal(res["moved"].numpy(), np.nonzero(new.numpy() != folds)[0])
    assert res["fold_counts_before"].tolist() == np.bincount(folds, minlength=5).tolist()
    assert res["fold_counts_after"].tolist() == np.bincount(new.numpy(), minlength=5).tolist()
    with pytest.raises(ValueError, match="fold ids"):
        eng.leak_free_folds([x], folds[:-1], 0.99)
    # the rows are taken as every other self-join method takes them: missing modalities skipped, plain lists accepted
    same = eng.leak_free_folds([None, x[:, :5], x[:, 5:]], folds.tolist(), 0.99)
    assert all(torch.equal(same[k], res[k]) for k in res)
    with pytest.raises(ValueError, match="fold ids"):
        eng.leak_free_folds([None, x.tolist()], folds[:-1], 0.99)


def test_tiny_budget_plans_no_more_parts_than_tiles(monkeypatch):
    """A count far above the budget is cut into at most one sub-band per 256-row tile, not into 2 c / budget parts."""
    import emr2a_b200.dist as d
    n = 2000
    x = _cluster_cohort(n, 16, [np.arange(0, 2000, 9)], 17)               # 223 rows: 24753 pairs
    eng = _StubEngine()
    asked = []
    real = d.self_join_ranges

    def spy(n_rows, fold_counts, world, *a, **k):
        asked.append(world)
        return real(n_rows, fold_counts, world, *a, **k)

    monkeypatch.setattr(d, "self_join_ranges", spy)
    with pytest.raises(ValueError, match="cannot be split further"):
        eng.duplicate_groups([x], 0.95, pair_budget=1)
    assert asked[0] == -(-n // 256) and max(asked) <= -(-n // 256)


def test_merge_of_per_rank_forests_equals_global_components():
    rng = np.random.default_rng(16)
    eng = _StubEngine()
    for trial in range(10):
        n = int(rng.integers(50, 800))
        edges = rng.integers(0, n, (int(rng.integers(0, n)), 2))
        for world in (2, 3, 8):
            cut = np.sort(rng.integers(0, edges.shape[0] + 1, world - 1))
            links = []
            for part in np.split(edges, cut):
                lab = eng.connected_components(part, n).numpy()
                v = np.nonzero(lab != np.arange(n))[0]
                links.append(np.stack([v, lab[v]], axis=1))
            merged = eng.connected_components(np.concatenate(links), n).numpy()
            assert np.array_equal(merged, _min_labels(n, edges)), (trial, world)
    # a start from a finished forest gives the components of both edge sets
    n = 300
    e1, e2 = rng.integers(0, n, (100, 2)), rng.integers(0, n, (100, 2))
    start = eng.connected_components(e1, n)
    both = eng.connected_components(e2, n, parent=start)
    assert both is start
    with pytest.raises(ValueError, match="forest"):
        eng.connected_components(e1, n, parent=torch.arange(n, dtype=torch.int64).flip(0).contiguous())
    assert np.array_equal(both.numpy(), _min_labels(n, np.concatenate([e1, e2])))


# ---------------------------------------------------------------------------------------------------------------
# duplicate_groups / leak_free_folds(distributed=True) under gloo: the cohort guard, the per-rank bands, the merge of
# the per-rank forests and the overflow raised on every rank, against distributed=False in the same process.
def _chain_cohort(n, dim, seed):
    """Random rows plus planted chains a ~ b ~ c (cos 0.4 = 0.92 >= 0.9 > cos 0.8 = 0.70 between a and c) and copies."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, dim)).astype(np.float64)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    for a, b, c in ((5, 900, 1402), (1300, 40, 777), (260, 261, 1499)):
        u = x[a]
        w = rng.standard_normal(dim)
        w -= (w @ u) * u
        w /= np.linalg.norm(w)
        x[b] = np.cos(0.4) * u + np.sin(0.4) * w
        x[c] = np.cos(0.8) * u + np.sin(0.8) * w
    x[1100:1104] = x[7]
    return x.astype(np.float32)


def _dg_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    n = 1500
    x = _chain_cohort(n, 24, 21)
    folds = np.random.default_rng(22).integers(0, 5, n).astype(np.uint8)
    eng = _StubEngine()
    out = {}
    for name, budget in (("one_shot", 1 << 26), ("split", 7)):
        got = eng.duplicate_groups([x[:, :10], x[:, 10:]], 0.9, pair_budget=budget, distributed=True)
        want = eng.duplicate_groups([x[:, :10], x[:, 10:]], 0.9, distributed=False)
        out[name] = (all(torch.equal(got[k], want[k]) for k in ("group", "keep", "group_size"))
                     and got["n_groups"] == want["n_groups"] and got["n_pairs"] == want["n_pairs"],
                     got["n_bands"], want["n_pairs"], got["group"].tolist())
    got = eng.leak_free_folds([x], folds, 0.9, distributed=True)
    want = eng.leak_free_folds([x], folds, 0.9)
    out["folds"] = all(torch.equal(got[k], want[k]) for k in want) and \
        eng.cross_fold_duplicates([x], got["folds"], 0.9)["i"].shape[0] == 0
    bad = x.copy()
    if rank == 1:
        bad[0, 0] += 1.0
    try:
        eng.duplicate_groups([bad], 0.9, distributed=True)
        out["guard"] = False
    except ValueError as e:
        out["guard"] = "different cohorts" in str(e)
    # an unsplittable band on one rank raises on every rank (no rank is left waiting in a collective); rank 0's
    # early rows are all copies of one row, rank 1's band is clean
    y = x.copy()
    y[:256] = y[0]
    try:
        eng.duplicate_groups([y], 0.9, pair_budget=1000, distributed=True)
        out["overflow"] = ""
    except ValueError as e:
        out["overflow"] = str(e)
    q.put((rank, out))
    dist.destroy_process_group()


def test_distributed_duplicate_groups_world2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 33500 + os.getpid() % 2000
    procs = [ctx.Process(target=_dg_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = sorted((q.get(timeout=300) for _ in procs), key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
    (_, r0), (_, r1) = out
    for r in (r0, r1):
        assert r["one_shot"][0] and r["split"][0], r
        assert r["split"][1] > r["one_shot"][1] >= 2, r            # a tiny budget splits the bands
        assert r["folds"] and r["guard"], r
    assert r0["one_shot"][3] == r1["one_shot"][3]                   # every rank returns the same groups
    group = np.asarray(r0["one_shot"][3])
    assert group[1402] == group[900] == 5 and group[777] == group[1300] == 40 and group[1499] == 260
    assert (group[1100:1104] == 7).all()
    assert "cannot be split further" in r0["overflow"]
    assert "another rank's band" in r1["overflow"]
