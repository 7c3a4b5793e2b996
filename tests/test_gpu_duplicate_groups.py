"""Near-duplicate groups on the GPU (include/emr2a.h: emr2a_components_union / emr2a_components_finish,
Engine.connected_components, duplicate_groups, leak_free_folds).

The union-find labels every vertex with the smallest vertex of its component, so the labels are compared bit for bit
with scipy's components mapped to their smallest vertex -- not only as partitions.  The groups are held to float64
brute force, and to themselves under every band plan."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GAP = 1e-5


@pytest.fixture(scope="module")
def eng():
    from emr2a_b200.engine import get_engine
    return get_engine()


def _min_labels(n, edges):
    import scipy.sparse as sp
    from scipy.sparse.csgraph import connected_components
    edges = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
    g = sp.coo_matrix((np.ones(edges.shape[0], dtype=np.int8), (edges[:, 0], edges[:, 1])), shape=(n, n))
    _, lab = connected_components(g, directed=False)
    smallest = np.full(lab.max() + 1 if n else 0, n, dtype=np.int64)
    np.minimum.at(smallest, lab, np.arange(n))
    return smallest[lab]


GRAPHS = ["empty", "single", "self_loops", "dup_reversed", "path_desc", "path_shuffled", "star", "clique",
          "random_2m_8m"]


def _graph(name):
    rng = np.random.default_rng(71)
    path = np.stack([np.arange(999_999), np.arange(1, 1_000_000)], axis=1)
    if name == "empty":
        return 5, np.zeros((0, 2), dtype=np.int64)
    if name == "single":
        return 1, np.array([[0, 0]])
    if name == "self_loops":
        return 50, np.array([[3, 3], [7, 7], [3, 9], [9, 9]])
    if name == "dup_reversed":
        return 40, np.array([[1, 30], [30, 1], [1, 30], [30, 12], [12, 30], [39, 2], [2, 39]])
    if name == "path_desc":
        return 1_000_000, path[::-1].copy()
    if name == "path_shuffled":
        return 1_000_000, path[rng.permutation(path.shape[0])]
    if name == "star":
        return 100_000, np.stack([np.full(99_999, 77_777), np.delete(np.arange(100_000), 77_777)], axis=1)
    if name == "clique":                                  # 3000 vertices, 4.5e6 edges, inside 4000 vertices
        return 4000, np.stack(np.triu_indices(3000, 1), axis=1) + 500
    return 2_000_000, rng.integers(0, 2_000_000, (8_000_000, 2))


@pytest.mark.parametrize("name", GRAPHS)
def test_labels_equal_scipy_smallest_vertex(eng, name):
    n, edges = _graph(name)
    got = eng.connected_components(edges, n).cpu().numpy()
    assert got.dtype == np.int64 and got.shape == (n,)
    assert np.array_equal(got, _min_labels(n, edges)), name


def test_labels_do_not_depend_on_order_or_calls(eng):
    """Shuffled edges, the same edges over 7 calls, and a start from a finished forest give identical labels."""
    import torch
    rng = np.random.default_rng(72)
    n = 500_000
    edges = rng.integers(0, n, (1_200_000, 2))
    want = eng.connected_components(edges, n)
    shuffled = eng.connected_components(edges[rng.permutation(edges.shape[0])][:, ::-1].copy(), n)
    assert torch.equal(want, shuffled)
    parent = torch.arange(n, dtype=torch.int64, device=eng.device)
    bad = torch.zeros(1, dtype=torch.int64, device=eng.device)
    for part in np.array_split(edges, 7):
        eng._components_union(parent, eng.to_device(part, torch.int64), bad)
    eng._components_finish(parent)
    assert torch.equal(parent, want) and int(bad.item()) == 0
    half = eng.connected_components(edges[:600_000], n)
    both = eng.connected_components(edges[600_000:], n, parent=half)
    assert torch.equal(both, want)
    assert torch.equal(want.cpu(), torch.from_numpy(_min_labels(n, edges)))


def test_out_of_range_edges_are_counted_and_skipped(eng):
    import torch
    n = 1000
    edges = np.array([[0, 5], [5, 999], [1000, 3], [3, -1], [-7, 2], [4, 1 << 40], [6, 7]])
    e = eng.to_device(edges, torch.int64)
    parent = torch.arange(n, dtype=torch.int64, device=eng.device)
    bad = torch.zeros(1, dtype=torch.int64, device=eng.device)
    assert eng.lib.emr2a_components_union(parent.data_ptr(), n, e.data_ptr(), edges.shape[0], bad.data_ptr(),
                                          eng._stream()) == 0
    assert eng.lib.emr2a_components_finish(parent.data_ptr(), n, eng._stream()) == 0
    assert int(bad.item()) == 4
    assert np.array_equal(parent.cpu().numpy(), _min_labels(n, edges[[0, 1, 6]]))
    with pytest.raises(ValueError, match="4 edges have an end outside"):
        eng.connected_components(edges, n)


def test_argument_errors_before_any_launch(eng):
    import torch
    from emr2a_b200 import native
    lib, st = eng.lib, eng._stream()
    parent = torch.arange(10, dtype=torch.int64, device=eng.device)
    edges = torch.tensor([[0, 9]], dtype=torch.int64, device=eng.device)
    bad = torch.zeros(1, dtype=torch.int64, device=eng.device)
    p, e, b = parent.data_ptr(), edges.data_ptr(), bad.data_ptr()
    for args in ((p, -1, e, 1, b), (p, 10, e, -1, b), (None, 10, e, 1, b), (p, 10, None, 1, b), (p, 10, e, 1, None),
                 (p, (1 << 32) - 1, e, 1, b)):
        assert lib.emr2a_components_union(*args, st) == native.ERR_INVALID, args
    for args in ((p, -1), (None, 10), (p, 1 << 33)):
        assert lib.emr2a_components_finish(*args, st) == native.ERR_INVALID, args
    assert "components_finish" in native.last_error()
    # empty inputs are no-ops: a NULL pointer is allowed where its size is 0
    assert lib.emr2a_components_union(None, 0, None, 0, None, st) == 0
    assert lib.emr2a_components_union(p, 10, None, 0, None, st) == 0
    assert lib.emr2a_components_finish(None, 0, st) == 0
    torch.cuda.synchronize()
    assert torch.equal(parent.cpu(), torch.arange(10)) and int(bad.item()) == 0
    with pytest.raises(ValueError, match="parent must be"):
        eng.connected_components(edges, 10, parent=parent.to(torch.int32))
    with pytest.raises(ValueError, match="shape"):
        eng.connected_components(torch.zeros((3, 3), dtype=torch.int64), 10)
    for wrong in (parent.flip(0).contiguous(), parent - 1):         # parent[v] > v, parent[v] < 0
        with pytest.raises(ValueError, match="forest"):
            eng.connected_components(edges, 10, parent=wrong)


def _chain_cohort(n, seed, t):
    """20k two-modal rows with planted chains a ~ b ~ c (s(a, c) < t), near copies, exact copies and zero rows."""
    from emr2a_b200 import synth
    data = synth.two_modal(n, 256, 256, 8, seed=seed)
    x = np.concatenate([data["image"], data["text"]], axis=1).astype(np.float64)
    rng = np.random.default_rng(seed + 1)
    rows = rng.choice(n, 3 * 40 + 2 * 30 + 12, replace=False)
    chains, copies, zeros = rows[:120].reshape(40, 3), rows[120:180].reshape(30, 2), rows[180:]
    theta = 0.035                                       # cos(theta) = 0.99939 >= t > cos(2 theta) = 0.99755
    for a, b, c in chains:
        u = x[a] / np.linalg.norm(x[a])
        w = rng.standard_normal(x.shape[1])
        w -= (w @ u) * u
        w /= np.linalg.norm(w)
        r = np.linalg.norm(x[a])
        x[b] = r * (np.cos(theta) * u + np.sin(theta) * w)
        x[c] = r * (np.cos(2 * theta) * u + np.sin(2 * theta) * w)
    for k, (a, b) in enumerate(copies):
        x[b] = x[a] if k % 2 else x[a] + 0.005 * np.linalg.norm(x[a]) / np.sqrt(512) * rng.standard_normal(512)
    x[zeros] = 0.0
    return x.astype(np.float32), chains, copies, zeros


def _brute_pairs(eng, x, t):
    """float64 pairs i < j with s >= t, and the pairs within GAP of t (either side)."""
    import torch
    xd = torch.from_numpy(x).to(eng.device, torch.float64)
    xd = xd / (xd.norm(dim=1, keepdim=True) + 1e-8)
    want, near = [], []
    for lo in range(0, xd.shape[0], 4096):
        s = xd[lo:lo + 4096] @ xd.T
        upper = torch.arange(lo, lo + s.shape[0], device=eng.device)[:, None] < torch.arange(xd.shape[0],
                                                                                           device=eng.device)[None]
        for mask, out in (((s >= t) & upper, want), (((s - t).abs() <= GAP) & upper, near)):
            ij = torch.nonzero(mask)
            ij[:, 0] += lo
            out.append(ij.cpu().numpy())
    return np.concatenate(want), np.concatenate(near)


def test_groups_equal_float64_brute_force(eng):
    import torch
    t, n = 0.999, 20_000
    x, chains, copies, zeros = _chain_cohort(n, 81, t)
    segs = [x[:, :256], x[:, 256:]]
    res = eng.duplicate_groups(segs, t)
    group = res["group"].cpu().numpy()
    want, near = _brute_pairs(eng, x, t)
    near_set = {tuple(p) for p in near.tolist()}
    sure = np.array([p for p in want.tolist() if tuple(p) not in near_set], dtype=np.int64).reshape(-1, 2)
    lo, hi = _min_labels(n, sure), _min_labels(n, np.concatenate([want, near]))
    assert np.array_equal(lo, hi), "a pair within 1e-5 of t changes the components: pick another seed"
    assert np.array_equal(group, lo)
    # the groups are the components of the pairs near_duplicates returns, bit for bit
    nd = eng.near_duplicates(segs, t)
    assert res["n_pairs"] == int(nd["i"].shape[0])
    pairs = np.stack([nd["i"].cpu().numpy(), nd["j"].cpu().numpy()], axis=1)
    assert np.array_equal(group, _min_labels(n, pairs))
    for a, b, c in chains:
        assert group[a] == group[b] == group[c] == min(a, b, c)
    assert {(min(a, c), max(a, c)) for a, _, c in chains}.isdisjoint(map(tuple, pairs.tolist()))   # a, c below t
    for a, b in copies:
        assert group[a] == group[b] == min(a, b)
    assert np.array_equal(group[zeros], zeros)
    assert torch.equal(res["keep"], res["group"] == torch.arange(n, device=eng.device))
    assert res["n_groups"] == int(res["keep"].sum()) == len(np.unique(lo))
    size = res["group_size"].cpu().numpy()
    assert np.array_equal(size, np.bincount(group, minlength=n)[group])
    assert (size[chains.ravel()] == 3).all() and (size[zeros] == 1).all()


def test_tiny_pair_budget_equals_one_shot(eng):
    import torch
    t, n = 0.999, 20_000
    x, _, _, _ = _chain_cohort(n, 82, t)
    segs = [x[:, :256], x[:, 256:]]
    one = eng.duplicate_groups(segs, t)
    assert one["n_bands"] == 1 and one["n_overflows"] == 0
    small = eng.duplicate_groups(segs, t, pair_budget=max(8, one["n_pairs"] // 6))
    assert small["n_bands"] >= 4 and small["n_overflows"] >= 1
    for k in ("group", "keep", "group_size"):
        assert torch.equal(small[k], one[k]), k
    assert (small["n_pairs"], small["n_groups"]) == (one["n_pairs"], one["n_groups"])


def test_leak_free_folds_leave_no_cross_fold_pair(eng):
    t, n = 0.999, 20_000
    x, chains, copies, _ = _chain_cohort(n, 83, t)
    segs = [x[:, :256], x[:, 256:]]
    folds = np.random.default_rng(84).integers(0, 5, n).astype(np.uint8)
    assert eng.cross_fold_duplicates(segs, folds, t)["i"].shape[0] > 0
    res = eng.leak_free_folds(segs, folds, t)
    new = res["folds"].cpu().numpy()
    assert new.dtype == np.uint8
    assert eng.cross_fold_duplicates(segs, new, t)["i"].shape[0] == 0
    group = res["group"].cpu().numpy()
    size = np.bincount(group, minlength=n)[group]
    assert np.array_equal(new[size == 1], folds[size == 1])                  # rows without partners keep their fold
    assert np.array_equal(new, folds[group])
    assert np.array_equal(res["moved"].cpu().numpy(), np.nonzero(new != folds)[0])
    assert res["fold_counts_after"].sum().item() == n == res["fold_counts_before"].sum().item()


def test_identical_cluster_above_the_budget(eng):
    """200k rows with one cluster of 3000 identical rows (4.5e6 pairs): a budget of 1e6 pairs still gives the groups."""
    n, d = 200_000, 128
    rng = np.random.default_rng(85)
    x = rng.standard_normal((n, d)).astype(np.float32)
    cluster = np.sort(rng.choice(n, 3000, replace=False))
    x[cluster] = x[cluster[0]]
    res = eng.duplicate_groups([x], 0.99, pair_budget=1_000_000)
    assert res["n_pairs"] == 3000 * 2999 // 2
    assert res["n_overflows"] >= 1 and res["n_bands"] >= 5
    want = np.arange(n)
    want[cluster] = cluster[0]
    assert np.array_equal(res["group"].cpu().numpy(), want)
    assert res["n_groups"] == n - 2999
    with pytest.raises(ValueError, match="exceed"):
        eng.near_duplicates([x], 0.99, max_results=1_000_000)
