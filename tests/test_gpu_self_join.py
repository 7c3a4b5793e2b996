"""Self-join (include/emr2a.h: emr2a_self_join, Engine.near_duplicates): every pair i < j of one row set with exact
score >= t, each pair once.

Held to float64 brute force (pairs within 1e-5 of t excepted) and, bit for bit, to the both-ends range search of the
same operand filtered to a < b: same pairs, same score bits.  Both tensor-core kernels are covered: bands of more than
128 query rows run on CTA pairs, bands of 128 rows or fewer on single CTAs."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GAP = 1e-5
FLT_MAX = float(np.finfo(np.float32).max)


@pytest.fixture(scope="module")
def eng():
    from emr2a_b200.engine import get_engine
    return get_engine()


def _prep(eng, x):
    from emr2a_b200 import native
    return eng.prepare(x, None, 1.0, 1.0, native.NF_ROWNORM, "rescore")


def _abi(eng, op, t, q0, q1, folds=None, fold_sorted=False, cand_cap=1 << 16, res_cap=1 << 16, ws_off=0,
         sentinel=False, **over):
    """One emr2a_self_join call; returns (rc, counts, results, cand).  ``sentinel``: counts start at 7 instead of 0
    (an error must leave them so); ``over`` replaces arguments by name."""
    import torch
    from emr2a_b200 import native
    from emr2a_b200.engine import _round_up, _ld
    ws_bytes = int(eng.lib.emr2a_self_join_workspace_bytes(op.n, op.dim))
    ws = torch.empty(ws_bytes + 512, dtype=torch.uint8, device=eng.device)
    cand = torch.zeros((max(cand_cap, 1), 2), dtype=torch.int64, device=eng.device)
    out = torch.zeros((max(res_cap, 1), 2), dtype=torch.int64, device=eng.device)
    counts = torch.full((2,), 7 if sentinel else 0, dtype=torch.int64, device=eng.device)
    a = dict(x_f32=op.f32.data_ptr(), ld_f32=_ld(op.f32), x_hi=op.hi.data_ptr(), ld_bf16=_ld(op.hi), n=op.n, D=op.dim,
             q0=q0, q1=q1, fold=native.ptr(folds), fold_sorted=int(fold_sorted), min_score=float(t),
             stats=op.stats.data_ptr(), ws=_round_up(ws.data_ptr(), 256) + ws_off)
    a.update(over)
    rc = eng.lib.emr2a_self_join(a["x_f32"], a["ld_f32"], a["x_hi"], a["ld_bf16"], a["n"], a["D"], a["q0"], a["q1"],
                                 a["fold"], a["fold_sorted"], a["min_score"], a["stats"], cand.data_ptr(), cand_cap,
                                 out.data_ptr(), res_cap, counts.data_ptr(), a["ws"], ws_bytes, eng._stream())
    torch.cuda.synchronize()
    return rc, counts.cpu().tolist(), out, cand


def _set(pairs):
    """{(i, key)} of int64 [m, 2] results (the key holds j and the exact score bits)."""
    p = pairs.cpu().numpy()
    return set(zip(p[:, 0].tolist(), p[:, 1].tolist()))


def _both_ends(eng, op, t, folds=None, fold_sorted=False):
    """The general range search of the operand against itself, filtered to a < b: {(a, key)}."""
    from emr2a_b200.engine import decode_keys
    pairs = eng._range_pairs(op, op, t, folds, folds, fold_sorted, 0, 1 << 24)
    _, b = decode_keys(pairs[:, 1])
    return _set(pairs[pairs[:, 0] < b])


def _cohort(n, d, seed, n_near=60, n_copy=10):
    """Clustered rows with planted near-duplicates (cosine ~0.9995) and exact copies."""
    rng = np.random.default_rng(seed)
    centres = rng.standard_normal((16, d)).astype(np.float32)
    x = centres[rng.integers(0, 16, n)] + 1.2 * rng.standard_normal((n, d)).astype(np.float32)
    src = rng.choice(n, n_near + n_copy, replace=False)
    dst = rng.choice(np.setdiff1d(np.arange(n), src), n_near + n_copy, replace=False)
    for k, (a, b) in enumerate(zip(src, dst)):
        noise = 0 if k >= n_near else 0.02 * np.linalg.norm(x[a]) / np.sqrt(d)
        x[b] = x[a] + noise * rng.standard_normal(d).astype(np.float32)
    return x, src, dst


def _brute(eng, x, t, folds=None):
    import torch
    xd = torch.from_numpy(x).to(eng.device, torch.float64)
    xd = xd / (xd.norm(dim=1, keepdim=True) + 1e-8)
    f = None if folds is None else torch.from_numpy(np.asarray(folds)).to(eng.device)
    want, near = set(), set()
    for lo in range(0, xd.shape[0], 4096):
        s = xd[lo:lo + 4096] @ xd.T
        ok = torch.ones_like(s, dtype=torch.bool)
        if f is not None:
            ok = f[lo:lo + 4096, None] != f[None, :]
        for i, j in torch.nonzero((s >= t) & ok).tolist():
            if lo + i < j:
                want.add((lo + i, j))
        for i, j in torch.nonzero(((s - t).abs() <= GAP) & ok).tolist():
            near.add((min(lo + i, j), max(lo + i, j)))
    return want, near


def test_oracle_pairs_without_folds(eng):
    """20k two-modal cohort, planted near-duplicates and exact copies: the float64 pair set, each pair once, no i == j."""
    from emr2a_b200 import synth
    data = synth.two_modal(20_000, 256, 256, 8, seed=61)
    x0 = np.concatenate([data["image"], data["text"]], axis=1)
    rng = np.random.default_rng(62)
    src = rng.choice(20_000, 70, replace=False)
    dst = rng.choice(np.setdiff1d(np.arange(20_000), src), 70, replace=False)
    for k, (a, b) in enumerate(zip(src, dst)):
        noise = 0 if k >= 60 else 0.01 * np.linalg.norm(x0[a]) / np.sqrt(512)
        x0[b] = x0[a] + noise * rng.standard_normal(512).astype(np.float32)
    t = 0.999
    res = eng.near_duplicates([x0[:, :256], x0[:, 256:]], t)
    assert set(res) == {"i", "j", "score"}
    i, j = res["i"].cpu().numpy(), res["j"].cpu().numpy()
    got = set(zip(i.tolist(), j.tolist()))
    assert np.all(i < j) and len(got) == len(i)
    assert np.all(np.lexsort((j, i)) == np.arange(len(i)))
    want, near = _brute(eng, x0, t)
    assert got - near == want - near
    assert {(min(a, b), max(a, b)) for a, b in zip(src, dst)} <= got
    assert np.all(res["score"].cpu().numpy() >= np.float32(t))


@pytest.mark.parametrize("band", [1000, 128, 100])          # CTA pairs / single CTAs
@pytest.mark.parametrize("folds_kind", [None, "sorted", "unsorted"])
def test_bit_identical_to_both_ends_range_search(eng, band, folds_kind):
    import torch
    n = 4_000 if band > 128 else 1_500
    x, _, _ = _cohort(n, 256, 70 + band)
    op = _prep(eng, x)
    rng = np.random.default_rng(band)
    folds = None
    if folds_kind is not None:
        f = rng.integers(0, 5, n).astype(np.uint8)
        folds = torch.from_numpy(np.sort(f) if folds_kind == "sorted" else f).to(eng.device)
    sample = _unit(x[:400]) @ _unit(x).T
    t = float(np.quantile(sample[sample < 0.9999], 0.998))             # a few pairs per row
    ref = _both_ends(eng, op, t, folds, folds_kind == "sorted")
    got = set()
    for q0 in range(0, n, band):
        part = eng.self_join_prepared(op, t, folds, q0, min(q0 + band, n))
        assert not (_set(part) & got)
        got |= _set(part)
    assert got == ref and len(ref) > n
    assert all(i < (0xFFFFFFFF - (key & 0xFFFFFFFF)) for i, key in list(ref)[:2000])


def _unit(x):
    x = np.asarray(x, dtype=np.float64)
    return x / (np.linalg.norm(x, axis=1, keepdims=True) + 1e-8)


def test_ragged_partition_equals_one_call(eng):
    """Bands with boundaries off the tile grid, empty bands, q_end = n with n not a multiple of 256."""
    import torch
    n = 5_077
    x, _, _ = _cohort(n, 192, 81)
    op = _prep(eng, x)
    folds = torch.from_numpy(np.sort(np.random.default_rng(82).integers(0, 3, n)).astype(np.uint8)).to(eng.device)
    sample = _unit(x[:300]) @ _unit(x).T
    t = float(np.quantile(sample[sample < 0.9999], 0.999))
    for f in (None, folds):
        whole = _set(eng.self_join_prepared(op, t, f))
        cuts = [0, 0, 37, 100, 357, 1000, 1000, 1129, 2500, 4999, n, n]
        union, total = set(), 0
        for a, b in zip(cuts, cuts[1:]):
            part = eng.self_join_prepared(op, t, f, a, b)
            total += int(part.shape[0])
            union |= _set(part)
            assert all(a <= i < b for i, _ in _set(part))
        assert union == whole and total == len(whole) and len(whole) > n // 2


@pytest.mark.parametrize("fold_kind", [None, "sorted", "unsorted"])
def test_lowest_finite_min_score_counts_every_pair(eng, fold_kind):
    import torch
    n = 1000
    rng = np.random.default_rng(91)
    x = rng.standard_normal((n, 128)).astype(np.float32)
    x[500] = x[3]                                                      # identical rows: a 1.0 tie, still one pair
    op = _prep(eng, x)
    folds, want = None, n * (n - 1) // 2
    if fold_kind is not None:
        f = rng.integers(0, 4, n).astype(np.uint8)
        f = np.sort(f) if fold_kind == "sorted" else f
        folds = torch.from_numpy(f).to(eng.device)
        want = (n * n - int(np.sum(np.bincount(f) ** 2))) // 2
    for q0, q1 in ((0, n), (0, 100)):                                  # CTA pairs / single CTAs
        rc, counts, out, _ = _abi(eng, op, -FLT_MAX, q0, q1, folds, fold_kind == "sorted", cand_cap=600_000,
                                  res_cap=600_000)
        assert rc == 0
        if q1 == n:
            assert counts == [want, want]
        p = out[:counts[1]].cpu().numpy()
        j = 0xFFFFFFFF - (p[:, 1] & 0xFFFFFFFF)
        assert np.all(p[:, 0] < j) and np.all((p[:, 0] >= q0) & (p[:, 0] < q1))
        assert len(set(zip(p[:, 0].tolist(), j.tolist()))) == counts[1]
        if q1 < n:
            i0 = np.arange(q0, q1)
            if folds is None:
                assert counts[1] == int(np.sum(n - 1 - i0))
            else:
                fn = folds.cpu().numpy()
                assert counts[1] == sum(int(np.sum(fn[i + 1:] != fn[i])) for i in i0)


def test_overflow_counts_and_retry(eng):
    import torch
    from emr2a_b200.engine import decode_keys
    n = 6_000
    x, _, _ = _cohort(n, 256, 101)
    op = _prep(eng, x)
    sample = _unit(x[:300]) @ _unit(x).T
    t = float(np.quantile(sample[sample < 0.9999], 0.995))
    ref = _set(eng.self_join_prepared(op, t))
    n_res = len(ref)
    rc, (c0, c1), _, _ = _abi(eng, op, t, 0, n, cand_cap=5, res_cap=3)     # candidates overflow: nothing re-scored
    assert rc == 0 and c0 > n_res and c1 == 0
    rc, (c0b, c1b), _, _ = _abi(eng, op, t, 0, n, cand_cap=c0, res_cap=3)  # results overflow: both counts exact
    assert rc == 0 and (c0b, c1b) == (c0, n_res)
    rc, counts, out, _ = _abi(eng, op, t, 0, n, cand_cap=c0, res_cap=n_res)
    assert rc == 0 and counts == [c0, n_res] and _set(out[:n_res]) == ref
    with pytest.raises(ValueError, match=f"{n_res} results exceed|{c0} filter candidates exceed"):
        eng.self_join_prepared(op, t, max_results=n_res - 1)
    # the Engine's first buffers hold one result per row: a dense band takes the retry and still completes
    dense = eng.self_join_prepared(op, -FLT_MAX, None, 0, 300, max_results=1 << 22)
    assert int(dense.shape[0]) == sum(n - 1 - i for i in range(300))
    s, j = decode_keys(dense[:, 1])
    assert bool((dense[:, 0] < j).all())


def test_invalid_arguments_fail_before_any_work(eng):
    from emr2a_b200 import native
    n = 2_000
    x = np.random.default_rng(111).standard_normal((n, 128)).astype(np.float32)
    op = _prep(eng, x)
    bad = [({"q0": -1}, native.ERR_INVALID), ({"q0": 10, "q1": 5}, native.ERR_INVALID),
           ({"q1": n + 1}, native.ERR_INVALID), ({"min_score": float("nan")}, native.ERR_INVALID),
           ({"min_score": float("inf")}, native.ERR_INVALID), ({"stats": None}, native.ERR_INVALID),
           ({"x_f32": None}, native.ERR_INVALID), ({"x_hi": None}, native.ERR_INVALID),
           ({"ld_f32": 100}, native.ERR_INVALID), ({"ld_bf16": 120}, native.ERR_UNSUPPORTED),
           ({"n": -1}, native.ERR_INVALID), ({"D": 0}, native.ERR_INVALID)]
    for over, code in bad:
        kw = {"q0": 0, "q1": n}
        kw.update(over)
        q0, q1 = kw.pop("q0"), kw.pop("q1")
        rc, counts, out, cand = _abi(eng, op, -1.0, q0, q1, sentinel=True, **kw)
        assert rc == code, (over, rc, native.last_error())
        assert counts == [7, 7] and int(out.abs().sum()) == 0 and int(cand.abs().sum()) == 0, over
    rc, counts, out, cand = _abi(eng, op, -1.0, 0, n, ws_off=16, sentinel=True)          # misaligned workspace
    assert rc == native.ERR_INVALID and "aligned" in native.last_error()
    assert counts == [7, 7] and int(out.abs().sum()) == 0 and int(cand.abs().sum()) == 0


def test_cross_fold_duplicates_is_near_duplicates_with_folds(eng):
    import torch
    n = 8_000
    x, _, _ = _cohort(n, 256, 121, n_near=80, n_copy=20)
    folds = np.random.default_rng(122).integers(0, 5, n).astype(np.uint8)
    a = eng.cross_fold_duplicates([x[:, :100], x[:, 100:]], folds, 0.999)
    b = eng.near_duplicates([x[:, :100], x[:, 100:]], 0.999, folds=folds)
    assert set(a) == set(b) == {"i", "j", "score", "fold_i", "fold_j"}
    assert all(torch.equal(a[k], b[k]) for k in a)
    assert int(a["i"].numel()) > 0
    fi = a["fold_i"].cpu().numpy()
    assert np.array_equal(fi, folds[a["i"].cpu().numpy()]) and np.all(fi != a["fold_j"].cpu().numpy())


def test_million_case_audit_equals_both_ends(eng):
    """1M x 256 cohort, 5 unsorted folds, planted near-duplicates: near_duplicates equals the both-ends range search
    (fold order, a < b) bit for bit, and 32 sampled rows are checked against float64."""
    import torch
    from emr2a_b200 import synth
    from emr2a_b200.engine import _fold_order, cross_fold_pairs
    n, d, t = 1_000_000, 256, 0.999
    x, _ = synth.device_block(0, n, d, 16, 131, eng.device)
    g = torch.Generator(device="cpu").manual_seed(132)
    src = torch.randperm(n, generator=g)[:4000].to(eng.device)
    dst = torch.randperm(n, generator=g)[:4000].to(eng.device)
    keep = src != dst
    src, dst = src[keep], dst[keep]
    x[dst] = x[src] + 0.01 * x[src].norm(dim=1, keepdim=True) / d ** 0.5 * torch.randn(
        (int(src.numel()), d), device=eng.device, generator=torch.Generator(device=eng.device).manual_seed(133))
    folds = torch.randint(0, 5, (n,), generator=g, dtype=torch.uint8).to(eng.device)
    res = eng.near_duplicates([x], t, folds=folds)
    perm = _fold_order(folds)
    xs, fs = x.index_select(0, perm), folds.index_select(0, perm)
    op = _prep(eng, xs)
    old = cross_fold_pairs(eng._range_pairs(op, op, t, fs, fs, True, 0, 1 << 24), perm, fs)
    del op
    for k in ("i", "j", "score", "fold_i", "fold_j"):
        assert torch.equal(res[k], old[k]), k
    assert int(res["i"].numel()) > 1000
    xn = x.double() / (x.double().norm(dim=1, keepdim=True) + 1e-8)
    rows = torch.randperm(n, generator=g)[:32].tolist()
    rows[:16] = src[:16].tolist()                                      # rows that do have partners
    i_all, j_all = res["i"].cpu().numpy(), res["j"].cpu().numpy()
    fl = folds.cpu().numpy()
    for r in rows:
        s = (xn @ xn[r]).cpu().numpy()
        ok = (fl != fl[r]) & (np.arange(n) != r)
        want = set(np.flatnonzero((s >= t) & ok).tolist())
        near = set(np.flatnonzero((np.abs(s - t) <= GAP) & ok).tolist())
        got = set(j_all[i_all == r].tolist()) | set(i_all[j_all == r].tolist())
        assert got - near == want - near, r
