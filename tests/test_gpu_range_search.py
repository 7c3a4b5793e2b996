"""Range search (include/emr2a.h: emr2a_range_search): every admissible pair with exact score >= t.

The tensor-core filter emits every pair with s~ >= t - E and the exact fp32 re-scoring keeps s >= t, so the answer is
held to float64 brute force: every pair farther than 1e-5 from t is classified the same way, scores within 1e-5.
Scores are bit-identical to the rescore arm's Top-K for the same pair."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GAP = 1e-5


@pytest.fixture(scope="module")
def eng():
    from emr2a_b200.engine import get_engine
    return get_engine()


def _unit64(x):
    x = np.asarray(x, dtype=np.float64)
    return x / (np.linalg.norm(x, axis=1, keepdims=True) + 1e-8)


def _rows(csr, q):
    lo, hi = int(csr["offsets"][q]), int(csr["offsets"][q + 1])
    return csr["idx"][lo:hi].cpu().numpy(), csr["scores"][lo:hi].cpu().numpy()


def _check_against(csr, s64, t, idx_base=0, admissible=None):
    """Classification of every pair farther than GAP from t, scores within GAP, CSR order (score desc, index asc)."""
    Q = s64.shape[0]
    assert int(csr["offsets"][-1]) == int(csr["idx"].numel()) == int(csr["scores"].numel())
    for q in range(Q):
        idx, sc = _rows(csr, q)
        local = idx - idx_base
        want = s64[q] >= t
        if admissible is not None:
            want &= admissible[q]
        clear = np.abs(s64[q] - t) > GAP
        got = np.zeros_like(want)
        got[local] = True
        assert len(np.unique(local)) == len(local)
        assert np.array_equal(got[clear], want[clear]), q
        assert np.all(np.abs(sc.astype(np.float64) - s64[q, local]) <= GAP), q
        assert np.all(sc >= np.float32(t))
        if admissible is not None:
            assert admissible[q, local].all()
        order = np.lexsort((idx, -sc.astype(np.float64)))
        assert np.array_equal(order, np.arange(len(idx))), q


def _t_for(s64, per_query):
    return float(np.median(np.sort(s64, axis=1)[:, -per_query]))


@pytest.mark.parametrize("Q", [300, 40])            # CTA pairs / single CTAs (<= 128 queries)
@pytest.mark.parametrize("defer", [False, True])
def test_oracle_sets(eng, Q, defer):
    from emr2a_b200 import native
    rng = np.random.default_rng(Q + defer)
    N, D = 50_003, 1024                              # ragged: not a multiple of the 256-row tile
    db = rng.standard_normal((N, D), dtype=np.float32)
    qs = db[rng.choice(N, Q, replace=False)] + 0.6 * rng.standard_normal((Q, D), dtype=np.float32)
    s64 = _unit64(qs) @ _unit64(db).T
    t = _t_for(s64, 20)
    dbo = eng.prepare(db, None, 1.0, 1.0, native.NF_ROWNORM, "rescore", defer_f32=defer)
    assert (dbo.lazy is not None) == defer
    qo = eng.prepare(qs, None, 1.0, 1.0, native.NF_ROWNORM, "rescore")
    csr = eng.range_search_prepared(qo, dbo, t)
    _check_against(csr, s64, t)
    assert int(csr["offsets"][-1]) > 10 * Q


@pytest.mark.parametrize("Q", [300, 40])
def test_scores_bit_identical_to_rescore_topk(eng, Q):
    """t = the smallest 10th-best score of the batch: the first ten entries of every CSR row are the Top-K keys."""
    import torch
    from emr2a_b200 import native
    from emr2a_b200.engine import unpack_keys
    rng = np.random.default_rng(7 + Q)
    N, D, K = 50_000, 1024, 10
    db = rng.standard_normal((N, D), dtype=np.float32)
    qs = db[rng.choice(N, Q, replace=False)] + 0.8 * rng.standard_normal((Q, D), dtype=np.float32)
    dbo = eng.prepare(db, None, 1.0, 1.0, native.NF_ROWNORM, "rescore", defer_f32=True)
    qo = eng.prepare(qs, None, 1.0, 1.0, native.NF_ROWNORM, "rescore")
    keys = eng.topk_search(qo, dbo, K, "rescore")
    assert eng.consume_status()[1] is False
    sc, idx = unpack_keys(keys)
    t = float(sc[:, K - 1].min())
    csr = eng.range_search_prepared(qo, dbo, t)
    off = csr["offsets"].cpu().numpy()
    assert np.all(np.diff(off) >= K)
    first = (off[:-1, None] + np.arange(K)[None, :])
    got_idx = csr["idx"].cpu().numpy()[first]
    got_sc = csr["scores"].cpu().numpy()[first]
    assert np.array_equal(got_idx, idx)
    assert np.array_equal(got_sc.view(np.uint32), sc.view(np.uint32))
    torch.cuda.synchronize()


@pytest.mark.parametrize("defer", [False, True])
def test_bf16_inputs_wide_rows(eng, defer):
    """bf16 raw rows at D = 5120 (K1's block variant), Q = 130 (not a multiple of 128), ragged N."""
    import torch
    from emr2a_b200 import native
    rng = np.random.default_rng(5)
    N, Q, D = 20_011, 130, 5120
    db = torch.from_numpy(rng.standard_normal((N, D), dtype=np.float32)).to(torch.bfloat16)
    qs = (db[torch.from_numpy(rng.choice(N, Q, replace=False))].float()
          + 0.6 * torch.from_numpy(rng.standard_normal((Q, D), dtype=np.float32))).to(torch.bfloat16)
    s64 = _unit64(qs.float().numpy()) @ _unit64(db.float().numpy()).T
    t = _t_for(s64, 20)
    dbo = eng.prepare(db.to(eng.device), None, 1.0, 1.0, native.NF_ROWNORM, "rescore", defer_f32=defer)
    assert (dbo.lazy is not None) == defer
    qo = eng.prepare(qs.to(eng.device), None, 1.0, 1.0, native.NF_ROWNORM, "rescore")
    _check_against(eng.range_search_prepared(qo, dbo, t), s64, t)


def test_idx_base_empty_and_t_above_every_score(eng):
    from emr2a_b200 import native
    rng = np.random.default_rng(9)
    N, Q, D = 3000, 70, 256
    db = rng.standard_normal((N, D), dtype=np.float32)
    qs = db[:Q] + 0.3 * rng.standard_normal((Q, D), dtype=np.float32)
    s64 = _unit64(qs) @ _unit64(db).T
    t = _t_for(s64, 5)
    dbo = eng.prepare(db, None, 1.0, 1.0, native.NF_ROWNORM, "rescore")
    qo = eng.prepare(qs, None, 1.0, 1.0, native.NF_ROWNORM, "rescore")
    _check_against(eng.range_search_prepared(qo, dbo, t, idx_base=1_000_000), s64, t, idx_base=1_000_000)
    for t_hi in (1.5, float(s64.max()) + 1e-3):
        csr = eng.range_search_prepared(qo, dbo, t_hi)
        assert csr["offsets"].shape == (Q + 1,) and int(csr["offsets"].abs().sum()) == 0 and csr["idx"].numel() == 0
    csr = eng.range_search([db[:0]], [qs], 0.0)                          # empty database
    assert csr["offsets"].shape == (Q + 1,) and csr["idx"].numel() == 0
    with pytest.raises(ValueError, match="finite"):
        eng.range_search_prepared(qo, dbo, float("nan"))


@pytest.mark.parametrize("Q", [700, 100])            # CTA pairs / single CTAs
@pytest.mark.parametrize("sorted_folds", [True, False])
def test_fold_rule(eng, sorted_folds, Q):
    """Pairs with equal fold ids are excluded.  Sorted folds: whole tiles of the query's own fold are skipped."""
    rng = np.random.default_rng(13)
    N, D = 40_000, 512
    db = rng.standard_normal((N, D), dtype=np.float32)
    pick = rng.choice(N, Q, replace=False)
    qs = db[pick] + 0.5 * rng.standard_normal((Q, D), dtype=np.float32)
    db_fold = rng.integers(0, 5, N).astype(np.uint8)
    q_fold = db_fold[pick].copy()
    if sorted_folds:
        db_fold.sort(); q_fold.sort()
    s64 = _unit64(qs) @ _unit64(db).T
    t = _t_for(s64, 20)
    csr = eng.range_search([db], [qs], t, q_fold=q_fold, db_fold=db_fold)
    _check_against(csr, s64, t, admissible=q_fold[:, None] != db_fold[None, :])


@pytest.mark.parametrize("Q", [10, 300])             # single CTAs / CTA pairs
@pytest.mark.parametrize("sorted_folds", [True, False])
def test_lowest_finite_min_score_returns_every_admissible_pair(eng, Q, sorted_folds):
    """min_score = -FLT_MAX: t - E rounds to -inf, the value the epilogue gives the columns past N and the fold-masked
    pairs.  The cut is clamped, so the answer is every admissible pair and nothing else: indices < N (ragged N), no
    pair of one fold."""
    from emr2a_b200 import native
    rng = np.random.default_rng(37 + Q)
    N, D = 1000, 128
    db = rng.standard_normal((N, D), dtype=np.float32)
    qs = rng.standard_normal((Q, D), dtype=np.float32)
    db_fold = rng.integers(0, 5, N).astype(np.uint8)
    q_fold = rng.integers(0, 5, Q).astype(np.uint8)
    if sorted_folds:
        db_fold.sort(); q_fold.sort()
    t = float(np.finfo(np.float32).min)
    for defer in (False, True):
        dbo = eng.prepare(db, None, 1.0, 1.0, native.NF_ROWNORM, "rescore", defer_f32=defer)
        qo = eng.prepare(qs, None, 1.0, 1.0, native.NF_ROWNORM, "rescore")
        csr = eng.range_search_prepared(qo, dbo, t, q_fold=q_fold, db_fold=db_fold, fold_sorted=sorted_folds)
        s64 = _unit64(qs) @ _unit64(db).T
        admissible = q_fold[:, None] != db_fold[None, :]
        assert int(csr["offsets"][-1]) == int(admissible.sum())
        idx = csr["idx"].cpu().numpy()
        assert idx.min() >= 0 and idx.max() < N
        _check_against(csr, s64, t, admissible=admissible)


def test_unsupported_deferred_rows_fail_before_any_work(eng):
    """An operand error of the refine stage is reported before the filter runs: counts_out stays as it was."""
    import torch
    from emr2a_b200 import native
    from emr2a_b200.engine import _round_up, _ld
    rng = np.random.default_rng(41)
    N, Q, D = 2000, 20, 128
    db = rng.standard_normal((N, D), dtype=np.float32)
    dbo = eng.prepare(db, None, 1.0, 1.0, native.NF_ROWNORM, "rescore")
    qo = eng.prepare(db[:Q], None, 1.0, 1.0, native.NF_ROWNORM, "rescore")
    row_div = torch.ones((N, 4), dtype=torch.float32, device=eng.device)
    lz = native.LazyRows(dbo.f32.data_ptr(), dbo.f32.data_ptr(), D - 2, 2, D, D, native.F32, 1.0, 1.0,
                         native.NF_ROWNORM, row_div.data_ptr())            # segment widths not multiples of 4
    ws_bytes = int(eng.lib.emr2a_range_search_workspace_bytes(Q, N, D))
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=eng.device)
    cand = torch.zeros((64, 2), dtype=torch.int64, device=eng.device)
    out = torch.zeros((64, 2), dtype=torch.int64, device=eng.device)
    counts = torch.full((2,), 7, dtype=torch.int64, device=eng.device)
    import ctypes as C
    rc = eng.lib.emr2a_range_search(
        qo.f32.data_ptr(), _ld(qo.f32), qo.hi.data_ptr(), _ld(qo.hi), None, 0, dbo.hi.data_ptr(), _ld(dbo.hi), Q, N, D,
        None, None, 0, 0, -1.0, qo.stats.data_ptr(), dbo.stats.data_ptr(), cand.data_ptr(), 64, out.data_ptr(), 64,
        counts.data_ptr(), _round_up(ws.data_ptr(), 256), ws_bytes, C.byref(lz), eng._stream())
    torch.cuda.synchronize()
    assert rc == native.ERR_UNSUPPORTED and "deferred" in native.last_error()
    assert counts.tolist() == [7, 7] and int(cand.abs().sum()) == 0


def test_bf16_exact_ladder_around_t(eng):
    """bf16-exact rows (r_q = r_d = 0: the arithmetic term of E alone separates the rungs), a ladder of rows whose
    scores fall 5e-6 apart below the query's self-score, t between two rungs: exact membership."""
    from test_gpu_rescore_bound import _bf16_exact, _ulp_down
    rng = np.random.default_rng(17)
    N, D = 30_000, 5120
    db = _bf16_exact(rng.standard_normal((N, D)).astype(np.float32) / np.sqrt(D))
    q = _bf16_exact(rng.standard_normal((1, D)).astype(np.float32) / np.sqrt(D))[0]
    gap = 5e-6
    d = np.abs(q).astype(np.float64) * np.abs(q - _ulp_down(q, 1)).astype(np.float64)
    pool = [i for i in rng.permutation(D) if 0 < d[i] <= gap / 3]
    row, used = q.copy(), 0
    db[1000] = row
    for j in range(1, 80):
        drop = 0.0
        while drop < gap and used < len(pool):
            i = pool[used]; used += 1
            row[i] = _ulp_down(row[i:i + 1], 1)[0]
            drop += d[i]
        assert drop >= gap
        db[1000 + 17 * j] = row
    qs = np.repeat(q[None], 3, axis=0)
    truth = qs.astype(np.float64) @ db.astype(np.float64).T
    ladder = np.sort(truth[0][1000 + 17 * np.arange(80)])[::-1]
    t = float((ladder[40] + ladder[41]) / 2)
    assert min(ladder[40] - t, t - ladder[41]) > 2e-6
    dbo = eng.prepare(db, None, 1.0, 1.0, 0, "rescore")
    qo = eng.prepare(qs, None, 1.0, 1.0, 0, "rescore")
    csr = eng.range_search_prepared(qo, dbo, t)
    for k in range(3):
        idx, _ = _rows(csr, k)
        assert set(idx.tolist()) == set(np.flatnonzero(truth[k] >= t).tolist())
        assert len(idx) == 41


def test_overflow_counts_and_retry(eng):
    """The ABI counts are exact past the capacities; a retry with buffers of those sizes gives the Engine's CSR;
    max_results raises with the count."""
    import torch
    from emr2a_b200 import native
    from emr2a_b200.engine import _round_up, _ld, csr_from_pairs
    rng = np.random.default_rng(21)
    N, Q, D = 20_000, 200, 512
    db = rng.standard_normal((N, D), dtype=np.float32)
    qs = db[:Q] + 0.5 * rng.standard_normal((Q, D), dtype=np.float32)
    s64 = _unit64(qs) @ _unit64(db).T
    t = _t_for(s64, 15)
    dbo = eng.prepare(db, None, 1.0, 1.0, native.NF_ROWNORM, "rescore")
    qo = eng.prepare(qs, None, 1.0, 1.0, native.NF_ROWNORM, "rescore")
    ref = eng.range_search_prepared(qo, dbo, t)
    n_res = int(ref["offsets"][-1])
    ws_bytes = int(eng.lib.emr2a_range_search_workspace_bytes(Q, N, D))
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=eng.device)

    def call(cand_cap, res_cap):
        cand = torch.zeros((max(cand_cap, 1), 2), dtype=torch.int64, device=eng.device)
        out = torch.zeros((max(res_cap, 1), 2), dtype=torch.int64, device=eng.device)
        counts = torch.zeros(2, dtype=torch.int64, device=eng.device)
        native.check(eng.lib.emr2a_range_search(
            qo.f32.data_ptr(), _ld(qo.f32), qo.hi.data_ptr(), _ld(qo.hi), dbo.f32.data_ptr(), _ld(dbo.f32),
            dbo.hi.data_ptr(), _ld(dbo.hi), Q, N, D, None, None, 0, 0, t, qo.stats.data_ptr(), dbo.stats.data_ptr(),
            cand.data_ptr(), cand_cap, out.data_ptr(), res_cap, counts.data_ptr(), _round_up(ws.data_ptr(), 256),
            ws_bytes, None, eng._stream()))
        return counts.cpu().tolist(), out

    (c0, c1), _ = call(5, 3)                         # candidates overflow: nothing is re-scored
    assert c0 > n_res and c1 == 0
    (c0b, c1b), _ = call(c0, 3)                      # results overflow: both counts exact
    assert c0b == c0 and c1b == n_res
    (c0c, c1c), out = call(c0, n_res)
    assert (c0c, c1c) == (c0, n_res)
    csr = csr_from_pairs(out[:n_res], Q)
    for name in ("offsets", "idx", "scores"):
        assert torch.equal(csr[name], ref[name]), name
    with pytest.raises(ValueError, match=f"{n_res} results exceed|{c0} filter candidates exceed"):
        eng.range_search_prepared(qo, dbo, t, max_results=n_res - 1)


def test_cross_fold_duplicate_audit(eng):
    """20k two-modal cohort, StratifiedKFold(5, shuffle=True, random_state=42) folds, ~50 planted near-duplicates
    (cosine >= 0.999), some in the same fold, some across: the audit returns exactly the cross-fold pairs of float64
    brute force (pairs within 1e-5 of t excepted)."""
    import torch
    from sklearn.model_selection import StratifiedKFold
    from emr2a_b200 import synth
    data = synth.two_modal(20_000, 512, 512, 8, seed=23)
    img, txt, labels = data["image"], data["text"], data["labels"]
    folds = np.zeros(len(labels), dtype=np.uint8)
    for f, (_, te) in enumerate(StratifiedKFold(5, shuffle=True, random_state=42).split(img, labels)):
        folds[te] = f
    rng = np.random.default_rng(29)
    src = rng.choice(len(labels), 50, replace=False)
    dst = rng.choice(np.setdiff1d(np.arange(len(labels)), src), 50, replace=False)
    for a, b in zip(src, dst):
        scale = 0.01 * np.sqrt(np.sum(img[a] ** 2) + np.sum(txt[a] ** 2)) / np.sqrt(1024)
        img[b] = img[a] + scale * rng.standard_normal(512).astype(np.float32)
        txt[b] = txt[a] + scale * rng.standard_normal(512).astype(np.float32)
    same = folds[src] == folds[dst]
    assert 3 <= same.sum() <= 47
    t = 0.999
    res = eng.cross_fold_duplicates([img, txt], folds, t)
    x = torch.from_numpy(np.concatenate([img, txt], axis=1)).to(eng.device, torch.float64)
    x = x / (x.norm(dim=1, keepdim=True) + 1e-8)
    f_t = torch.from_numpy(folds).to(eng.device)
    want, near = set(), set()
    for lo in range(0, x.shape[0], 4096):
        s = x[lo:lo + 4096] @ x.T
        cross = f_t[lo:lo + 4096, None] != f_t[None, :]
        for i, j in torch.nonzero((s >= t) & cross).tolist():
            if lo + i < j:
                want.add((lo + i, j))
        for i, j in torch.nonzero(((s - t).abs() <= GAP) & cross).tolist():
            near.add((min(lo + i, j), max(lo + i, j)))
    i, j = res["i"].cpu().numpy(), res["j"].cpu().numpy()
    got = set(zip(i.tolist(), j.tolist()))
    assert np.all(i < j) and len(got) == len(i)
    assert got - near == want - near
    assert len(want) >= 50 - same.sum()
    assert np.array_equal(res["fold_i"].cpu().numpy(), folds[i]) and np.array_equal(res["fold_j"].cpu().numpy(), folds[j])
    assert np.all(folds[i] != folds[j]) and np.all(res["score"].cpu().numpy() >= np.float32(t))
    planted = {(min(a, b), max(a, b)) for a, b, sm in zip(src, dst, same) if not sm}
    assert planted <= got


def test_database_index_range_search(eng):
    rng = np.random.default_rng(31)
    N, Q = 30_000, 150
    img = rng.standard_normal((N, 256), dtype=np.float32)
    txt = rng.standard_normal((N, 256), dtype=np.float32)
    labels = rng.integers(0, 4, N).astype(np.int32)
    qi = img[:Q] + 0.5 * rng.standard_normal((Q, 256), dtype=np.float32)
    qt = txt[:Q] + 0.5 * rng.standard_normal((Q, 256), dtype=np.float32)
    t = 0.15                                         # about ten rows per query (scores of random 512-d rows: std 0.044)
    index = eng.build_index([img, txt], labels, 4, precision="rescore")
    a = index.range_search([qi, qt], t)
    b = eng.range_search([img, txt], [qi, qt], t)
    assert int(a["offsets"][-1]) > Q
    for name in ("offsets", "idx", "scores"):
        assert np.array_equal(a[name].cpu().numpy(), b[name].cpu().numpy()), name
    other = eng.build_index([img, txt], labels, 4, precision="bf16x3")
    with pytest.raises(ValueError, match="precision='rescore'"):
        other.range_search([qi, qt], t)


def test_full_size_c2_shape(eng):
    """C2 shape: 1M x 1024 database, 10k queries, t for about 20 rows per query; 32 sampled queries against float64
    scores over all rows."""
    import torch
    from emr2a_b200 import native, synth
    N, Q, D = 1_000_000, 10_000, 1024
    db, _ = synth.device_block(0, N, D, 16, seed=41, device=eng.device)
    qs, _ = synth.device_block(N, Q, D, 16, seed=41, device=eng.device)
    sample = np.random.default_rng(43).choice(Q, 32, replace=False)
    db64 = db.double()
    db64 /= db64.norm(dim=1, keepdim=True) + 1e-8
    q64 = qs[torch.from_numpy(sample).to(eng.device)].double()
    q64 /= q64.norm(dim=1, keepdim=True) + 1e-8
    s64 = (q64 @ db64.T).cpu().numpy()
    del db64
    t = _t_for(s64, 20)
    dbo = eng.prepare(db, None, 1.0, 1.0, native.NF_ROWNORM, "rescore", defer_f32=True)
    qo = eng.prepare(qs, None, 1.0, 1.0, native.NF_ROWNORM, "rescore")
    csr = eng.range_search_prepared(qo, dbo, t)
    n = int(csr["offsets"][-1])
    print(f"C2 range search: t={t:.5f}, {n} results, {n / Q:.1f} per query")
    assert 5 * Q < n < 80 * Q
    off = csr["offsets"].cpu().numpy()
    idx_all, sc_all = csr["idx"].cpu().numpy(), csr["scores"].cpu().numpy()
    for k, q in enumerate(sample):
        sub_off = np.array([0, off[q + 1] - off[q]])
        sub = {"offsets": torch.from_numpy(sub_off), "idx": torch.from_numpy(idx_all[off[q]:off[q + 1]]),
               "scores": torch.from_numpy(sc_all[off[q]:off[q + 1]])}
        _check_against(sub, s64[k:k + 1], t)
