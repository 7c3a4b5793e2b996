"""The range search's selection argument and host-side assembly, without a GPU (numpy / CPU torch stand-ins).

emr2a_range_search: the tensor-core filter emits every pair with s~ >= t - E, the exact re-scoring keeps s >= t.  With
|s~ - s| <= E that is exactly {d : s(q, d) >= t}, whatever the filter errors inside E are."""
import numpy as np
import torch

from emr2a_b200.engine import (cross_fold_pairs, csr_from_pairs, decode_keys, range_retry_caps,
                               unpack_keys)


def _pack(score, idx):
    """Packed keys of include/emr2a.h (numpy float32 scores, int indices) as int64."""
    b = np.asarray(score, dtype=np.float32).view(np.uint32).astype(np.uint64)
    o = np.where(b & np.uint64(0x80000000), ~b & np.uint64(0xFFFFFFFF), b ^ np.uint64(0x80000000))
    return ((o << np.uint64(32)) | (np.uint64(0xFFFFFFFF) - np.asarray(idx, dtype=np.uint64))).view(np.int64)


def _emit_keep(s, err, t, E):
    approx = s + err
    cand = approx >= t - E
    return cand & (s >= t), cand


def test_emit_within_bound_then_keep_equals_brute_force():
    rng = np.random.default_rng(0)
    for trial in range(200):
        E = float(rng.uniform(1e-4, 5e-3))
        t = float(rng.uniform(-0.5, 0.9))
        s = t + rng.uniform(-3 * E, 3 * E, 4096)
        s[:8] = t                                               # exact ties with t belong to the answer
        s[8:16] = np.nextafter(t, -np.inf)
        # adversarial filter errors inside the bound: the largest understatement for the members, the largest
        # overstatement for the rows just below t, random elsewhere
        err = rng.uniform(-E, E, s.shape)
        err[s >= t] = np.where(rng.random((s >= t).sum()) < 0.5, -E, err[s >= t])
        err[(s < t) & (s > t - E)] = E
        got, cand = _emit_keep(s, err, t, E)
        assert np.array_equal(got, s >= t), trial
        assert cand.sum() >= (s >= t).sum()


def test_a_cut_above_t_minus_E_misses_members():
    """The cut must be t - E rounded DOWN: at s = t with s~ = s - E, any larger cut drops a member."""
    t, E = 0.5, 3e-3
    s = np.array([t])
    cut = np.nextafter(np.float32(t - E), np.float32(1))
    assert not ((s - E) >= cut).any()
    assert ((s - E) >= t - E).all()


def test_csr_assembly_matches_a_python_sort():
    rng = np.random.default_rng(1)
    Q, n = 37, 5000
    q = rng.integers(0, Q, n)
    q[q == 5] = 6                                               # an empty row
    sc = rng.choice(np.float32([-0.5, -0.25, 0.0, 0.125, 0.5, 0.75]), n) + rng.integers(0, 3, n).astype(np.float32) * 1e-3
    idx = rng.permutation(1 << 20)[:n]
    pairs = torch.from_numpy(np.stack([q, _pack(sc, idx)], axis=1).astype(np.int64))
    csr = csr_from_pairs(pairs, Q)
    off = csr["offsets"].numpy()
    assert off[0] == 0 and off[-1] == n and off[6] == off[5]
    for k in range(Q):
        rows = sorted(((-float(sc[i]), int(idx[i])) for i in np.flatnonzero(q == k)))
        got = list(zip((-csr["scores"][off[k]:off[k + 1]].double()).tolist(), csr["idx"][off[k]:off[k + 1]].tolist()))
        assert got == rows, k
    empty = csr_from_pairs(torch.zeros((0, 2), dtype=torch.int64), 4)
    assert empty["offsets"].tolist() == [0, 0, 0, 0, 0] and empty["idx"].numel() == 0


def test_decode_keys_equals_unpack_keys():
    rng = np.random.default_rng(2)
    sc = np.concatenate([rng.standard_normal(1000).astype(np.float32), np.float32([0.0, -0.0, 1.0, -1.0, 3e-38])])
    idx = rng.integers(0, 0xFFFFFFFE, sc.shape)
    keys = torch.from_numpy(_pack(sc, idx))
    s1, i1 = decode_keys(keys)
    s2, i2 = unpack_keys(keys)
    assert np.array_equal(s1.numpy().view(np.uint32), s2.view(np.uint32)) and np.array_equal(i1.numpy(), i2)


def test_cross_fold_pair_extraction():
    """Self-join results (both directions of every pair, fold-ordered rows) -> each pair once, i < j in caller rows."""
    rng = np.random.default_rng(3)
    n = 300
    folds_caller = rng.integers(0, 5, n).astype(np.uint8)
    perm = np.argsort(folds_caller, kind="stable")             # fold-ordered row r is caller row perm[r]
    folds = folds_caller[perm]
    want = {}
    rows = []
    for _ in range(400):
        a, b = rng.integers(0, n, 2)
        if folds[a] == folds[b] or (min(perm[a], perm[b]), max(perm[a], perm[b])) in want:
            continue
        s = np.float32(rng.uniform(0.99, 1.0))
        want[(min(perm[a], perm[b]), max(perm[a], perm[b]))] = s
        rows += [(a, _pack(s, b)), (b, _pack(s, a))]
    order = rng.permutation(len(rows))
    pairs = torch.tensor([[int(rows[k][0]), int(rows[k][1])] for k in order], dtype=torch.int64)
    res = cross_fold_pairs(pairs, torch.from_numpy(perm), torch.from_numpy(folds))
    i, j = res["i"].numpy(), res["j"].numpy()
    assert np.all(i < j)
    assert sorted(zip(i.tolist(), j.tolist())) == list(zip(i.tolist(), j.tolist())) == sorted(want)
    assert np.array_equal(res["score"].numpy(), np.float32([want[k] for k in zip(i.tolist(), j.tolist())]))
    assert np.array_equal(res["fold_i"].numpy(), folds_caller[i]) and np.array_equal(res["fold_j"].numpy(), folds_caller[j])


def test_retry_sizing():
    import pytest
    assert range_retry_caps(10, 5, 100, 50, 1000) is None
    assert range_retry_caps(100, 50, 100, 50, 1000) is None                  # exactly full is complete
    assert range_retry_caps(101, 0, 100, 50, 1000) == (101, 101)             # candidates overflowed: results <= candidates
    assert range_retry_caps(5000, 0, 100, 50, 2000) == (5000, 2000)          # ... and never past max_results
    assert range_retry_caps(80, 60, 100, 50, 1000) == (100, 60)              # results overflowed: exact count
    with pytest.raises(ValueError, match="1001 results exceed max_results = 1000"):
        range_retry_caps(2000, 1001, 4000, 500, 1000)
    with pytest.raises(ValueError, match="4001 filter candidates"):
        range_retry_caps(4001, 0, 100, 50, 1000)
