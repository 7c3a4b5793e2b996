"""CPU-only checks: the C-ABI library builds, loads and exports every symbol the header
declares; host-side logic (label coding, metrics, splits, result materialisation)."""
import os
import re

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from emr2a_b200 import build, native
    build.build()
    return native.load()


def test_library_exports_every_header_symbol(lib):
    from emr2a_b200 import native
    header = open(os.path.join(REPO, "include", "emr2a.h")).read()
    declared = set(re.findall(r"\b(emr2a_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/emr2a.h but not exported"
        assert name in native.symbols(), f"{name} has no ctypes signature"
    assert lib.emr2a_abi_version() == native.ABI_VERSION
    m = re.search(r"#define EMR2A_ABI_VERSION (\d+)", header)
    assert int(m.group(1)) == native.ABI_VERSION


def test_binding_argument_lists_match_the_header():
    """Every ctypes signature has as many arguments as the C declaration, pointer / integer / float in the same places
    (an argument added on one side only would otherwise corrupt the call silently), and the emr2a_lazy_rows struct has
    the header's field order."""
    import ctypes as C
    from emr2a_b200 import native
    header = open(os.path.join(REPO, "include", "emr2a.h")).read()
    header = re.sub(r"/\*.*?\*/", " ", header, flags=re.S)
    decls = dict(re.findall(r"\b(?:int|size_t|const char\*)\s+(emr2a_[a-z0-9_]+)\s*\(([^;]*?)\)\s*;", header, flags=re.S))
    assert len(decls) >= 25
    def kind(param):
        param = param.strip()
        if "*" in param:
            return "p"
        if re.match(r"(const\s+)?float\b", param):
            return "f"
        return "i"
    for name, params in decls.items():
        res, args = native._SIGNATURES[name]
        plist = [] if params.strip() in ("", "void") else [x for x in params.split(",")]
        assert len(plist) == len(args), (name, len(plist), len(args))
        for param, ctype in zip(plist, args):
            want = kind(param)
            got = "f" if ctype is C.c_float else ("p" if (ctype is C.c_void_p or ctype is C.c_char_p or hasattr(ctype, "contents")) else "i")
            assert want == got, (name, param.strip(), ctype)
    m = re.search(r"typedef struct emr2a_lazy_rows \{(.*?)\} emr2a_lazy_rows;", header, flags=re.S)
    fields = [re.split(r"[\s\*]+", f.strip())[-1] for f in m.group(1).replace(",", ";").split(";") if f.strip()]
    assert fields == [n for n, _ in native.LazyRows._fields_], fields


def test_header_enums_match_binding():
    from emr2a_b200 import native
    header = open(os.path.join(REPO, "include", "emr2a.h")).read()
    for name, val in (("EMR2A_PREC_FP32", native.PREC_FP32), ("EMR2A_PREC_BF16X3", native.PREC_BF16X3),
                      ("EMR2A_PREC_BF16X1", native.PREC_BF16X1), ("EMR2A_NF_SEGNORM", native.NF_SEGNORM),
                      ("EMR2A_NF_ROWNORM", native.NF_ROWNORM), ("EMR2A_NF_ZERO_GUARD", native.NF_ZERO_GUARD),
                      ("EMR2A_SCORE_ZSCORE", native.SCORE_ZSCORE), ("EMR2A_SCORE_MINMAX", native.SCORE_MINMAX),
                      ("EMR2A_BF16", native.BF16), ("EMR2A_ERR_WORKSPACE", native.ERR_WORKSPACE)):
        m = re.search(name + r"\s*=\s*(\d+)", header)
        assert m and int(m.group(1)) == val, name


def test_product_path_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from emr2a_b200.engine import get_engine
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        get_engine()
    from emr2a_b200.retrieval import compute_cosine_similarity
    with pytest.raises(RuntimeError):
        compute_cosine_similarity(np.ones(4, np.float32), np.ones((2, 4), np.float32))


def test_product_never_imports_the_oracle():
    for root, _, files in os.walk(os.path.join(REPO, "emr2a_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(root, f)).read()
                assert "emr2a_oracle" not in src and "import oracle" not in src, f


def test_metrics_against_reference_golden(golden):
    from emr2a_b200.utils import (compute_accuracy, compute_confusion_matrix, compute_precision_recall_f1,
                                  compute_top_k_accuracy)
    g = golden("primitives.npz")
    names = lambda codes: [f"class_{int(c)}" for c in codes]      # noqa: E731
    labs = [f"class_{c}" for c in range(4)]
    pred, truth = names(g["m_pred"]), names(g["m_truth"])
    prf = compute_precision_recall_f1(pred, truth, labs)
    got = np.array([[prf[l]["precision"], prf[l]["recall"], prf[l]["f1"], prf[l]["support"]] for l in labs])
    np.testing.assert_allclose(got, g["m_prf"], atol=1e-15)
    cm = compute_confusion_matrix(pred, truth, labs)
    assert np.array_equal(np.array([[cm[a][b] for b in labs] for a in labs]), g["m_cm"])
    assert isinstance(cm["class_0"]["class_1"], int)
    assert compute_accuracy(pred, truth) == float(g["m_acc"])
    pl = [names(r) for r in g["m_predlists"]]
    assert compute_top_k_accuracy(pl, truth, 3) == float(g["m_top3"])
    with pytest.raises(ValueError, match="same length"):
        compute_accuracy(["a"], ["a", "b"])
    # labels outside the list are ignored by the confusion matrix, counted by P/R/F1
    cm = compute_confusion_matrix(["x", "a"], ["a", "a"], ["a"])
    assert cm == {"a": {"a": 1}}
    assert compute_precision_recall_f1(["x", "a"], ["a", "a"], ["a"])["a"]["recall"] == 0.5
    # prf_from_confusion == compute_precision_recall_f1 when every label is known
    from emr2a_b200.utils.metrics import prf_from_confusion
    p2 = prf_from_confusion(g["m_cm"], labs)
    for l in labs:
        for k in ("precision", "recall", "f1", "support"):
            assert p2[l][k] == prf[l][k]


def test_cv_stratified_split_matches_reference(golden):
    from emr2a_b200 import synth
    from emr2a_b200.utils.cv_evaluator import CVRetrievalEvaluator
    g = golden("cv_small.npz")
    n = int(g["meta"][0])
    ids = synth.patient_ids(n)
    labels = [f"class_{int(c)}" for c in g["labels"]]
    splits = CVRetrievalEvaluator(cv_folds=5, seed=42).stratified_split(ids, labels)
    assert len(splits) == 5
    for f, (tr, te) in enumerate(splits):
        assert tr == [ids[j] for j in g[f"f{f}_train_idx"]]
        assert te == [ids[j] for j in g[f"f{f}_test_idx"]]
        assert isinstance(tr, list) and isinstance(tr[0], str)


def test_holdout_stratified_split_matches_reference(golden):
    from emr2a_b200.retrieval import RetrievalEvaluator
    g = golden("holdout_small.npz")
    labels = ["solo" if c == 4 else f"class_{int(c)}" for c in g["ss_labels"]]
    ev = RetrievalEvaluator(test_ratio=0.2, seed=42)
    tr, te = ev.stratified_split(labels)
    assert tr == list(g["ss_train1"]) and te == list(g["ss_test1"])
    tr, te = ev.stratified_split(labels)
    assert tr == list(g["ss_train2"]) and te == list(g["ss_test2"])


def test_label_helpers():
    from emr2a_b200.labels import encode, gather_lists, score_lists
    classes, (a, b) = encode(["b", "a", "c"], ["c", "c"])
    assert classes == ["a", "b", "c"] and list(a) == [1, 0, 2] and list(b) == [2, 2] and a.dtype == np.int32
    idx = np.array([[2, 0], [1, -1]])
    valid = np.array([2, 1])
    assert gather_lists(["x", "y", "z"], idx, valid) == [["z", "x"], ["y"]]
    assert gather_lists(["x", "y", "z"], np.array([[2, 0], [1, 1]]), np.array([2, 2])) == [["z", "x"], ["y", "y"]]
    sl = score_lists(np.array([[0.5, 0.25], [0.125, 0.0]], dtype=np.float32), valid)
    assert sl == [[0.5, 0.25], [0.125]] and isinstance(sl[0][0], float)


def test_summary_and_serialisation_host_logic(tmp_path):
    from emr2a_b200.utils.cv_evaluator import CVRetrievalEvaluator
    ev = CVRetrievalEvaluator()
    folds = [{m: np.float64(0.1 * (i + 1)) for m in ("top1", "top3", "top5", "vote_acc", "weighted_vote_acc",
                                                     "macro_precision", "macro_recall", "macro_f1")} for i in range(5)]
    s = ev._compute_summary(folds)
    assert list(s) == ["top1", "top3", "top5", "vote_acc", "weighted_vote_acc", "macro_precision", "macro_recall", "macro_f1"]
    assert abs(s["top1"]["mean"] - 0.3) < 1e-12 and abs(s["top1"]["std"] - np.std([.1, .2, .3, .4, .5])) < 1e-12
    assert isinstance(s["top1"]["max"], float)
    out = ev._make_serializable({"a": np.float32(1.5), "b": [np.int64(2), np.bool_(True)], "c": np.arange(2)})
    assert out == {"a": 1.5, "b": [2, True], "c": [0, 1]} and type(out["b"][0]) is int
    ev._save_summary_csv(s, tmp_path / "s.csv")
    rows = open(tmp_path / "s.csv").read().strip().splitlines()
    assert rows[0] == "Metric,Mean,Std,Min,Max" and rows[1] == "top1,0.3000,0.1414,0.1000,0.5000"


def test_dropin_shims_exist_for_every_reference_module():
    base = os.path.join(REPO, "emr2a_b200", "dropin")
    assert os.path.exists(os.path.join(base, "retrieval", "__init__.py"))
    assert os.path.exists(os.path.join(base, "utils", "__init__.py"))
    import emr2a_b200.retrieval as r
    import emr2a_b200.utils as u
    assert r.__all__ == ["compute_cosine_similarity", "compute_euclidean_similarity", "late_fusion", "early_fusion",
                         "RetrievalEvaluator"]
    assert u.__all__ == ["l2_normalize", "concat_embeddings", "compute_accuracy", "compute_top_k_accuracy",
                         "compute_precision_recall_f1", "compute_confusion_matrix"]


# The next three tests launch the reference project's own scripts, so they need a checkout of it; the repository
# cannot carry that tree.  tests/test_gpu_scripts_replay.py checks the same entry points against stored outputs.
REFERENCE = os.environ.get("EMR2A_REFERENCE", "")
NO_REFERENCE = "set EMR2A_REFERENCE to a checkout of the reference project to run its scripts on the drop-in"


@pytest.mark.skipif(not (REFERENCE and os.path.isdir(os.path.join(REFERENCE, "pipelines"))), reason=NO_REFERENCE)
def test_reference_scripts_run_on_the_dropin(tmp_path):
    """The reference's own step-3 script, launched unchanged through emr2a_b200/run.py from the reference
    root, must reach THIS implementation: without a GPU it stops at our 'no CPU fallback' error instead of
    silently running the reference's numpy path; with a GPU it completes and writes retrieval_results.json."""
    import json
    import subprocess
    import sys
    rng = np.random.default_rng(0)
    manifest = tmp_path / "manifest.jsonl"
    emb = {}
    with manifest.open("w") as fh:
        for i in range(40):
            pid = f"p{i:03d}"
            fh.write(json.dumps({"patient_id": pid, "label": f"class_{i % 2}", "slices": [], "meta": {}}) + "\n")
            emb[pid] = rng.standard_normal((3, 16)).astype(np.float32)
    np.savez(tmp_path / "emb.npz", **emb)
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    env.pop("PYTHONPATH", None)
    out = subprocess.run([sys.executable, os.path.join(REPO, "emr2a_b200", "run.py"), "pipelines.step3_retrieval.run",
                          "--manifest_path", str(manifest), "--embeddings_path", str(tmp_path / "emb.npz"),
                          "--output_dir", str(tmp_path / "out")], cwd=REFERENCE, env=env, capture_output=True, text=True)
    import torch
    if torch.cuda.is_available():
        assert out.returncode == 0, out.stderr[-2000:]
        res = json.load(open(tmp_path / "out" / "retrieval_results.json"))
        assert set(res) == {"image_top1", "image_top3", "image_top5", "image_weighted"}
    else:
        assert out.returncode != 0
        assert "no CPU fallback" in out.stderr, out.stderr[-2000:]
        assert "emr2a_b200" in out.stderr


@pytest.mark.skipif(not (REFERENCE and os.path.isdir(os.path.join(REFERENCE, "analysis"))), reason=NO_REFERENCE)
def test_dropin_import_resolution_from_reference_root():
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r); import utils, retrieval, utils.cv_evaluator as c, utils.vlm_review as v; "
            "import pipelines.step3_retrieval.evaluate_retrieval as s3; "
            "print(c.CVRetrievalEvaluator.__module__, s3.RetrievalEvaluator.__module__, v.__file__)"
            % os.path.join(REPO, "emr2a_b200", "dropin"))
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    env.pop("PYTHONPATH", None)
    out = subprocess.run([sys.executable, "-c", code], cwd=REFERENCE, env=env, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr[-1500:]
    a, b, c = out.stdout.strip().splitlines()[-1].split()
    assert a == "emr2a_b200.utils.cv_evaluator" and b == "emr2a_b200.retrieval.evaluator"
    assert c == os.path.join(REFERENCE, "utils", "vlm_review.py")


def test_auto_mode_follows_sklearn_solver_choice():
    from emr2a_b200.utils.cv_evaluator import CVRetrievalEvaluator
    from emr2a_b200.retrieval.evaluator import RetrievalEvaluator
    ev = CVRetrievalEvaluator(pca_dim=128)
    assert ev.preprocess == os.environ.get("EMR2A_PREPROCESS", "auto")          # the default
    ev.preprocess = "auto"
    assert not ev._preprocess_on_gpu(240, 48)        # sklearn "full": deterministic there, 2e-4 from the exact basis -> host
    assert ev._preprocess_on_gpu(8000, 512)          # sklearn "covariance_eigh": 2e-6 from the exact basis -> device
    assert ev._preprocess_on_gpu(1600, 512)          # sklearn "randomized", unseeded in the reference -> device (C1's shape)
    ev.preprocess = "host"
    assert not ev._preprocess_on_gpu(240, 48)
    ev.preprocess = "bogus"
    with pytest.raises(ValueError):
        ev._preprocess_on_gpu(240, 48)
    ho = RetrievalEvaluator(use_pca=False)
    ho.preprocess = "auto"
    assert ho._preprocess_on_gpu(1600, 512)          # scaler only: bit-identical to sklearn
    ho = RetrievalEvaluator(use_pca=True, pca_dim=16)
    ho.preprocess = "auto"
    assert not ho._preprocess_on_gpu(200, 32) and ho._preprocess_on_gpu(5000, 64)


def test_public_signatures_match_the_reference():
    """Every public function / class / method of the reference's hot-path modules exists here under the same name with
    the same parameter names, order and defaults (tests/golden/signatures.json, recorded from the reference by
    tests/golden/make_signatures.py).  Extra methods and extra trailing keyword parameters with defaults are allowed."""
    import importlib
    import inspect
    import json
    with open(os.path.join(REPO, "tests", "golden", "signatures.json")) as fh:
        ref = json.load(fh)

    def check(where, fn, want):
        got = [[p.name, p.kind.name, None if p.default is inspect.Parameter.empty else repr(p.default)]
               for p in inspect.signature(fn).parameters.values()]
        assert got[:len(want)] == want, f"{where}: {got} != {want}"
        for extra in got[len(want):]:
            assert extra[2] is not None, f"{where}: extra parameter {extra[0]} has no default"

    import emr2a_b200.retrieval as ours_retrieval
    for name in ref.pop("retrieval.__all__"):
        assert callable(getattr(ours_retrieval, name)), name
    checked = 0
    for mod_name, api in ref.items():
        mod = importlib.import_module("emr2a_b200." + mod_name)
        for name, want in api.items():
            obj = getattr(mod, name)
            if isinstance(want, dict):
                for meth, sig in want["methods"].items():
                    check(f"{mod_name}.{name}.{meth}", getattr(obj, meth), sig)
                    checked += 1
            else:
                check(f"{mod_name}.{name}", obj, want)
                checked += 1
    assert checked >= 35


@pytest.mark.skipif(not (REFERENCE and os.path.isdir(os.path.join(REFERENCE, "analysis"))), reason=NO_REFERENCE)
def test_run_cv_experiments_script_reaches_the_dropin(tmp_path):
    """analysis/run_cv_experiments.py launched UNCHANGED through emr2a_b200/run.py from the reference root
    (--skip_encoding, the layout of :111-128): every import of the script resolves (encoders, utils.vlm_review through
    the drop-in package's extended path, utils.cv_evaluator = ours) and the run gets as far as the first kernel call
    of OUR CVRetrievalEvaluator -- which, without a GPU, stops with 'no CPU fallback' instead of running the
    reference's numpy loop.  (With a GPU it completes and writes the experiment directory; the value-for-value check
    of those files is tests/test_gpu_scripts_replay.py.)"""
    import json
    import subprocess
    import sys
    rng = np.random.default_rng(1)
    n = 60
    manifest = tmp_path / "manifest.jsonl"
    with manifest.open("w") as fh:
        for i in range(n):
            fh.write(json.dumps({"patient_id": f"p{i:03d}", "label": f"class_{i % 3}", "slices": [], "meta": {}}) + "\n")
    np.savez(tmp_path / "emb.npz", patient_ids=np.array([f"p{i:03d}" for i in range(n)], dtype=object),
             image_matrix=rng.standard_normal((n, 2, 24)).astype(np.float32),
             text_matrix=rng.standard_normal((n, 20)).astype(np.float32))
    # modules the reference imports at module level but that this image lacks (SURVEY App. D): stubbed via sitecustomize
    site = tmp_path / "site"
    site.mkdir()
    (site / "sitecustomize.py").write_text(
        "import sys, types, importlib.machinery as im\n"
        "def stub(name, **kw):\n"
        "    m = types.ModuleType(name); m.__spec__ = im.ModuleSpec(name, None); m.__path__ = []; m.__dict__.update(kw)\n"
        "    sys.modules[name] = m; return m\n"
        "noop = lambda *a, **k: None\n"
        "for name in ('qwen_vl_utils', 'timm', 'timm.data', 'open_clip'):\n"
        "    try:\n"
        "        __import__(name)\n"
        "    except Exception:\n"
        "        stub(name, process_vision_info=noop, create_transform=noop, resolve_data_config=noop, create_model=noop)\n")
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1", PYTHONPATH=str(site))
    out = subprocess.run([sys.executable, os.path.join(REPO, "emr2a_b200", "run.py"), "analysis.run_cv_experiments",
                          "--manifest_path", str(manifest), "--skip_encoding", "--embeddings_path", str(tmp_path / "emb.npz"),
                          "--output_dir", str(tmp_path / "out"), "--experiment_id", "t", "--pca_dim", "8", "--top_k", "3",
                          "--device", "cpu"], cwd=REFERENCE, env=env, capture_output=True, text=True)
    import torch
    if torch.cuda.is_available():
        assert out.returncode == 0, out.stderr[-3000:]
        m = json.load(open(tmp_path / "out" / "exp_t" / "fold_1" / "metrics.json"))
        assert {"all_top_labels", "all_top_scores", "all_top_patient_ids", "test_patient_ids", "top1"} <= set(m)
    else:
        assert out.returncode != 0
        assert "no CPU fallback" in out.stderr, out.stderr[-3000:]
        assert "emr2a_b200/utils/cv_evaluator.py" in out.stderr.replace("\\", "/")      # it was OUR evaluator that ran
        assert "Running experiment: t" in out.stderr                                      # the script's own driver code ran
