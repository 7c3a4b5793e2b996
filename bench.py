"""EMR2A retrieval hot path benchmark (BASELINE.json metric: queries/sec, cosine Top-K + vote).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c1|c2|c2k5|c3|c4|c5|small]
                    [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline workload ("c2", BASELINE.json configs[1]): 1M-case database, 512-d image + 512-d text
embeddings (fp32, synthetic class-structured Gaussians), concat fusion to 1024-d, 10k queries,
K=10, 3 classes.  A STEP = the whole hot path over that batch:
    K1 normalise+fuse (database shard AND queries) -> K2 similarity + fused Top-K
    -> K3 merge -> [N > 1, cooperative shards: NCCL all-reduce (MAX) of the K-th best filter score, exact re-scoring,
    NCCL all-gather of exact Top-K + bounds, K3 merge, verification of the merged lists] -> K4 vote + metrics.
N > 1: the SAME 1M-row database is sharded row-wise over the ranks (strong scaling), and the line carries a "c5"
sub-record: BASELINE.json configs[4] (every case a query, 5-fold CV rule, K=5) on all N GPUs -- the full
10M-case cohort at N = 8, sqrt(N/8)-scaled row counts below (same per-GPU time), see run_c5.

value  : queries/sec with the raw embeddings resident in HBM.
e2e    : queries/sec through Engine.search_and_vote_host with the inputs in PINNED HOST
         memory: every step copies the database shard + queries host->device (chunked,
         overlapped with compute) and the results device->host.  N > 1: shards sized by each rank's measured
         concurrent H2D rate, query rows copied once per node and all-gathered over NVLink (emr2a_b200/dist.py).
roofline: the K2 kernel (tensor pipe) ALONE: algorithmic FLOPs 2*D*Q*N_local / its duration, from CUDA events the library
         records on the launching stream right before and after the kernel launch (emr2a_debug_tc_timing); the whole
         search call (kernel + merge of partial lists + re-scoring) is reported as search_ms; traffic = DRAM bytes
         of that kernel from the committed ncu capture listed in profiles/k2_traffic.json.
cpu_baseline: the reference's algorithm (oracle port: per-query np.dot sgemv over every admissible row + full np.argsort
         + python votes, utils/cv_evaluator.py:232-300) on the host cores for a SAMPLE of queries against ALL database
         rows, the database streamed from the GPU in chunks (oracle.StreamedReferenceSample), with the parity of the
         GPU results on that sample (index rows / votes under the gap rule) -- every workload, C2 to C5.
--impl reference: the same algorithm timed alone; inputs are the GPU arm's (synth.device_block on the box's GPU,
         copied to the host).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

if "reference" in sys.argv and os.environ.get("OMP_NUM_THREADS") == "1" and os.environ.get("TORCHELASTIC_RUN_ID"):
    # torchrun exports OMP_NUM_THREADS=1 to every rank and OpenBLAS sizes its pool from it when numpy loads; the
    # reference arm (rank 0 only, no GPU work) gets every host thread BLAS can use, as in the N=1 launch
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(os.cpu_count() or 1)

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

WORKLOADS = {
    # name: (n_db, d_img, d_txt, n_q, k, n_classes, seed)
    "c2": (1_000_000, 512, 512, 10_000, 10, 3, 11),
    "c2k5": (1_000_000, 512, 512, 10_000, 5, 3, 11),
    "small": (100_000, 256, 256, 2_048, 10, 3, 11),
    "c1": (2_000, 512, 512, 2_000, 5, 3, 7),     # BASELINE.json configs[0] (the reference's own CPU-sized case)
    # BASELINE.json configs[2]: late fusion (w_text*<T,T> + (1-w_text)*<I,I>, merge-then-Top-K), 5M cases
    "c3": (5_000_000, 512, 512, 10_000, 10, 3, 13),
    # BASELINE.json configs[3]: Qwen3-VL-shaped 4096-d image + 1024-d text, bf16 INPUTS, fp32 accumulation, 2M cases
    "c4": (2_000_000, 4096, 1024, 10_000, 10, 3, 17),
    # BASELINE.json configs[4]: every case is a query against the other folds (n_q == n_db); multi-GPU workload
    "c5": (10_000_000, 512, 512, -1, 5, 3, 19),
}
C3_W_TEXT = 0.25
Q_ROW0 = 50_003_968          # first synthetic row of the query block (far outside any database)
DUMP_BYTES = 64 << 20        # --dump-outputs: all files together
DUMP_QUERIES = 65536         # --dump-outputs: per-query arrays of larger workloads keep a seeded sample of this many rows
# --dump-outputs leaves out the packed (score, index) keys, which repeat top_scores / top_idx, and the rescore arm's
# internal status word
NOT_DUMPED = ("keys", "status")


def at_least(minimum):
    def parse_count(text):
        value = int(text)
        if value < minimum:
            raise argparse.ArgumentTypeError(f"must be >= {minimum}, got {value}")
        return value
    return parse_count


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=at_least(1), default=10, help="timed steps")
    ap.add_argument("--warmup", type=at_least(0), default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("EMR2A_BENCH_WORKLOAD", "c2"), choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default=os.environ.get("EMR2A_BENCH_PRECISION", "rescore"))
    ap.add_argument("--cpu-sample", type=int, default=int(os.environ.get("EMR2A_BENCH_CPU_SAMPLE", 32)))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-c5", action="store_true", help="N > 1: skip the C5 sub-record next to the C2 headline")
    ap.add_argument("--shard-of", type=int, default=int(os.environ.get("EMR2A_BENCH_SHARD_OF", 1)),
                    help="profiling aid (single GPU): search only shard 0 of this many row shards, i.e. the kernel a rank of "
                         "an N-GPU run launches -- ncu cannot follow a multi-rank job; the line is marked and is not a bench value")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the arrays the last timed step returned as DIR/<name>.npy "
                         "(see dump_outputs)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the b200 arm; --impl reference has none to write")
    return args


def dump_outputs(out_dir, results, n_queries):
    """Write what the last timed step returned to its caller as ``out_dir/<name>.npy``, so that two builds can be
    compared output for output: the inputs are seeded, the same arguments give the same arrays.  ``results`` maps
    names to tensors; those named in NOT_DUMPED are not written.  Floating-point arrays are written as float32
    (float64 stays float64), integer ones as float64, which holds every index and count exactly.  When there are
    more than DUMP_QUERIES queries, per-query arrays (first dimension ``n_queries``) keep a fixed, seeded sample of
    DUMP_QUERIES rows; their query numbers are written as query_rows.npy."""
    import torch
    rows = None
    if n_queries > DUMP_QUERIES:
        rows = np.sort(np.random.default_rng(0).choice(n_queries, DUMP_QUERIES, replace=False))
    arrays = {}
    for name, t in results.items():
        if not torch.is_tensor(t) or name in NOT_DUMPED:
            continue
        if rows is not None and t.dim() > 0 and t.shape[0] == n_queries:
            t = t[torch.from_numpy(rows).to(t.device)]
        a = t.cpu().numpy()
        arrays[name] = a.astype(np.float32 if a.dtype.kind == "f" and a.itemsize <= 4 else np.float64)
    if rows is not None:
        arrays["query_rows"] = rows.astype(np.float64)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_string(name, n_db=None):
    n, d_img, d_txt, n_q, k, n_cls, _ = WORKLOADS[name]
    n_db = n if n_db is None else n_db
    if name == "c5":
        return f"c5: {n_db}-case {d_img + d_txt}-d fused database, every case a query, 5-fold CV rule, K={k}"
    fusion = f"late fusion (w_text={C3_W_TEXT}, merge-then-Top-K)" if name == "c3" else "concat fusion"
    dtype = " (bf16 in)" if name == "c4" else " (fp32 in)"
    return f"{name}: {n_db}-case database, {d_img}+{d_txt}-d {fusion}{dtype}, {n_q} queries, K={k}, {n_cls} classes"


def peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return {"hbm_gbs": p["hbm_gbs"], "tflops": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "tflops_burst": p["bf16_tflops"], "src": "measured"}
    return {"hbm_gbs": 6650.0, "tflops": 1590.0, "tflops_burst": 1590.0, "src": "fallback"}


def tensor_peak(pk, load_seconds):
    """Roofline denominator for the tensor-bound kernel: MEASURED_PEAKS.json holds a burst figure (best of ten
    0.7 ms GEMMs, boost clocks) and a sustained one (GEMMs back to back for 4 s, power-capped clocks).
    ``load_seconds`` = continuous GPU load of the run (warm-up + timed steps).  Short runs (C2: 0.2 s) are compared
    with the burst figure -- the conservative choice --, runs that keep the GPU under load for 1.5 s or more
    (C4, C5) are in the power-capped regime the sustained figure describes.  Both fractions are reported."""
    if load_seconds >= 1.5:
        return pk["tflops"], f"bf16 sustained (continuous load {load_seconds:.1f} s >= 1.5 s)"
    return pk["tflops_burst"], f"bf16 burst (continuous load {load_seconds:.1f} s < 1.5 s)"


def device_index():
    """CUDA device of this rank.  With fewer ranks than visible GPUs the ranks are spread evenly over the devices
    (emr2a_b200.dist.spread_device: neighbouring GPUs share a host bridge and its host-memory bandwidth)."""
    from emr2a_b200.dist import spread_device
    lr = int(os.environ.get("LOCAL_RANK", 0))
    return spread_device(lr, int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", 1))))


def k2_traffic(workload, precision, world):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture for this workload
    (profiles/k2_traffic.json names the capture each figure comes from); None when there is no capture of it."""
    path = os.path.join(REPO, "profiles", "k2_traffic.json")
    try:
        with open(path) as fh:
            table = json.load(fh)
    except Exception:
        return None, None
    rec = table.get(f"{workload}/{precision}/{world}gpu")
    if not rec:
        return None, None
    return rec.get("dram_bytes_per_launch"), rec.get("source")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def summary(self, windows=None):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, r in list(self.rows):
            if windows and not any(a <= ts <= b + 0.12 for a, b in windows):
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for n, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "window": "timed regions, nvidia-smi -lms 100"}

    def stop(self, windows=None):
        """Summary of the samples that arrived inside the given (t0, t1) wall-clock windows (the timed regions)."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        return self.summary(windows)


def _oracle():
    sys.path.insert(0, os.path.join(REPO, "oracle"))
    import emr2a_oracle as oracle
    import streamed_feed
    return oracle, streamed_feed


def _blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return int(max([i.get("num_threads", 1) for i in threadpool_info()] or [1]))
    except Exception:
        return int(os.cpu_count() or 1)


def cpu_sample_leg(mode, k, n_db, fetch, q_img, q_txt, db_labels, q_labels, full_q, w_text=0.5, q_fold=None,
                   chunk_rows=65536, timed_rows=131072, prep_passes=1.0, got=None):
    """The reference's loop on the host cores for a sample of queries against ALL ``n_db`` rows (streamed through
    ``fetch``), its throughput extrapolated to the full workload, and the parity of the GPU results ``got``
    (dict of top_idx / top_scores / pred_vote / pred_weighted rows for the same queries) under the gap rule.
    ``prep_passes``: how many times the reference normalises/fuses an n_db-row matrix for the whole workload (1 for
    C2-C4; 5 for the 5-fold CV, whose train + test matrices add up to the cohort once per fold)."""
    oracle, feed = _oracle()
    s = oracle.StreamedReferenceSample(mode, k, n_db, q_img, q_txt, w_text=w_text, q_fold=q_fold)
    t0 = time.perf_counter()
    try:        # torchrun pins every rank to OMP_NUM_THREADS=1; the CPU leg (rank 0 only) may use every host thread
        from threadpoolctl import threadpool_limits
        limit = threadpool_limits(limits=os.cpu_count() or 1)
    except Exception:
        limit = None
    try:
        feed.feed(s, n_db, fetch, chunk_rows=chunk_rows, timed_rows=timed_rows)
        ref = s.finish(db_labels, q_labels)
        threads = _blas_threads()
    finally:
        if limit is not None:
            limit.restore_original_limits()
    wall = time.perf_counter() - t0
    t_prep, t_q = ref["prep_seconds"] * prep_passes, ref["seconds_per_query"]
    qps = full_q / (t_prep + full_q * t_q)
    info = {"value": qps, "unit": "queries/s", "cores": threads, "kind": "port",
            "sample": f"{len(q_labels)} of {full_q} queries, each scored against every admissible row of the {n_db}-row "
                      f"database (sgemv timed on the first {ref['timed_rows']} rows and scaled by rows; np.argsort over all "
                      f"{n_db} scores + python votes timed per query: {t_q * 1e3:.1f} ms/query) + database normalise/fuse "
                      f"({t_prep:.1f} s, from {ref['timed_prep_seconds']:.2f} s on the timed rows), extrapolated to the "
                      f"full step; {wall:.0f} s of host time; host has {os.cpu_count()} logical cores"}
    if got is not None:
        par = oracle.sample_parity(ref, got["top_idx"], got["top_scores"], got.get("pred_vote"), got.get("pred_weighted"))
        info["parity_on_sample"] = par
    return info, ref


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port; the reference is pure Python and /root/reference does
    not exist on the GPU box), every host thread BLAS can use.  Inputs: the GPU arm's own generator
    (``synth.device_block`` on the box's GPU, copied to the host) -- identical arrays.  A step = a bounded, proportional
    sample of the workload: ``sample`` of the n_q queries through the reference loop against the full prepared
    database (sgemv over all rows + full argsort + votes, utils/cv_evaluator.py:269-300) PLUS the same fraction of the
    database normalise/fuse pass (utils/cv_evaluator.py:95-105; n_db * sample / n_q rows re-done inside the step).
    ``value`` = sample / measured step time; ``ms_per_step`` is that measured time."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    import torch
    from emr2a_b200 import synth
    oracle, _ = _oracle()
    name = args.workload if args.workload != "c5" else "c2"
    n_db, d_img, d_txt, n_q, k, n_cls, seed = WORKLOADS[name]
    dev = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
    mode = "late" if name == "c3" else "concat"
    dt = torch.bfloat16 if name == "c4" else None

    def host_block(row0, rows, dim, s):
        out = np.empty((rows, dim), dtype=np.float32)
        for r0 in range(0, rows, 262144):
            r1 = min(r0 + 262144, rows)
            out[r0:r1] = synth.device_block(row0 + r0, r1 - r0, dim, n_cls, s, dev, label_seed=seed, dtype=dt)[0].float().cpu().numpy()
        return out
    img, txt = host_block(0, n_db, d_img, seed), host_block(0, n_db, d_txt, seed + 1)
    q_img, q_txt = host_block(Q_ROW0, n_q, d_img, seed), host_block(Q_ROW0, n_q, d_txt, seed + 1)
    db_lab = synth.device_labels(0, n_db, n_cls, seed, dev).cpu().numpy()
    q_lab = synth.device_labels(Q_ROW0, n_q, n_cls, seed, dev).cpu().numpy()

    def prep(a, b):
        if mode == "late":
            return oracle.unit_rows(a), oracle.unit_rows(b)
        return oracle.fuse_concat_cv(oracle.unit_rows(a), oracle.unit_rows(b))
    t0 = time.perf_counter()
    db = prep(img, txt)
    t_prep_full = time.perf_counter() - t0
    sample = max(4, min(args.cpu_sample, 16))
    share = max(1, n_db * sample // n_q)                       # database rows whose preparation belongs to one step
    times = []
    for s in range(args.warmup + args.steps):
        lo = (s * sample) % (n_q - sample)
        r0 = (s * share) % (n_db - share)
        t0 = time.perf_counter()
        prep(img[r0:r0 + share], txt[r0:r0 + share])            # this step's share of the normalise/fuse pass
        qs = prep(q_img[lo:lo + sample], q_txt[lo:lo + sample])
        if mode == "late":
            for i in range(sample):
                sims = C3_W_TEXT * np.dot(db[1], qs[1][i]) + (1 - C3_W_TEXT) * np.dot(db[0], qs[0][i])
                idx = np.argsort(sims)[-k:][::-1]
                labs = [int(db_lab[j]) for j in idx]
                oracle.vote_majority(labs), oracle.vote_weighted(labs, [float(sims[j]) for j in idx], "f64")
        else:
            oracle.reference_style_search_and_vote(qs, db, db_lab, q_lab[lo:lo + sample], k)
        dt_s = time.perf_counter() - t0
        if s >= args.warmup:
            times.append(dt_s)
    t_step = sum(times) / len(times)
    qps = sample / t_step
    threads = _blas_threads()
    line = {"impl": "reference", "metric": "queries/sec (cosine Top-K + vote)", "value": qps, "unit": "queries/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * t_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(name), "parallelism": "cpu",
                       "step": f"{sample} of the {n_q} queries (reference loop against the full {n_db}-row database) + the same "
                               f"fraction of the database normalise/fuse pass ({share} rows)",
                       "inputs": "synth.device_block on " + ("the box's GPU, copied to the host (the GPU arm's arrays)"
                                                             if dev.type == "cuda" else "the CPU generator (no GPU present)")},
            "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": threads, "kind": "port",
                             "sample": f"each step = {sample} queries against the full database + {share} database rows "
                                       f"normalised/fused; {os.cpu_count()} logical cores"},
            "extrapolated_full_step_ms": 1e3 * t_step * n_q / sample,
            "full_database_prepare_s": t_prep_full,
            "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def c5_rows_for(world):
    """Cohort size of the C5 record: the full 10M cases at 8 GPUs (and for an explicit EMR2A_C5_N); sqrt(world/8) of
    it below, which keeps the per-GPU work -- the pair count N^2 / world -- the same at every GPU count."""
    if "EMR2A_C5_N" in os.environ:
        return int(os.environ["EMR2A_C5_N"])
    n = WORKLOADS["c5"][0]
    if world >= 8:
        return n
    return int(round(n * (world / 8.0) ** 0.5 / 100_000.0)) * 100_000


def c5_record(args, eng, dev, world, rank, local_rank, n, steps, warm_full, cpu_sample, dump_dir=None):
    """BASELINE.json configs[4]: N-case 1024-d fused database, EVERY case a query, 5-fold CV rule (a case is never
    retrieved from its own fold), K=5.  Rows are in fold order (fold = contiguous fifths of the synthetic,
    label-shuffled rows) and sharded FOLD-BALANCED: rank r holds piece r of every fold (SURVEY 8e).  Per step and
    rank: K1 once on the shard; query blocks walked owner by owner, the owner's prepared rows broadcast over NVLink
    (double-buffered, block b+1 in flight while block b is searched); fold-masked K2 against the local shard (whole
    own-fold tiles skipped); all-gather of the local Top-K, K3 merge, K4 vote with per-fold counters
    (emr2a_b200/dist.py: sharded_cv_search_and_vote)."""
    import torch
    import torch.distributed as dist
    from emr2a_b200 import native, synth
    from emr2a_b200.dist import fold_balanced_ranges, ranges_to_rows, sharded_cv_search_and_vote

    _, d_img, d_txt, _, k, n_cls, seed = WORKLOADS["c5"]
    n_folds, dim = 5, d_img + d_txt
    q_block = int(os.environ.get("EMR2A_C5_QBLOCK", 262144))
    flags = native.NF_SEGNORM | native.NF_ROWNORM
    prec = args.precision

    def fold_vector(m):
        return (torch.arange(m, device=dev, dtype=torch.int64) * n_folds // m).to(torch.uint8)

    def build(m):
        fold = fold_vector(m)
        counts = torch.bincount(fold.long(), minlength=n_folds).cpu().tolist()
        ranges = fold_balanced_ranges(counts, rank, world)
        img = torch.cat([synth.device_block(g0, c, d_img, n_cls, seed, dev, label_seed=seed)[0] for g0, c in ranges])
        txt = torch.cat([synth.device_block(g0, c, d_txt, n_cls, seed + 1, dev, label_seed=seed)[0] for g0, c in ranges])
        return img, txt, synth.device_labels(0, m, n_cls, seed, dev), fold, ranges_to_rows(ranges, dev)

    def step(data, want_lists):
        img, txt, labels, fold, rows = data
        r = sharded_cv_search_and_vote(eng, (img, txt), labels, fold, n_cls, k, 0, flags, k_list=[1, 3, 5],
                                       precision=prec, n_folds=n_folds, q_block=q_block, fold_sorted=True,
                                       want_lists=want_lists, row_ids=rows)
        if r["precision"] != prec:
            raise RuntimeError("rescore re-scan list overflowed on this workload; run with --precision bf16x3")
        return r

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if not warm_full:                                   # sub-record: load the fold-masked kernels on a small cohort
        step(build(200_000), False)
    data = build(n)
    if warm_full:
        step(data, True)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    l0 = eng.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.time()
    e0.record()
    for _ in range(steps):
        out = step(data, True)
    e1.record()
    barrier()
    windows = [(w0, time.time())]
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0]) / steps
    clocks = sampler.stop(windows) if rank == 0 else None
    launches = eng.launches - l0
    peak_mem = torch.cuda.max_memory_allocated(dev)
    if rank == 0 and dump_dir:
        dump_outputs(dump_dir, out, n)
    rec = None
    if rank == 0:
        pk = peaks()
        hits, votes, sizes = out["hit_counts"], out["vote_counts"], out["group_sizes"]
        pairs = float(n) * float(n) * (1.0 - 1.0 / n_folds)          # same-fold pairs are not counted
        tf = 2.0 * dim * pairs / (ms / 1e3) / 1e12
        load = ms * (steps + (1 if warm_full else 0)) / 1e3
        t_peak, t_src = tensor_peak(pk, load)
        cpu = None
        if cpu_sample > 0:
            # oracle sample: `cpu_sample` cases spread over the folds, each against ALL cases of the other folds; the
            # cohort is regenerated chunk by chunk on this rank's GPU (the shards of the other ranks never leave them)
            _, feed = _oracle()
            pick = torch.linspace(0, n - 1, cpu_sample, device=dev).long()
            fold = data[3]
            q_img = torch.cat([synth.device_block(int(r), 1, d_img, n_cls, seed, dev, label_seed=seed)[0] for r in pick])
            q_txt = torch.cat([synth.device_block(int(r), 1, d_txt, n_cls, seed + 1, dev, label_seed=seed)[0] for r in pick])
            fetch = feed.generated_fetcher(lambda r0, m: synth.device_block(r0, m, d_img, n_cls, seed, dev, label_seed=seed)[0],
                                           lambda r0, m: synth.device_block(r0, m, d_txt, n_cls, seed + 1, dev, label_seed=seed)[0],
                                           lambda r0, m: fold[r0:r0 + m].cpu().numpy())
            got = {nm: out[nm][pick].cpu().numpy() for nm in ("top_idx", "top_scores", "pred_vote", "pred_weighted")}
            labels_h = data[2].cpu().numpy()
            cpu, _ = cpu_sample_leg("concat", k, n, fetch, q_img.cpu().numpy(), q_txt.cpu().numpy(), labels_h,
                                    labels_h[pick.cpu().numpy()], n, q_fold=fold[pick].cpu().numpy(), prep_passes=float(n_folds),
                                    got=got)
        rec = {"metric": "queries/sec (cosine Top-K + vote)", "value": n / (ms / 1e3), "unit": "queries/s", "n_gpus": world,
               "steps": steps, "warmup": 1 if warm_full else 0, "ms_per_step": ms, "higher_is_better": True,
               "scaling": "strong", "vs_baseline": None, "dtype": {"rescore": "bf16+f32"}.get(prec, prec), "data": "synthetic",
               "config": {"workload": workload_string("c5", n),
                          "parallelism": f"fold-balanced row shards x{world} (a slice of every fold per GPU); K1 once per shard; "
                                         f"query blocks of {q_block} prepared rows broadcast from their owner over NVLink "
                                         f"(double-buffered), searched locally; NCCL all-gather of local Top-K",
                          "l2": "inputs larger than L2"},
               "clocks": clocks, "e2e": None, "gpu_launches": launches,
               "roofline": {"bound": "tensor", "achieved": tf / world, "peak": t_peak, "unit": "TFLOP/s per GPU",
                            "frac": tf / world / t_peak, "peak_source": pk["src"] + " " + t_src,
                            "frac_of_burst": tf / world / pk["tflops_burst"], "frac_of_sustained": tf / world / pk["tflops"],
                            "traffic": None,
                            "note": "whole step (K1 + query-block broadcasts + K2 + key gather + K3 + K4) over admissible pairs only"},
               "cpu_baseline": cpu, "unverified_queries": int(out["unverified"]),
               "peak_memory_gb_rank0": peak_mem / 1e9,
               "accuracy": {"top1": float(hits[:, 0].sum()) / n, "top5": float(hits[:, 2].sum()) / n,
                            "vote_acc": float(votes[:, 1].sum()) / n,
                            "per_fold_top1": [float(hits[f, 0]) / max(float(sizes[f]), 1.0) for f in range(n_folds)]}}
    barrier()
    del data, out
    torch.cuda.empty_cache()
    return rec


def run_c5(args):
    import torch
    import torch.distributed as dist
    from emr2a_b200.engine import get_engine
    world = int(os.environ.get("WORLD_SIZE", 1)); rank = int(os.environ.get("RANK", 0))
    local_rank = device_index()
    torch.cuda.set_device(local_rank); dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    eng = get_engine(dev)
    n = int(os.environ.get("EMR2A_C5_N", WORKLOADS["c5"][0]))
    rec = c5_record(args, eng, dev, world, rank, local_rank, n, max(1, args.steps), warm_full=args.warmup > 0,
                    cpu_sample=0 if args.no_cpu_baseline else min(args.cpu_sample, 16), dump_dir=args.dump_outputs)
    if rank == 0:
        emit(rec)
    if world > 1:
        dist.destroy_process_group()


def run_c1(args):
    """BASELINE.json configs[0]: 2,000 cases, 512-d image + 512-d text, 3 classes, 5-fold CV, K=5, pca_dim=128.
    value : the GPU hot path from the processed (scaler+PCA'd, unit-row) arrays of all five folds.
    e2e   : CVRetrievalEvaluator.run_cv through the reference's own signature -- sklearn split/scaler/PCA on
            the host (93 % of the reference's wall time, SURVEY §0.5), GPU hot path, python list outputs.
    cpu_baseline : the same sklearn preprocessing + the oracle's per-query loop (the reference algorithm)."""
    import torch
    from emr2a_b200 import native, synth
    from emr2a_b200.engine import get_engine
    from emr2a_b200.utils.cv_evaluator import CVRetrievalEvaluator
    oracle, _ = _oracle()
    torch.cuda.set_device(0)
    eng = get_engine()
    n, d, n_cls, k = 2000, 512, 3, 5
    data = synth.two_modal(n, d, d, n_cls, seed=7)
    ids = synth.patient_ids(n)
    labels = synth.label_names(data["labels"], n_cls)
    emb = {pid: {"image": data["image"][j], "text": data["text"][j]} for j, pid in enumerate(ids)}
    ev = CVRetrievalEvaluator(cv_folds=5, pca_dim=128, top_k=k, seed=42)
    ev.preprocess = "host"
    # processed arrays per fold (host, sklearn) -- shared by the device-resident leg and the CPU leg
    np.random.seed(0)
    t0 = time.perf_counter()
    folds = []
    for tr_ids, te_ids in ev.stratified_split(ids, labels):
        tr = np.array([int(p[1:]) for p in tr_ids]); te = np.array([int(p[1:]) for p in te_ids])
        a_tr, a_te = ev.process_embeddings(data["image"][tr], data["image"][te])
        b_tr, b_te = ev.process_embeddings(data["text"][tr], data["text"][te])
        folds.append((tr, te, a_tr, b_tr, a_te, b_te))
    t_prep = time.perf_counter() - t0
    dev = [[torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in f[2:]] for f in folds]
    codes = data["labels"].astype(np.int32)
    lab = [(torch.from_numpy(codes[f[0]]).cuda(), torch.from_numpy(codes[f[1]]).cuda()) for f in folds]

    def gpu_pass():
        out = []
        for (a_tr, b_tr, a_te, b_te), (ltr, lte) in zip(dev, lab):
            out.append(eng.search_and_vote((a_tr, b_tr), (a_te, b_te), ltr, lte, n_cls, k, db_flags=native.NF_ROWNORM,
                                           q_flags=native.NF_ROWNORM, k_list=[1, 3, 5, 5]))
        return out
    for _ in range(max(args.warmup, 3)):
        res = gpu_pass()
    torch.cuda.synchronize()
    l0 = eng.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        res = gpu_pass()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    launches = eng.launches - l0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {f"fold{f + 1}_{name}": t for f, r in enumerate(res) for name, t in r.items()
                                         if name not in NOT_DUMPED}, n)
    # e2e: the public run_cv, host preprocessing (the reference's own sklearn calls)
    np.random.seed(0)
    t0 = time.perf_counter()
    full = ev.run_cv(ids, labels, emb, fusion="concat", top_k_list=[1, 3, 5, 5])
    t_e2e = time.perf_counter() - t0
    # the same public call as a user gets it by default (preprocess = "auto": scaler + exact PCA on the device
    # wherever sklearn's own solver choice is deterministic; otherwise sklearn on the host).  First call timed
    # separately: it creates the cuSOLVER handles (one-off, ~0.3 s); the steady-state call is what repeats.
    ev_def = CVRetrievalEvaluator(cv_folds=5, pca_dim=128, top_k=k, seed=42)
    t0 = time.perf_counter()
    ev_def.run_cv(ids, labels, emb, fusion="concat", top_k_list=[1, 3, 5, 5])
    torch.cuda.synchronize()
    t_e2e_default_first = time.perf_counter() - t0
    t0 = time.perf_counter()
    ev_def.run_cv(ids, labels, emb, fusion="concat", top_k_list=[1, 3, 5, 5])
    torch.cuda.synchronize()
    t_e2e_default = time.perf_counter() - t0
    # the same public call with the per-fold scaler + PCA on the device (SURVEY 8f-3; deterministic exact basis)
    ev_gpu = CVRetrievalEvaluator(cv_folds=5, pca_dim=128, top_k=k, seed=42)
    ev_gpu.preprocess = "gpu"
    ev_gpu.run_cv(ids, labels, emb, fusion="concat", top_k_list=[1, 3, 5, 5])          # warm-up (cuSOLVER handles)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    full_gpu = ev_gpu.run_cv(ids, labels, emb, fusion="concat", top_k_list=[1, 3, 5, 5])
    torch.cuda.synchronize()
    t_e2e_gpu = time.perf_counter() - t0
    # the API hot path alone: numpy in -> reference-shaped dict out, per fold (what evaluate_fold does after preprocessing)
    t0 = time.perf_counter()
    for tr, te, a_tr, b_tr, a_te, b_te in folds:
        ev.evaluate_processed_fold(a_tr, b_tr, a_te, b_te, [labels[j] for j in tr], [labels[j] for j in te],
                                   [ids[j] for j in te], fusion="concat", top_k_list=[1, 3, 5, 5], train_ids=[ids[j] for j in tr])
    t_api = time.perf_counter() - t0
    # CPU: oracle loop on the same processed arrays
    t0 = time.perf_counter()
    o = [oracle.cv_fold_eval(f[2], f[3], f[4], f[5], codes[f[0]], codes[f[1]], n_cls, fusion="concat", top_k=k,
                             top_k_list=(1, 3, 5, 5)) for f in folds]
    t_cpu = time.perf_counter() - t0
    same = float(np.mean([np.mean(np.all(r["top_idx"].cpu().numpy() == oo["top_idx"], axis=1)) for r, oo in zip(res, o)]))
    line = {"metric": "queries/sec (cosine Top-K + vote)", "value": n / (ms / 1e3), "unit": "queries/s", "n_gpus": 1,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": res[0]["precision"], "data": "synthetic",
            "config": {"workload": "c1: 2000 cases, 512+512-d, 3 classes, 5-fold CV, K=5, pca_dim=128 (concat fusion)",
                       "step": "five folds, from processed arrays: K1 fuse (db+queries) -> K2 -> K4",
                       "l2": "inputs (1.6 MB per fold) are L2-resident by nature of the configuration"},
            "clocks": None, "gpu_launches": launches,
            "e2e": {"value": n / t_e2e, "unit": "queries/s", "seconds": t_e2e,
                    "h2d_bytes_per_step": int(sum(x.numel() * 4 for f in dev for x in f)), "d2h_bytes_per_step": n * k * 16,
                    "api": "CVRetrievalEvaluator.run_cv, preprocess='host' (StratifiedKFold + StandardScaler + PCA by sklearn "
                           f"as in the reference, ~{t_prep:.2f} s; GPU hot path; python list outputs)",
                    "api_hot_path_seconds": t_api, "api_hot_path_qps": n / t_api,
                    "default_preprocess": {"mode": ev_def.preprocess, "value": n / t_e2e_default, "seconds": t_e2e_default,
                                           "first_call_seconds": t_e2e_default_first},
                    "gpu_preprocess": {"value": n / t_e2e_gpu, "unit": "queries/s", "seconds": t_e2e_gpu,
                                       "api": "CVRetrievalEvaluator.run_cv with preprocess='gpu' (StandardScaler + exact "
                                              "PCA on the device), python list outputs",
                                       "top1": float(np.mean([r["top1"] for r in full_gpu["fold_results"]])),
                                       "vote_acc": float(np.mean([r["vote_acc"] for r in full_gpu["fold_results"]]))}},
            "roofline": None,
            "cpu_baseline": {"value": n / (t_prep + t_cpu), "unit": "queries/s", "cores": os.cpu_count(), "kind": "port",
                             "sample": f"all 2000 queries: sklearn preprocessing {t_prep:.2f} s + oracle per-query loop {t_cpu:.2f} s",
                             "hot_path_only_qps": n / t_cpu, "parity": {"topk_rows_identical": same}},
            "accuracy": {"top1": float(np.mean([r["top1"] for r in full["fold_results"]])),
                         "vote_acc": float(np.mean([r["vote_acc"] for r in full["fold_results"]]))}}
    emit(line)


_REAL_STDOUT = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner to
    stdout on rank 0, python logging of the evaluators, ...), so file descriptor 1 is pointed at stderr for the
    whole run and the JSON line alone goes to the real stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    sys.stdout.flush()
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    args = parse()
    quiet_stdout()
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "c5":
        return run_c5(args)
    if args.workload == "c1":
        return run_c1(args)

    import torch
    import torch.distributed as dist
    from emr2a_b200 import native, synth
    from emr2a_b200.dist import gather_keys, h2d_rates, shard_range, sharded_search_and_vote, weighted_ranges
    from emr2a_b200.engine import get_engine

    world = int(os.environ.get("WORLD_SIZE", 1))
    rank = int(os.environ.get("RANK", 0))
    local_rank = device_index()           # the GPU of this rank: spread over the visible devices (dist.spread_device)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    eng = get_engine(dev)

    n_db, d_img, d_txt, n_q, k, n_cls, seed = WORKLOADS[args.workload]
    dim = d_img + d_txt
    lo, hi = shard_range(n_db, rank, world)
    if world == 1 and args.shard_of > 1:
        lo, hi = shard_range(n_db, 0, args.shard_of)
    flags = native.NF_SEGNORM | native.NF_ROWNORM          # normalise each modality, concat, normalise (a12+a13)
    q_weights = (1.0, 1.0)
    in_dtype = torch.float32
    if args.workload == "c3":                              # late fusion: unit modalities, weights folded into the queries
        flags = native.NF_SEGNORM
        q_weights = (np.float32(1 - C3_W_TEXT), np.float32(C3_W_TEXT))
    if args.workload == "c4":
        in_dtype = torch.bfloat16
    k_list = [1, 3, 5, k]

    # ---- synthetic inputs, generated on the device (per shard; same rows for any N) ----
    gen_dt = None if in_dtype == torch.float32 else in_dtype
    db_img, _ = synth.device_block(lo, hi - lo, d_img, n_cls, seed, dev, label_seed=seed, dtype=gen_dt)
    db_txt, _ = synth.device_block(lo, hi - lo, d_txt, n_cls, seed + 1, dev, label_seed=seed, dtype=gen_dt)
    # labels must be global (the vote gathers labels by global row index)
    db_labels = synth.device_labels(0, n_db, n_cls, seed, dev)
    q_img, q_labels = synth.device_block(Q_ROW0, n_q, d_img, n_cls, seed, dev, label_seed=seed, dtype=gen_dt)
    q_txt, _ = synth.device_block(Q_ROW0, n_q, d_txt, n_cls, seed + 1, dev, label_seed=seed, dtype=gen_dt)
    torch.cuda.synchronize()

    timers = {"k2_start": torch.cuda.Event(enable_timing=True), "k2_end": torch.cuda.Event(enable_timing=True)}
    k2_ms = []

    deferred = []      # rescore status of every timed step, verified right after the timed region (one sync)

    def step(record_k2=False):
        r = sharded_search_and_vote(eng, (db_img, db_txt), (q_img, q_txt), db_labels, q_labels, n_cls, k,
                                    row_offset=lo, db_flags=flags, q_flags=flags, q_weights=q_weights, k_list=k_list,
                                    precision=args.precision, timers=timers if record_k2 else None,
                                    defer_status=True)
        if "status" in r:
            deferred.append(r["status"])
        return r

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)      # started early: nvidia-smi needs ~0.2 s before its first sample
    if rank == 0:
        sampler.start()
    windows = []
    for attempt in range(2):
        for _ in range(max(args.warmup, 3)):
            res = step()
        barrier()
        deferred.clear()

        # ---- timed region: device-resident ----
        native.check(eng.lib.emr2a_debug_tc_timing(1))     # CUDA events around the Top-K kernel of every search (fresh series)
        launches0 = eng.launches
        w0 = time.time()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        k2_events = []
        for _ in range(args.steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            timers["k2_start"], timers["k2_end"] = e0, e1
            res = step(record_k2=True)
            k2_events.append((e0, e1))
        ev1.record()
        barrier()
        w1 = time.time()
        import ctypes as _C
        tc_buf = (_C.c_float * max(args.steps, 1))()
        tc_n = _C.c_int(0)
        native.check(eng.lib.emr2a_debug_tc_elapsed(tc_buf, max(args.steps, 1), _C.byref(tc_n)))
        native.check(eng.lib.emr2a_debug_tc_timing(0))
        tc_ms = [float(tc_buf[i]) for i in range(tc_n.value)]
        unverified_total, overflow = eng.check_deferred(deferred)
        if not overflow:
            windows.append((w0, w1))
            break
        # Cooperative shards defer the repair of queries the merged lists cannot verify (status[1]); a timed step that
        # needed it is not a valid step.  Every rank sees the same status, so all of them repeat the measurement with
        # self-contained shards (exact re-scan inside the step).
        assert attempt == 0 and world > 1 and os.environ.get("EMR2A_COOP_SHARDS", "1") != "0", \
            "rescore re-scan list overflowed: results of the timed steps are not valid"
        os.environ["EMR2A_COOP_SHARDS"] = "0"
    ms = ev0.elapsed_time(ev1)
    launches = eng.launches - launches0
    k2_ms = [a.elapsed_time(b) for a, b in k2_events]
    tc_avg = sum(tc_ms) / len(tc_ms) if tc_ms else 0.0
    t = torch.tensor([ms, sum(k2_ms) / len(k2_ms), tc_avg], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, k2_avg_ms, tc_avg_ms = float(t[0]), float(t[1]), float(t[2])
    if tc_avg_ms <= 0.0:                      # arms without a tensor-core kernel (fp32): the search call is the kernel
        tc_avg_ms = k2_avg_ms
    ms_per_step = ms_total / args.steps
    qps = n_q / (ms_per_step / 1e3)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, res, n_q)

    # ---- e2e: host (pinned) inputs through the public host-buffer API ----
    e2e = None
    if not args.no_e2e:
        # Host-resident shards: the step is bound by the copy to the device, and the ranks' links to host memory are
        # not equally fast under concurrent load (8-GPU boxes of this pool: 23 GB/s per GPU for GPUs 0-3, 35 GB/s for
        # GPUs 4-7, tools/h2d_probe.py).  The rows are therefore dealt out in proportion to each rank's measured
        # concurrent H2D rate, so that all ranks finish their copies together (dist.h2d_rates / weighted_ranges;
        # EMR2A_E2E_WEIGHTED=0: equal shards).  Row indices are global, the results do not depend on the split.
        e_lo, e_hi, h2d_gbs = lo, hi, None
        if world > 1 and os.environ.get("EMR2A_E2E_WEIGHTED", "1") != "0":
            h2d_gbs = h2d_rates(dev)
            e_lo, e_hi = weighted_ranges(n_db, h2d_gbs)[rank]
        if (e_lo, e_hi) == (lo, hi):
            h_img = db_img.cpu().pin_memory(); h_txt = db_txt.cpu().pin_memory()
        else:
            del db_img, db_txt
            h_img = synth.device_block(e_lo, e_hi - e_lo, d_img, n_cls, seed, dev, label_seed=seed, dtype=gen_dt)[0].cpu().pin_memory()
            h_txt = synth.device_block(e_lo, e_hi - e_lo, d_txt, n_cls, seed + 1, dev, label_seed=seed, dtype=gen_dt)[0].cpu().pin_memory()
            db_img = db_txt = None
        hq_img = q_img.cpu().pin_memory(); hq_txt = q_txt.cpu().pin_memory()
        h_lab = db_labels.cpu().pin_memory(); hq_lab = q_labels.cpu().pin_memory()

        def reduce_fn(keys):
            return eng.topk_merge(gather_keys(keys), k) if world > 1 else keys

        def e2e_step():
            return eng.search_and_vote_host((h_img, h_txt), (hq_img, hq_txt), h_lab, hq_lab, n_cls, k,
                                            db_flags=flags, q_flags=flags, q_weights=q_weights, k_list=k_list,
                                            precision=args.precision, row_offset=e_lo, reduce_fn=reduce_fn,
                                            gather_queries=world > 1 and os.environ.get("EMR2A_E2E_GATHER_Q", "1") != "0",
                                            chunk_rows=(int(os.environ["EMR2A_E2E_CHUNK"]) if "EMR2A_E2E_CHUNK" in os.environ else None))
        for _ in range(2):
            out = e2e_step()
        barrier()
        e_steps = max(2, min(args.steps, 5))
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
        w0 = time.time()
        t0.record()
        for _ in range(e_steps):
            out = e2e_step()
        t1.record()
        barrier()
        windows.append((w0, time.time()))
        te = torch.tensor([t0.elapsed_time(t1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e_ms = float(te[0]) / e_steps
        e2e = {"value": n_q / (e_ms / 1e3), "unit": "queries/s", "h2d_bytes_per_step": int(out["h2d_bytes"]),
               "d2h_bytes_per_step": int(out["d2h_bytes"]), "ms_per_step": e_ms,
               "api": "emr2a_b200.engine.Engine.search_and_vote_host (pinned host inputs, chunked H2D overlapped with K1/K2)"}
        if world > 1:
            e2e["h2d_bytes_per_step_note"] = "rank 0's bytes; every rank copies its own shard"
            if h2d_gbs is not None:
                e2e["shards"] = {"rows_rank0": e_hi - e_lo, "split": "proportional to each rank's concurrent H2D rate",
                                 "h2d_gbs_per_rank": [round(x, 1) for x in h2d_gbs]}
        # the two paths must agree bit for bit
        assert torch.equal(out["top_idx"], res["top_idx"].cpu()), "e2e and device-resident results differ"
        del h_img, h_txt
        # serving shape: the database stays resident in HBM (Engine.build_index), a step copies only the queries
        # host->device and the result lists device->host
        if world == 1:
            index = eng.build_index((db_img, db_txt), db_labels, n_cls, flags=flags, precision=args.precision,
                                    expected_queries=n_q, k=k)
            for _ in range(2):
                r2 = index.search((hq_img, hq_txt), hq_lab, k=k, q_weights=q_weights, k_list=k_list)
                lists = [r2[nm].cpu() for nm in ("top_idx", "top_scores", "top_labels", "pred_vote")]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(e_steps):
                r2 = index.search((hq_img, hq_txt), hq_lab, k=k, q_weights=q_weights, k_list=k_list)
                lists = [r2[nm].cpu() for nm in ("top_idx", "top_scores", "top_labels", "pred_vote")]
            torch.cuda.synchronize()
            r_ms = (time.perf_counter() - t0) / e_steps * 1e3
            assert torch.equal(lists[0], res["top_idx"].cpu())
            e2e["resident_index"] = {"value": n_q / (r_ms / 1e3), "unit": "queries/s", "ms_per_step": r_ms,
                                     "h2d_bytes_per_step": int(hq_img.numel() * hq_img.element_size() + hq_txt.numel() * hq_txt.element_size()
                                                               + hq_lab.numel() * 4),
                                     "api": "Engine.build_index once + DatabaseIndex.search per step (queries from pinned host memory)"}
            del index

    clocks = sampler.summary(windows) if rank == 0 else None

    # ---- roofline of the dominant kernel (K2, tensor pipe) ----
    coop_shards = world > 1 and res["precision"] == "rescore" and os.environ.get("EMR2A_COOP_SHARDS", "1") != "0"
    pk = peaks()
    flops = 2.0 * dim * n_q * (hi - lo)
    passes = {"bf16x3": 3, "bf16x1": 1, "fp32": 1, "rescore": 1}[res["precision"]]
    achieved = flops / (tc_avg_ms / 1e3) / 1e12       # the dominant kernel ALONE (events around its launch, on its stream)
    traffic, traffic_src = k2_traffic(args.workload, res["precision"], world)
    t_peak, t_src = tensor_peak(pk, ms_per_step * (args.steps + max(args.warmup, 3)) / 1e3)
    roofline = {"bound": "tensor", "achieved": achieved, "peak": t_peak, "unit": "TFLOP/s",
                "frac": achieved / t_peak, "traffic": traffic, "traffic_unit": "bytes per launch (ncu dram read+write)",
                "traffic_source": traffic_src,
                "peak_source": pk["src"] + " " + t_src,
                "frac_of_burst": achieved / pk["tflops_burst"], "frac_of_sustained": achieved / pk["tflops"],
                "kernel": "tc2_topk_kernel (tcgen05 cta_group::2, TMA, fused Top-K): one launch per step, timed alone by CUDA events "
                          "recorded on its stream right before and after the launch (emr2a_debug_tc_timing)",
                "kernel_ms": tc_avg_ms,
                "search_ms": k2_avg_ms,
                "search": ("emr2a_topk_filter = that kernel + K3 merge of its partial lists (the exact re-scoring follows the shards' "
                           "exchange of their K-th best filter score)" if coop_shards else
                           "emr2a_topk_search = that kernel + K3 merge of its partial lists"
                           + (" + exact fp32 re-scoring of the candidates + re-scan of unverifiable queries" if res["precision"] == "rescore" else "")),
                "search_tflops": flops / (k2_avg_ms / 1e3) / 1e12,
                "issued_tflops": achieved * passes, "issued_frac": achieved * passes / t_peak,
                "share_of_step": tc_avg_ms / ms_per_step}

    # ---- CPU baseline + parity on the sample (rank 0, N = 1): the reference loop against ALL database rows ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.shard_of == 1:
        _, feed = _oracle()
        pick = torch.linspace(0, n_q - 1, min(args.cpu_sample, n_q), device=dev).long()
        got = {nm: res[nm][pick].cpu().numpy() for nm in ("top_idx", "top_scores", "pred_vote", "pred_weighted")}
        wide = args.workload == "c4"
        cpu, _ = cpu_sample_leg("late" if args.workload == "c3" else "concat", k, n_db, feed.device_fetcher(db_img, db_txt),
                                q_img[pick].float().cpu().numpy(), q_txt[pick].float().cpu().numpy(),
                                db_labels.cpu().numpy(), q_labels[pick].cpu().numpy(), n_q, w_text=C3_W_TEXT,
                                chunk_rows=16384 if wide else 65536, timed_rows=32768 if wide else 131072, got=got)

    line = None
    if rank == 0:
        hits = res["hit_counts"][0].cpu().numpy()
        line = {"metric": "queries/sec (cosine Top-K + vote)", "value": qps, "unit": "queries/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": {"bf16x3": "bf16x3", "bf16x1": "bf16", "fp32": "f32", "rescore": "bf16+f32"}[res["precision"]],
                "data": "synthetic",
                "config": {"workload": workload_string(args.workload),
                           "parallelism": (f"database row-sharded x{world}, cooperative shards: NCCL all-reduce (MAX) of the K-th best filter "
                                           "score, exact re-scoring of the surviving candidates, NCCL all-gather of exact Top-K + bounds, "
                                           "verification of the merged lists" if coop_shards else
                                           f"database row-sharded x{world}, NCCL all-gather of local Top-K") if world > 1 else "single GPU",
                           "arithmetic": {"bf16x3": "tcgen05 bf16 2-way split (hi*lo + lo*hi + hi*hi), fp32 accumulate",
                                          "bf16x1": "tcgen05 bf16 operands, fp32 accumulate", "fp32": "CUDA-core fp32 FMA",
                                          "rescore": "tcgen05 bf16 filter (fp32 accumulate) + exact f32 re-scoring of the "
                                                     "candidates, selection verified by an error bound"}[res["precision"]],
                           "l2": "inputs (multi-GB database) larger than L2; no flush needed",
                           "step": "K1 normalise+fuse (db shard + queries) -> K2 GEMM+Top-K -> K3 merge -> K4 vote"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
                "unverified_queries": int(unverified_total),
                **({"profiling_aid": f"shard 0 of {args.shard_of} only ({hi - lo} rows): not a bench value"}
                   if world == 1 and args.shard_of > 1 else {}),
                "accuracy": {"top1": float(hits[0]) / n_q, f"top{k}": float(hits[3]) / n_q,
                             "vote_acc": float(res["vote_counts"][0, 1]) / n_q}}

    # ---- N > 1: BASELINE.json configs[4] on all N GPUs next to the C2 headline ----
    if world > 1 and args.workload == "c2" and not args.no_c5 and os.environ.get("EMR2A_BENCH_C5", "1") != "0":
        del db_img, db_txt, res
        torch.cuda.empty_cache()
        rec = c5_record(args, eng, dev, world, rank, local_rank, c5_rows_for(world), 1, warm_full=False,
                        cpu_sample=0 if args.no_cpu_baseline else min(args.cpu_sample, 16))
        if rank == 0:
            line["c5"] = rec
    if rank == 0:
        sampler.stop()
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
