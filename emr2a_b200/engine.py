"""Host orchestration of the B200 retrieval hot path.

PyTorch is plumbing here (device memory, streams, pinned staging); every
computation is a libemr2a.so kernel reached through the C-ABI in
``include/emr2a.h``.  There is no CPU fallback.

Pipeline (per database/query pair):
    K1 normalize_fuse  ->  K2 topk_search (+K3 merge of partial lists)  ->  K4 vote_metrics
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import native

_PREC = {"fp32": native.PREC_FP32, "bf16x3": native.PREC_BF16X3, "bf16x1": native.PREC_BF16X1,
         "rescore": native.PREC_BF16_RESCORE}
_RESCORE_MAX_K = 10
_QPAD_MAX = int(os.environ.get("EMR2A_QPAD_MAX", 256))     # resident-index batches up to this size are filled to 64-row multiples
# tensor cores pay off once the contraction is large; below this the exact fp32 arm is used
_TC_MIN_MACS = float(os.environ.get("EMR2A_TC_MIN_MACS", 2.0e9))


def _round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


def _ld(t: torch.Tensor) -> int:
    """Leading dimension in elements (a 1-row tensor may carry an arbitrary row stride)."""
    return int(t.stride(0)) if t.shape[0] > 1 else int(t.shape[1])


@dataclass
class Operand:
    """Rows prepared by K1 for K2: fp32 rows and/or bf16 hi/lo planes."""
    n: int
    dim: int
    f32: Optional[torch.Tensor] = None      # [n, dim]
    hi: Optional[torch.Tensor] = None       # [n, ld] bf16 bits (int16 storage)
    lo: Optional[torch.Tensor] = None
    inv_norm: Optional[torch.Tensor] = None
    stats: Optional[torch.Tensor] = None    # [max row norm, max ||row - bf16(row)||]  (rescore error bound)
    lazy: Optional["DeferredRows"] = None   # rescore arm: fp32 rows re-created from the raw rows instead of ``f32``

    @property
    def ld_planes(self) -> int:
        return 0 if self.hi is None else self.hi.shape[1]


@dataclass
class DeferredRows:
    """Deferred fp32 rows (include/emr2a.h: emr2a_lazy_rows): the raw rows K1 read and the divisors it recorded.  The
    tensors are referenced here so they stay alive as long as the operand does."""
    seg0: torch.Tensor
    seg1: Optional[torch.Tensor]
    code: int
    w0: float
    w1: float
    flags: int
    row_div: torch.Tensor                   # float32 [n, 4]

    def struct(self, lo: int = 0, hi: Optional[int] = None) -> "native.LazyRows":
        a = self.seg0[lo:hi]
        b = self.seg1[lo:hi] if self.seg1 is not None else None
        return native.LazyRows(a.data_ptr(), b.data_ptr() if b is not None else None, int(a.shape[1]),
                               int(b.shape[1]) if b is not None else 0, _ld(a), _ld(b) if b is not None else 0, self.code,
                               float(self.w0), float(self.w1), int(self.flags), self.row_div[lo:hi].data_ptr())

    def slice(self, lo: int, hi: int) -> "DeferredRows":
        return DeferredRows(self.seg0[lo:hi], self.seg1[lo:hi] if self.seg1 is not None else None, self.code, self.w0,
                            self.w1, self.flags, self.row_div[lo:hi])


def _lazy_arg(op: "Operand"):
    """(ctypes argument, keep-alive) for the db_lazy parameter of the rescore entry points."""
    if op.lazy is None:
        return None, None
    st = op.lazy.struct()
    return C.byref(st), st


_DEFER_F32 = os.environ.get("EMR2A_DEFER_F32", "1") != "0"
# Deferred fp32 rows pay when re-creating elements is rare next to K1's saving: the re-scoring stage re-creates ~18 rows
# per query, and the exact re-scan of unverifiable queries is FILTERED (it streams the bf16 plane and re-creates only the
# rows within the error bound of the known K-th best score), so a pass costs the same on deferred and on materialised
# rows (profiles/r02_rescore_stages.md).  C4 (D = 5120, bf16 inputs): 174.6 -> 172.8 ms per step and 41 GB of HBM less.
# The UNFILTERED re-scan (exact_rescan without seed lists) re-creates the whole database at 2.8x the instructions of a
# pass over materialised rows; the pipelines always have seed lists.  Rows wider than this stay materialised.
_DEFER_MAX_DIM = int(os.environ.get("EMR2A_DEFER_MAX_DIM", 8192))


class Engine:
    """One engine per process/GPU (the multi-GPU path runs one process per GPU)."""

    def __init__(self, device: Optional[torch.device] = None):
        if not torch.cuda.is_available():
            raise RuntimeError("emr2a_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.lib = native.load()
        with torch.cuda.device(self.device):
            self.sm_count, self.cc_major, self.cc_minor = native.device_check()
        self.launches = 0       # kernels of ours launched through this engine (bench reports it)
        self._status_log: List[torch.Tensor] = []   # status_out of rescore searches not yet checked
        self._dense = set()     # (rows, dim) of databases whose score neighbourhoods defeated the rescore bound
        self.last_unverified: Optional[torch.Tensor] = None   # uint8 [Q] of the latest rescore search

    # ------------------------------------------------------------------ utils
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def to_device(self, x, dtype=None) -> torch.Tensor:
        if isinstance(x, np.ndarray):
            t = torch.from_numpy(np.ascontiguousarray(x))
        elif isinstance(x, torch.Tensor):
            t = x
        else:
            t = torch.as_tensor(np.asarray(x))
        if dtype is not None and t.dtype != dtype:
            t = t.to(dtype)
        if t.device != self.device:
            t = t.to(self.device, non_blocking=True)
        return t.contiguous()

    def _embedding(self, x) -> Tuple[torch.Tensor, int]:
        """Device matrix + emr2a dtype code.  float64/float16 inputs are computed in fp32."""
        if isinstance(x, np.ndarray) and x.dtype not in (np.float32,):
            x = x.astype(np.float32)
        t = self.to_device(x)
        if t.dtype == torch.bfloat16:
            code = native.BF16
        else:
            if t.dtype != torch.float32:
                t = t.float()
            code = native.F32
        if t.dim() == 1:
            t = t.unsqueeze(0)
        return t.contiguous(), code

    # --------------------------------------------------------------------- K1
    def normalize_fuse(self, seg0, seg1=None, w0: float = 1.0, w1: float = 1.0, flags: int = native.NF_ROWNORM,
                       want_f32: bool = True, want_planes: bool = False, want_lo: bool = True,
                       want_inv_norm: bool = False, want_stats: bool = False,
                       col_std: Optional[torch.Tensor] = None, defer_f32: bool = False) -> Operand:
        """K1.  ``col_std`` (float32 [3, d0 + d1]: per-column mean | scale | 1/scale of a fitted StandardScaler) with
        ``native.NF_STANDARDIZE`` in ``flags`` standardises the raw rows inside the same pass."""
        a, code = self._embedding(seg0)
        n, d0 = a.shape
        b = None
        d1 = 0
        if seg1 is not None:
            b, code_b = self._embedding(seg1)
            if b.shape[0] != n:
                raise ValueError("normalize_fuse: segments have different row counts")
            if code_b != code:
                a, b, code = a.float(), b.float(), native.F32
            d1 = b.shape[1]
        dim = d0 + d1
        out = Operand(n=n, dim=dim)
        row_div = None
        if defer_f32:          # no fp32 copy of the rows: K1 records its divisors, the search re-creates what it needs
            if not self.can_defer(a, b, flags):
                raise ValueError("normalize_fuse(defer_f32): needs segment widths / strides that are multiples of 4 and no fused standardisation")
            want_f32 = False
            row_div = torch.empty((n, 4), dtype=torch.float32, device=self.device)
            out.lazy = DeferredRows(a, b, code, float(w0), float(w1), int(flags), row_div)
        if want_f32:
            out.f32 = torch.empty((n, dim), dtype=torch.float32, device=self.device)
        ld_planes = 0
        if want_planes:
            ld_planes = _round_up(dim, 64)
            out.hi = torch.empty((n, ld_planes), dtype=torch.int16, device=self.device)
            if want_lo:
                out.lo = torch.empty((n, ld_planes), dtype=torch.int16, device=self.device)
        if want_inv_norm:
            out.inv_norm = torch.empty((n,), dtype=torch.float32, device=self.device)
        if want_stats and want_planes:
            out.stats = torch.zeros((2,), dtype=torch.float32, device=self.device)
        if n == 0:
            return out
        with torch.cuda.device(self.device):
            native.check(self.lib.emr2a_normalize_fuse(
                a.data_ptr(), native.ptr(b), n, d0, d1, _ld(a), _ld(b) if b is not None else 0,
                float(w0), float(w1), int(flags), code,
                native.ptr(out.f32), dim, native.ptr(out.hi), native.ptr(out.lo), ld_planes,
                native.ptr(out.inv_norm), native.ptr(out.stats), native.ptr(col_std), native.ptr(row_div), self._stream()))
        self.launches += 1
        return out

    @staticmethod
    def defer_default(dim: int) -> bool:
        """What the pipelines (search_and_vote, the sharded search, the host-buffer path) pass as ``defer_f32``."""
        return _DEFER_F32 and dim <= _DEFER_MAX_DIM

    @staticmethod
    def can_defer(a: torch.Tensor, b: Optional[torch.Tensor], flags: int) -> bool:
        """Shapes the deferred-fp32-rows arithmetic takes (row_math.cuh): 4-element chunks must not straddle segments."""
        if flags & native.NF_STANDARDIZE:
            return False
        al = 16 if a.dtype == torch.float32 else 8
        for t in (a, b):
            if t is None:
                continue
            if int(t.shape[1]) % 4 or (int(t.shape[0]) > 1 and int(t.stride(0)) % 4) or t.data_ptr() % al or t.stride(1) != 1:
                return False
        return True

    # ----------------------------------------------------------------- scores
    def scores(self, q: torch.Tensor, db: torch.Tensor) -> torch.Tensor:
        """Full fp32 score matrix [Q, N] (CUDA cores)."""
        q = self.to_device(q, torch.float32)
        db = self.to_device(db, torch.float32)
        if q.dim() == 1:
            q = q.unsqueeze(0)
        Q, D = q.shape
        N = db.shape[0]
        if db.shape[1] != D:
            raise ValueError(f"scores: query dim {D} != database dim {db.shape[1]}")
        out = torch.empty((Q, N), dtype=torch.float32, device=self.device)
        if Q and N:
            with torch.cuda.device(self.device):
                native.check(self.lib.emr2a_scores(q.data_ptr(), db.data_ptr(), Q, N, D, _ld(q), _ld(db),
                                                   out.data_ptr(), N, self._stream()))
            self.launches += 1
        return out

    def euclid_scores(self, q: torch.Tensor, db: torch.Tensor) -> torch.Tensor:
        q = self.to_device(q, torch.float32).reshape(-1)
        db = self.to_device(db, torch.float32)
        N, D = db.shape
        out = torch.empty((N,), dtype=torch.float32, device=self.device)
        ws = torch.empty((16,), dtype=torch.uint8, device=self.device)
        if N:
            with torch.cuda.device(self.device):
                native.check(self.lib.emr2a_euclid_scores(q.data_ptr(), db.data_ptr(), N, D, _ld(db),
                                                          out.data_ptr(), ws.data_ptr(), 16, self._stream()))
            self.launches += 2
        return out

    def late_fuse_scores(self, text_scores, image_scores, w_text: float, mode: int) -> torch.Tensor:
        ts = self.to_device(text_scores, torch.float32)
        im = self.to_device(image_scores, torch.float32)
        one_d = ts.dim() == 1
        if one_d:
            ts, im = ts.unsqueeze(0), im.unsqueeze(0)
        Q, N = ts.shape
        out = torch.empty((Q, N), dtype=torch.float32, device=self.device)
        if Q and N:
            with torch.cuda.device(self.device):
                native.check(self.lib.emr2a_late_fuse_scores(ts.data_ptr(), im.data_ptr(), Q, N, _ld(ts),
                                                             float(np.float32(w_text)), float(np.float32(1 - w_text)),
                                                             mode, out.data_ptr(), N, self._stream()))
            self.launches += 1
        return out[0] if one_d else out

    def topk_from_scores(self, scores, k: int) -> torch.Tensor:
        s = self.to_device(scores, torch.float32)
        if s.dim() == 1:
            s = s.unsqueeze(0)
        Q, N = s.shape
        keys = torch.zeros((Q, k), dtype=torch.int64, device=self.device)
        if Q and N:
            with torch.cuda.device(self.device):
                native.check(self.lib.emr2a_topk_from_scores(s.data_ptr(), Q, N, _ld(s), k, keys.data_ptr(),
                                                             self._stream()))
            self.launches += 1
        return keys

    def segment_mean(self, x, offsets) -> torch.Tensor:
        """Mean over the slices of each patient: rows [offsets[p], offsets[p+1]) of ``x`` -> row p."""
        x = self.to_device(x, torch.float32)
        off = self.to_device(offsets, torch.int64)
        n_seg = int(off.shape[0]) - 1
        out = torch.empty((max(n_seg, 0), x.shape[1]), dtype=torch.float32, device=self.device)
        if n_seg > 0:
            with torch.cuda.device(self.device):
                native.check(self.lib.emr2a_segment_mean(x.data_ptr(), _ld(x), off.data_ptr(), n_seg, int(x.shape[1]),
                                                         out.data_ptr(), int(x.shape[1]), self._stream()))
            self.launches += 1
        return out

    # --------------------------------------------------------------------- K2
    def pick_precision(self, Q: int, N: int, D: int, K: int, requested: str = "auto") -> str:
        req = os.environ.get("EMR2A_PRECISION", requested) if requested == "auto" else requested
        if req != "auto":
            if req not in _PREC:
                raise ValueError(f"unknown precision {req!r}")
            return req
        if float(Q) * float(N) * float(D) >= _TC_MIN_MACS:
            if K <= _RESCORE_MAX_K and (N, D) not in self._dense:
                return "rescore"
            if K <= 32:
                return "bf16x3"
        return "fp32"

    def prepare(self, seg0, seg1=None, w0=1.0, w1=1.0, flags=native.NF_ROWNORM, precision="fp32",
                defer_f32: bool = False) -> Operand:
        """K1 with the outputs the chosen K2 arm consumes.  ``defer_f32`` (rescore arm, DATABASE side): do not write the
        fp32 rows -- the search re-creates the few it needs from the raw rows (``DeferredRows``); silently falls back
        to materialised rows for shapes that arithmetic does not take or with ``EMR2A_DEFER_F32=0``."""
        if precision == "fp32":
            return self.normalize_fuse(seg0, seg1, w0, w1, flags, want_f32=True, want_planes=False)
        if precision == "rescore":
            if defer_f32 and _DEFER_F32:
                a = self._embedding(seg0)[0]
                b = self._embedding(seg1)[0] if seg1 is not None else None
                if (b is None or a.dtype == b.dtype) and self.can_defer(a, b, flags):
                    return self.normalize_fuse(a, b, w0, w1, flags, want_planes=True, want_lo=False, want_stats=True,
                                               defer_f32=True)
            return self.normalize_fuse(seg0, seg1, w0, w1, flags, want_f32=True, want_planes=True, want_lo=False,
                                       want_stats=True)
        return self.normalize_fuse(seg0, seg1, w0, w1, flags, want_f32=False, want_planes=True,
                                   want_lo=(precision == "bf16x3"))

    def topk_search(self, q: Operand, db: Operand, k: int, precision: str = "fp32",
                    q_fold: Optional[torch.Tensor] = None, db_fold: Optional[torch.Tensor] = None,
                    fold_sorted: bool = False, idx_base: int = 0, row_ids: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Packed Top-K keys [Q, k] (int64 storage of the uint64 keys), best first.  ``row_ids`` (int32 [N],
        ASCENDING): global index of every database row of this operand, for shards that are not one contiguous
        range (``emr2a_keys_map_rows``); default: ``idx_base + local row``."""
        if q.dim != db.dim:
            raise ValueError(f"topk_search: query dim {q.dim} != database dim {db.dim}")
        prec = _PREC[precision]
        Q, N, D = q.n, db.n, q.dim
        keys = torch.empty((Q, k), dtype=torch.int64, device=self.device)
        if Q == 0:
            return keys
        ws_bytes = int(self.lib.emr2a_topk_search_workspace_bytes(Q, N, D, k, prec))
        ws = torch.empty((ws_bytes + 256,), dtype=torch.uint8, device=self.device)
        ws_ptr = _round_up(ws.data_ptr(), 256)
        need_f32 = prec in (native.PREC_FP32, native.PREC_BF16_RESCORE)
        need_hi = prec != native.PREC_FP32
        lazy_arg, _lazy_keep = (None, None)
        if prec == native.PREC_BF16_RESCORE and db.f32 is None:
            lazy_arg, _lazy_keep = _lazy_arg(db)
        if need_f32 and (q.f32 is None or (db.f32 is None and lazy_arg is None)):
            raise ValueError(f"topk_search({precision}) needs fp32 operands")
        if need_hi and (q.hi is None or db.hi is None or (prec == native.PREC_BF16X3 and (q.lo is None or db.lo is None))):
            raise ValueError(f"topk_search({precision}) needs bf16 operand planes")
        status = None
        if prec == native.PREC_BF16_RESCORE:
            if q.stats is None or db.stats is None:
                raise ValueError("topk_search(rescore) needs operands prepared with stats")
            if k > _RESCORE_MAX_K:
                raise ValueError(f"topk_search(rescore): K={k} > {_RESCORE_MAX_K}")
            status = torch.zeros((4,), dtype=torch.int32, device=self.device)
            self.last_unverified = torch.empty((Q,), dtype=torch.uint8, device=self.device)
        if q_fold is not None:
            q_fold = self.to_device(q_fold, torch.uint8)
            db_fold = self.to_device(db_fold, torch.uint8)
        with torch.cuda.device(self.device):
            native.check(self.lib.emr2a_topk_search(
                native.ptr(q.f32), _ld(q.f32) if q.f32 is not None else 0,
                native.ptr(q.hi), native.ptr(q.lo), _ld(q.hi) if q.hi is not None else 0,
                native.ptr(db.f32), _ld(db.f32) if db.f32 is not None else 0,
                native.ptr(db.hi), native.ptr(db.lo), _ld(db.hi) if db.hi is not None else 0,
                Q, N, D, native.ptr(q_fold), native.ptr(db_fold), int(fold_sorted),
                int(idx_base), int(k), prec, native.ptr(q.stats), native.ptr(db.stats),
                keys.data_ptr(), native.ptr(status), native.ptr(self.last_unverified if status is not None else None),
                ws_ptr, ws_bytes, lazy_arg, self._stream()))
        self.launches += 2 if status is None else 6
        if status is not None:
            self._status_log.append(status)
        if row_ids is not None:
            row_ids = self.to_device(row_ids, torch.int32)
            if int(row_ids.shape[0]) != N:
                raise ValueError(f"topk_search: row_ids has {int(row_ids.shape[0])} entries for {N} database rows")
            with torch.cuda.device(self.device):
                native.check(self.lib.emr2a_keys_map_rows(keys.data_ptr(), Q * k, row_ids.data_ptr(), N, int(idx_base),
                                                          self._stream()))
            self.launches += 1
        return keys

    # ------------------------------------------------ K2 in stages (cooperative row shards, include/emr2a.h)
    CAND_WIDTH = 64

    def topk_filter(self, q: Operand, db: Operand, k: int, q_fold=None, db_fold=None, fold_sorted: bool = False,
                    idx_base: int = 0) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """Stage 1: tensor-core filter of this shard.  Returns (cand int64 [Q, 64], tau int32 [Q], kth float32 [Q])."""
        if q.hi is None or db.hi is None:
            raise ValueError("topk_filter needs bf16 operand planes")
        if k > _RESCORE_MAX_K:
            raise ValueError(f"topk_filter: K={k} > {_RESCORE_MAX_K}")
        Q, N, D = q.n, db.n, q.dim
        cand = torch.empty((Q, self.CAND_WIDTH), dtype=torch.int64, device=self.device)
        tau = torch.empty((Q,), dtype=torch.int32, device=self.device)
        kth = torch.empty((Q,), dtype=torch.float32, device=self.device)
        if Q == 0:
            return cand, tau, kth
        ws_bytes = int(self.lib.emr2a_topk_filter_workspace_bytes(Q, N, D, k))
        ws = torch.empty((ws_bytes + 256,), dtype=torch.uint8, device=self.device)
        if q_fold is not None:
            q_fold = self.to_device(q_fold, torch.uint8)
            db_fold = self.to_device(db_fold, torch.uint8)
        with torch.cuda.device(self.device):
            native.check(self.lib.emr2a_topk_filter(
                q.hi.data_ptr(), _ld(q.hi), db.hi.data_ptr() if N else None, _ld(db.hi) if N else 0, Q, N, D,
                native.ptr(q_fold), native.ptr(db_fold), int(fold_sorted), int(idx_base), int(k),
                cand.data_ptr(), tau.data_ptr(), kth.data_ptr(), _round_up(ws.data_ptr(), 256), ws_bytes, self._stream()))
        self.launches += 3
        return cand, tau, kth

    def rescore_candidates(self, cand: torch.Tensor, tau: torch.Tensor, kth_floor: Optional[torch.Tensor], q: Operand,
                           db: Operand, k: int, idx_base: int = 0) -> torch.Tensor:
        """Stage 3: exact fp32 scores of the candidates that can reach the global Top-K.  Returns ONE int64 buffer
        [Q*k + ceil(Q/2)] -- the shard's exact keys [Q, k] followed by its float32 bounds [Q] -- so that keys and
        bounds travel in a single all-gather (``split_payload`` takes it apart)."""
        lazy_arg, _lazy_keep = _lazy_arg(db) if db.f32 is None else (None, None)
        if q.f32 is None or (db.f32 is None and lazy_arg is None and db.n) or q.stats is None or db.stats is None:
            raise ValueError("rescore_candidates needs fp32 operands prepared with stats")
        Q, N, D = q.n, db.n, q.dim
        payload = torch.zeros((Q * k + (Q + 1) // 2,), dtype=torch.int64, device=self.device)
        if Q == 0:
            return payload
        keys, bounds = self.split_payload(payload, Q, k)
        if N == 0:
            bounds.fill_(float("-inf"))
            return payload
        with torch.cuda.device(self.device):
            native.check(self.lib.emr2a_rescore_candidates(
                cand.data_ptr(), tau.data_ptr(), native.ptr(kth_floor), q.f32.data_ptr(), _ld(q.f32), native.ptr(db.f32),
                _ld(db.f32) if db.f32 is not None else 0, Q, N, D, int(idx_base), int(k), q.stats.data_ptr(),
                db.stats.data_ptr(), keys.data_ptr(), bounds.data_ptr(), lazy_arg, self._stream()))
        self.launches += 1
        return payload

    @staticmethod
    def split_payload(payload: torch.Tensor, Q: int, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """payload [..., Q*k + ceil(Q/2)] int64 -> (keys [..., Q, k] int64, bounds [..., Q] float32), both views."""
        lead = payload.shape[:-1]
        keys = payload[..., :Q * k].unflatten(-1, (Q, k)) if lead else payload[:Q * k].view(Q, k)
        bounds = payload[..., Q * k:].view(torch.float32)[..., :Q]
        return keys, bounds

    def verify_merged(self, keys: torch.Tensor, all_payload: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """Stage 5.  ``keys`` [Q, k]: the merged exact lists; ``all_payload`` [P, Q*k + ceil(Q/2)]: the gathered stage-3
        buffers.  Returns (flags uint8 [Q], status int32 [4]); status[0] = number of flagged queries."""
        Q = int(keys.shape[0])
        P, width = all_payload.shape
        flags = torch.zeros((Q,), dtype=torch.uint8, device=self.device)
        status = torch.zeros((4,), dtype=torch.int32, device=self.device)
        if Q:
            bounds_ptr = all_payload.data_ptr() + 8 * Q * k
            with torch.cuda.device(self.device):
                native.check(self.lib.emr2a_verify_merged(keys.data_ptr(), int(k), Q, bounds_ptr, int(P),
                                                          int(all_payload.stride(0)) * 2, flags.data_ptr(),
                                                          status.data_ptr(), self._stream()))
            self.launches += 1
        return flags, status

    def merge_payload(self, all_payload: torch.Tensor, Q: int, k: int) -> torch.Tensor:
        """Stage 4: K3 merge of the key part of the gathered stage-3 buffers [P, Q*k + ceil(Q/2)] -> [Q, k]."""
        P = int(all_payload.shape[0])
        out = torch.empty((Q, k), dtype=torch.int64, device=self.device)
        if Q:
            with torch.cuda.device(self.device):
                native.check(self.lib.emr2a_topk_merge(all_payload.data_ptr(), P, Q, k, int(all_payload.stride(0)), k, k,
                                                       out.data_ptr(), self._stream()))
            self.launches += 1
        return out

    def exact_rescan(self, q: Operand, db: Operand, flag_list: torch.Tensor, k: int, idx_base: int = 0, q_fold=None,
                     db_fold=None, seed_keys: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Stage 6: exact fp32 search of this shard for the queries in ``flag_list`` (int32, the same on every shard).
        Returns compact keys [n_flagged, k].  With ``seed_keys`` [n_flagged, k] -- exact keys already known for these
        queries, e.g. the merged lists -- and operands prepared for the rescore arm (bf16 plane + stats) the re-scan is
        FILTERED: the plane is streamed and only rows within the error bound of the best known K-th exact score are
        scored exactly.  Every row of the exact Top-K passes; rows that cannot beat the seed's K-th best are dropped,
        so a shard may return fewer than k keys -- the merge over the shards is the exact Top-K."""
        flag_list = self.to_device(flag_list, torch.int32)
        n = int(flag_list.shape[0])
        out = torch.zeros((n, k), dtype=torch.int64, device=self.device)
        if n == 0:
            return out
        lazy_arg, _lazy_keep = _lazy_arg(db) if (db.f32 is None and db.n) else (None, None)
        if q.f32 is None or (db.n and db.f32 is None and lazy_arg is None):
            raise ValueError("exact_rescan needs fp32 operands")
        ws_bytes = int(self.lib.emr2a_exact_rescan_workspace_bytes(n, k))
        ws = torch.empty((ws_bytes + 256,), dtype=torch.uint8, device=self.device)
        if q_fold is not None:
            q_fold = self.to_device(q_fold, torch.uint8)
            db_fold = self.to_device(db_fold, torch.uint8)
        filtered = seed_keys is not None and db.hi is not None and q.stats is not None and db.stats is not None
        if seed_keys is not None:
            seed_keys = seed_keys.contiguous()
            if tuple(seed_keys.shape) != (n, k):
                raise ValueError(f"exact_rescan: seed_keys must be [{n}, {k}]")
        with torch.cuda.device(self.device):
            native.check(self.lib.emr2a_exact_rescan(
                q.f32.data_ptr(), _ld(q.f32), native.ptr(db.f32) if db.n else q.f32.data_ptr(),
                (_ld(db.f32) if db.f32 is not None else 0) if db.n else q.dim,
                db.n, q.dim, int(idx_base), int(k), native.ptr(q_fold), native.ptr(db_fold), flag_list.data_ptr(), n,
                out.data_ptr(), _round_up(ws.data_ptr(), 256), ws_bytes, lazy_arg,
                native.ptr(db.hi) if (filtered and db.n) else None, _ld(db.hi) if (filtered and db.n) else 0,
                native.ptr(q.stats) if filtered else None, native.ptr(db.stats) if filtered else None,
                native.ptr(seed_keys) if filtered else None, self._stream()))
        self.launches += 2
        return out

    def pop_status_tensor(self) -> Optional[torch.Tensor]:
        """Device-side status (int32[4], element-wise max over the pending rescore searches) without a
        host synchronisation; the caller decides when to look at it."""
        if not self._status_log:
            return None
        st = torch.stack(self._status_log)
        self._status_log = []
        return torch.stack([st[:, 0].sum(), st[:, 1].max(), st[:, 2].max(), st[:, 3].max()]).to(torch.int32)

    @staticmethod
    def check_deferred(statuses: Sequence[torch.Tensor]) -> Tuple[int, bool]:
        """Evaluate status tensors returned by calls made with ``defer_status=True`` (one sync for all)."""
        if not statuses:
            return 0, False
        st = torch.stack(list(statuses)).cpu().numpy()
        return int(st[:, 0].sum()), bool(st[:, 1].any())

    def consume_status(self) -> Tuple[int, bool]:
        """(number of queries the rescore bound could not verify -- they were re-searched exactly --,
        overflow of the re-scan list) over all rescore searches since the last call.  Synchronises."""
        if not self._status_log:
            return 0, False
        st = torch.stack(self._status_log).cpu().numpy()
        self._status_log = []
        return int(st[:, 0].sum()), bool(st[:, 1].any())

    # --------------------------------------------------------------------- K3
    def topk_merge(self, parts: torch.Tensor, k_out: int) -> torch.Tensor:
        """parts: [P, Q, K_in] packed keys -> [Q, k_out]."""
        P, Q, K_in = parts.shape
        parts = parts.contiguous()
        out = torch.empty((Q, k_out), dtype=torch.int64, device=self.device)
        if Q:
            with torch.cuda.device(self.device):
                native.check(self.lib.emr2a_topk_merge(parts.data_ptr(), P, Q, K_in, Q * K_in, K_in, k_out,
                                                       out.data_ptr(), self._stream()))
            self.launches += 1
        return out

    # --------------------------------------------------------------------- K4
    def vote_metrics(self, keys: torch.Tensor, db_labels, q_labels, n_classes: int,
                     k_list: Sequence[int] = (1, 3, 5), wacc_f32: bool = False,
                     q_group: Optional[torch.Tensor] = None, n_groups: int = 1, label_base: int = 0,
                     per_query: bool = True, want_lists: bool = True) -> Dict[str, torch.Tensor]:
        Q, K = keys.shape
        db_labels = self.to_device(db_labels, torch.int32)
        q_labels = self.to_device(q_labels, torch.int32)
        if q_group is not None:
            q_group = self.to_device(q_group, torch.uint8)
        nk = len(k_list)
        dev = self.device
        nk_alloc = max(nk, 1)                   # keep the hit-counter pointer non-null when k_list is empty
        counters = torch.zeros((n_groups * (nk_alloc + 3 + 1 + 2 * n_classes * n_classes),), dtype=torch.int64, device=dev)
        o = 0
        hit = counters[o:o + n_groups * nk_alloc]; o += n_groups * nk_alloc
        votes = counters[o:o + n_groups * 3]; o += n_groups * 3
        sizes = counters[o:o + n_groups]; o += n_groups
        conf = counters[o:]
        res: Dict[str, torch.Tensor] = {}
        if want_lists:
            res["top_idx"] = torch.empty((Q, K), dtype=torch.int64, device=dev)
            res["top_scores"] = torch.empty((Q, K), dtype=torch.float32, device=dev)
            res["top_labels"] = torch.empty((Q, K), dtype=torch.int32, device=dev)
        if per_query:
            for name in ("pred_top1", "pred_vote", "pred_weighted"):
                res[name] = torch.empty((Q,), dtype=torch.int32, device=dev)
        kl = (C.c_int32 * max(nk, 1))(*[int(k) for k in k_list])
        if Q:
            with torch.cuda.device(dev):
                native.check(self.lib.emr2a_vote_metrics(
                    keys.data_ptr(), Q, K, db_labels.data_ptr(), int(label_base), q_labels.data_ptr(),
                    native.ptr(q_group), n_groups, n_classes, kl, nk, int(wacc_f32),
                    native.ptr(res.get("top_idx")), native.ptr(res.get("top_scores")), native.ptr(res.get("top_labels")),
                    native.ptr(res.get("pred_top1")), native.ptr(res.get("pred_vote")), native.ptr(res.get("pred_weighted")),
                    hit.data_ptr(), votes.data_ptr(), conf.data_ptr(), sizes.data_ptr(), self._stream()))
            self.launches += 1
        res["hit_counts"] = hit.view(n_groups, nk_alloc)[:, :nk]
        res["vote_counts"] = votes.view(n_groups, 3)
        res["group_sizes"] = sizes
        res["confusion"] = conf.view(n_groups, 2, n_classes, n_classes)
        return res

    # --------------------------------------------------------- fused pipeline
    def search_and_vote(self, db_segs: Sequence, q_segs: Sequence, db_labels, q_labels, n_classes: int, k: int,
                        db_weights=(1.0, 1.0), q_weights=(1.0, 1.0), db_flags: int = native.NF_ROWNORM,
                        q_flags: int = native.NF_ROWNORM, k_list: Sequence[int] = (1, 3, 5),
                        precision: str = "auto", wacc_f32: bool = False, q_fold=None, db_fold=None,
                        q_group=None, n_groups: int = 1, want_lists: bool = True) -> Dict[str, torch.Tensor]:
        """normalize+fuse both sides, Top-K search, vote + metrics; everything stays on the device."""
        n_db = int(db_segs[0].shape[0])
        n_q = int(q_segs[0].shape[0])
        dim = sum(int(s.shape[1]) for s in db_segs if s is not None)
        prec = self.pick_precision(n_q, n_db, dim, k, precision)
        db = self.prepare(db_segs[0], db_segs[1] if len(db_segs) > 1 else None, db_weights[0], db_weights[1], db_flags, prec,
                          defer_f32=self.defer_default(dim))      # fp32 rows re-created for the re-scored candidates only
        qs = self.prepare(q_segs[0], q_segs[1] if len(q_segs) > 1 else None, q_weights[0], q_weights[1], q_flags, prec)
        keys = self.topk_search(qs, db, k, prec, q_fold=q_fold, db_fold=db_fold)
        res = self.vote_metrics(keys, db_labels, q_labels, n_classes, k_list=k_list, wacc_f32=wacc_f32,
                                q_group=q_group, n_groups=n_groups, want_lists=want_lists)
        if prec == "rescore":
            unverified, overflow = self.consume_status()      # the step's only host sync, after all work is queued
            if overflow:
                # More unverifiable queries than the exact re-scan list holds (dense score neighbourhoods):
                # re-search ONLY those queries with the 3-pass arm, patch their keys, vote again.
                flagged = torch.nonzero(self.last_unverified).squeeze(1)
                if int(flagged.numel()) * 2 > n_q:
                    self._dense.add((n_db, dim))      # mostly unverifiable: "auto" goes straight to bf16x3 next time
                q_dev = [self._embedding(s)[0].index_select(0, flagged) for s in q_segs if s is not None]
                db3 = self.prepare(db_segs[0], db_segs[1] if len(db_segs) > 1 else None, db_weights[0], db_weights[1],
                                   db_flags, "bf16x3")
                qs3 = self.prepare(q_dev[0], q_dev[1] if len(q_dev) > 1 else None, q_weights[0], q_weights[1], q_flags,
                                   "bf16x3")
                qf = self.to_device(q_fold, torch.uint8).index_select(0, flagged) if q_fold is not None else None
                keys3 = self.topk_search(qs3, db3, k, "bf16x3", q_fold=qf, db_fold=db_fold)
                keys.index_copy_(0, flagged, keys3)
                res = self.vote_metrics(keys, db_labels, q_labels, n_classes, k_list=k_list, wacc_f32=wacc_f32,
                                        q_group=q_group, n_groups=n_groups, want_lists=want_lists)
                res["precision"] = "rescore+bf16x3"
                res["unverified"] = int(flagged.numel())
                res["keys"] = keys
                return res
            res["unverified"] = unverified
        res["keys"] = keys
        res["precision"] = prec
        return res


    # ------------------------------------------------------ resident database
    def build_index(self, db_segs: Sequence, db_labels, n_classes: int, flags: int = native.NF_ROWNORM,
                    weights=(1.0, 1.0), precision: str = "auto", expected_queries: int = 4096, k: int = 10) -> "DatabaseIndex":
        """Prepare a database ONCE (K1: normalise + fuse + bf16 planes) and keep it in HBM; every later
        ``DatabaseIndex.search`` only pays for the queries.  The reference re-normalises the database on every
        call (retrieval/similarity.py:5-6); a serving deployment does not have to."""
        n_db = int(db_segs[0].shape[0])
        dim = sum(int(s.shape[1]) for s in db_segs if s is not None)
        prec = self.pick_precision(expected_queries, n_db, dim, k, precision)
        op = self.prepare(db_segs[0], db_segs[1] if len(db_segs) > 1 else None, weights[0], weights[1], flags, prec)
        return DatabaseIndex(self, op, self.to_device(db_labels, torch.int32), n_classes, flags, prec)

    # ------------------------------------------------- all folds at once (CV)
    @staticmethod
    def _rows(op: "Operand", lo: int, hi: int) -> "Operand":
        """View of rows [lo, hi) of a prepared operand (no copy)."""
        cut = lambda t: None if t is None else t[lo:hi]          # noqa: E731
        return Operand(n=hi - lo, dim=op.dim, f32=cut(op.f32), hi=cut(op.hi), lo=cut(op.lo),
                       inv_norm=cut(op.inv_norm), stats=op.stats)

    def cv_search_and_vote(self, segs: Sequence, labels, folds, n_classes: int, k: int,
                           flags: int = native.NF_ROWNORM, q_weights=(1.0, 1.0),
                           k_list: Sequence[int] = (1, 3, 5), precision: str = "auto",
                           n_folds: Optional[int] = None, q_block: int = 1 << 20,
                           want_lists: bool = True, distributed: Optional[bool] = None) -> Dict[str, torch.Tensor]:
        """The whole CV loop in one pass: every row is a query against the rows of the OTHER folds
        (utils/cv_evaluator.py:349-376 builds exactly these train/test pairs, one fold at a time).
        Rows are brought into fold order so the search can skip whole tiles of the query's own fold;
        indices and per-query outputs are mapped back to the caller's row order.  Counters are
        per fold (``hit_counts[f]``, ``vote_counts[f]``, ``confusion[f]``, ``group_sizes[f]``).
        Equals the reference's per-fold evaluation whenever the preprocessing does not depend on
        the fold (the rows passed in are the processed embeddings).
        ``distributed=True`` (or ``EMR2A_CV_DISTRIBUTED=1`` with the default ``None``): under ``torchrun`` with an
        NCCL process group, when every rank calls this with the same arrays (verified with a checksum), each rank
        searches against its own fold-balanced shard of the rows and the Top-K lists are exchanged over NCCL --
        same results, bit for bit, in 1/world of the time."""
        folds_t = self.to_device(folds, torch.uint8)
        n = int(folds_t.shape[0])
        if n_folds is None:
            n_folds = int(folds_t.max().item()) + 1 if n else 1
        labels_t = self.to_device(labels, torch.int32)
        mats = [self._embedding(x)[0] for x in segs if x is not None]
        perm = _fold_order(folds_t)
        if perm is not None:
            mats = [m.index_select(0, perm) for m in mats]
            labels_t = labels_t.index_select(0, perm)
            folds_t = folds_t.index_select(0, perm)
        dim = sum(int(m.shape[1]) for m in mats)
        prec = self.pick_precision(n, n, dim, k, precision)
        import torch.distributed as tdist
        if distributed is None:
            # sharding is opt-in: an NCCL group alone does not say that every rank holds the same cohort (ordinary
            # data-parallel callers pass different data per rank).  EMR2A_CV_DISTRIBUTED=1 turns the automatic mode on.
            distributed = (os.environ.get("EMR2A_CV_DISTRIBUTED") == "1" and tdist.is_available() and tdist.is_initialized()
                           and tdist.get_world_size() > 1 and tdist.get_backend() == "nccl")
        if distributed:
            # one process per GPU (torchrun), every rank called with the same arrays: this rank searches all queries
            # against ITS fold-balanced shard of the fold-ordered rows, query blocks travel from their owners and the
            # Top-K lists are exchanged over NCCL (emr2a_b200/dist.py)
            from .dist import fold_balanced_ranges, ranges_to_rows, sharded_cv_search_and_vote
            world, rank = tdist.get_world_size(), tdist.get_rank()
            # cheap guard against ranks that were handed different cohorts: (n, fold / label checksums) must agree
            sig = torch.stack([torch.tensor(float(n), device=self.device, dtype=torch.float64),
                               folds_t.double().sum(), (labels_t.double() * (torch.arange(n, device=self.device) % 8191 + 1)).sum()])
            lo_sig, hi_sig = sig.clone(), sig.clone()
            tdist.all_reduce(lo_sig, op=tdist.ReduceOp.MIN)
            tdist.all_reduce(hi_sig, op=tdist.ReduceOp.MAX)
            if not torch.equal(lo_sig, hi_sig):
                raise ValueError("cv_search_and_vote(distributed=True): the ranks were called with different cohorts "
                                 "(row count / fold / label checksums differ); every rank must pass the same arrays")
            counts = torch.bincount(folds_t.long(), minlength=n_folds).cpu().tolist()
            rows = ranges_to_rows(fold_balanced_ranges(counts, rank, world), self.device)
            res = sharded_cv_search_and_vote(self, [m.index_select(0, rows.long()) for m in mats], labels_t, folds_t,
                                             n_classes, k, 0, flags, q_weights, k_list, prec, n_folds,
                                             min(q_block, 1 << 18), True, want_lists, None, rows)
            return self._cv_unpermute(res, perm, want_lists)
        seg1 = mats[1] if len(mats) > 1 else None
        db = self.prepare(mats[0], seg1, 1.0, 1.0, flags, prec)
        same_q = float(q_weights[0]) == 1.0 and float(q_weights[1]) == 1.0
        qs_all = db if same_q else self.prepare(mats[0], seg1, q_weights[0], q_weights[1], flags, prec)
        outs: List[Dict[str, torch.Tensor]] = []
        unverified = 0
        for lo in range(0, n, q_block):
            hi = min(lo + q_block, n)
            keys = self.topk_search(self._rows(qs_all, lo, hi), db, k, prec, q_fold=folds_t[lo:hi], db_fold=folds_t,
                                    fold_sorted=True)
            r = self.vote_metrics(keys, labels_t, labels_t[lo:hi], n_classes, k_list=k_list, q_group=folds_t[lo:hi],
                                  n_groups=n_folds, want_lists=want_lists)
            r["keys"] = keys
            outs.append(r)
            if prec == "rescore":
                u, overflow = self.consume_status()
                if overflow:
                    return self.cv_search_and_vote(segs, labels, folds, n_classes, k, flags, q_weights, k_list,
                                                   "bf16x3", n_folds, q_block, want_lists, False)
                unverified += u
        res: Dict[str, torch.Tensor] = {}
        for name in ("hit_counts", "vote_counts", "confusion", "group_sizes"):
            res[name] = torch.stack([o[name] for o in outs]).sum(dim=0)
        per_query = [nm for nm in ("keys", "top_idx", "top_scores", "top_labels", "pred_top1", "pred_vote", "pred_weighted")
                     if nm in outs[0]]
        for name in per_query:
            res[name] = torch.cat([o[name] for o in outs])
        res["precision"] = prec
        res["unverified"] = unverified
        return self._cv_unpermute(res, perm, want_lists)

    @staticmethod
    def _cv_unpermute(res: Dict[str, torch.Tensor], perm: Optional[torch.Tensor], want_lists: bool) -> Dict[str, torch.Tensor]:
        """Per-query outputs of a fold-ordered CV pass back to the caller's row order / row numbers."""
        if perm is None:
            return res
        if "top_idx" in res:
            ti = res["top_idx"]
            res["top_idx"] = torch.where(ti >= 0, perm[ti.clamp(min=0)], ti)
        for name in ("top_idx", "top_scores", "top_labels", "pred_top1", "pred_vote", "pred_weighted"):
            if name in res:
                out = torch.empty_like(res[name])
                out[perm] = res[name]
                res[name] = out
        res.pop("keys", None)                                  # packed keys carry fold-order indices: not exported
        return res

    # ------------------------------------------------------------ range search
    def range_search(self, db_segs: Sequence, q_segs: Sequence, min_score: float, db_weights=(1.0, 1.0),
                     q_weights=(1.0, 1.0), db_flags: int = native.NF_ROWNORM, q_flags: int = native.NF_ROWNORM,
                     q_fold=None, db_fold=None, max_results: int = 1 << 26) -> Dict[str, torch.Tensor]:
        """Every admissible database row with exact fp32 score >= ``min_score``, per query -- not a fixed K.  K1 in the
        rescore layout (deferred database rows where ``defer_default`` says so), then ``emr2a_range_search``: the
        tensor-core filter emits every pair within the error bound below ``min_score`` and each is re-scored exactly,
        so the answer is exact and the scores equal the ones ``topk_search(precision="rescore")`` reports.  Weights
        and flags are those of ``search_and_vote`` (early / concat fusion, late fusion ``none``).  ``q_fold`` /
        ``db_fold``: the CV rule (pairs with equal fold ids are excluded).
        Returns a CSR dict: ``offsets`` int64 [Q+1], ``idx`` int64, ``scores`` float32; query q's rows are
        ``idx[offsets[q]:offsets[q+1]]``, by score descending, then index ascending.  More than ``max_results`` results
        (or more than 4 x ``max_results`` filter candidates) raise ValueError before any buffer of that size is made."""
        dim = sum(int(s.shape[1]) for s in db_segs if s is not None)
        db = self.prepare(db_segs[0], db_segs[1] if len(db_segs) > 1 else None, db_weights[0], db_weights[1], db_flags,
                          "rescore", defer_f32=self.defer_default(dim))
        qs = self.prepare(q_segs[0], q_segs[1] if len(q_segs) > 1 else None, q_weights[0], q_weights[1], q_flags, "rescore")
        fold_sorted = False
        if (q_fold is None) != (db_fold is None):
            raise ValueError("range_search: q_fold and db_fold must be given together")
        if q_fold is not None:
            q_fold = self.to_device(q_fold, torch.uint8)
            db_fold = self.to_device(db_fold, torch.uint8)
            fold_sorted = _non_decreasing(q_fold) and _non_decreasing(db_fold)
        return self.range_search_prepared(qs, db, min_score, q_fold, db_fold, fold_sorted, max_results=max_results)

    def range_search_prepared(self, q: Operand, db: Operand, min_score: float, q_fold=None, db_fold=None,
                              fold_sorted: bool = False, idx_base: int = 0, max_results: int = 1 << 26
                              ) -> Dict[str, torch.Tensor]:
        """``range_search`` on operands prepared for the rescore arm (``prepare(..., "rescore")``).  ``fold_sorted``
        promises non-decreasing fold vectors (whole tiles of the query's own fold are skipped); ``idx_base`` is added
        to the database row numbers."""
        pairs = self._range_pairs(q, db, min_score, q_fold, db_fold, fold_sorted, idx_base, max_results)
        return csr_from_pairs(pairs, q.n)

    def _range_pairs(self, q: Operand, db: Operand, min_score: float, q_fold, db_fold, fold_sorted: bool, idx_base: int,
                     max_results: int, first_per_query: int = 32) -> torch.Tensor:
        """The ABI call (plus at most one retry with buffers sized from the counts): int64 [n, 2] (query, key).  The
        first call holds ``first_per_query`` results and four times as many candidates per query."""
        if q.dim != db.dim:
            raise ValueError(f"range_search: query dim {q.dim} != database dim {db.dim}")
        if not np.isfinite(min_score):
            raise ValueError(f"range_search: min_score must be finite, got {min_score}")
        lazy_arg, _lazy_keep = _lazy_arg(db) if db.f32 is None else (None, None)
        if q.f32 is None or (db.f32 is None and lazy_arg is None) or q.hi is None or db.hi is None or q.stats is None \
                or db.stats is None:
            raise ValueError("range_search needs operands prepared for the rescore arm (fp32 rows, bf16 planes, stats)")
        Q, N, D = q.n, db.n, q.dim
        if Q == 0 or N == 0:
            return torch.zeros((0, 2), dtype=torch.int64, device=self.device)
        if q_fold is not None:
            q_fold = self.to_device(q_fold, torch.uint8)
            db_fold = self.to_device(db_fold, torch.uint8)
        ws_bytes = int(self.lib.emr2a_range_search_workspace_bytes(Q, N, D))
        ws = torch.empty((ws_bytes + 256,), dtype=torch.uint8, device=self.device)

        def call(cand, cand_cap, out, res_cap, counts):
            return self.lib.emr2a_range_search(
                q.f32.data_ptr(), _ld(q.f32), q.hi.data_ptr(), _ld(q.hi), native.ptr(db.f32),
                _ld(db.f32) if db.f32 is not None else 0, db.hi.data_ptr(), _ld(db.hi), Q, N, D,
                native.ptr(q_fold), native.ptr(db_fold), int(fold_sorted), int(idx_base), float(min_score),
                q.stats.data_ptr(), db.stats.data_ptr(), cand.data_ptr(), cand_cap, out.data_ptr(), res_cap,
                counts.data_ptr(), _round_up(ws.data_ptr(), 256), ws_bytes, lazy_arg, self._stream())
        return self._pairs_with_retry(call, min(max_results, max(1 << 16, first_per_query * Q)), max_results,
                                      "range_search")

    def _pairs_with_retry(self, call, res_cap: int, max_results: int, who: str) -> torch.Tensor:
        """Run a range-type ABI call (emr2a_range_search / emr2a_self_join) with ``res_cap`` results and four times as
        many candidates, plus at most one retry with buffers sized from the exact counts: int64 [n, 2] (query, key)."""
        cand_cap = 4 * res_cap
        for attempt in range(2):
            cand = torch.empty((cand_cap, 2), dtype=torch.int64, device=self.device)
            out = torch.empty((res_cap, 2), dtype=torch.int64, device=self.device)
            counts = torch.zeros((2,), dtype=torch.int64, device=self.device)
            with torch.cuda.device(self.device):
                native.check(call(cand, cand_cap, out, res_cap, counts))
            self.launches += 2
            n_cand, n_res = (int(x) for x in counts.cpu().tolist())      # the call's one host synchronisation
            caps = range_retry_caps(n_cand, n_res, cand_cap, res_cap, max_results)
            if caps is None:
                return out[:n_res]
            if attempt == 1:
                raise RuntimeError(f"{who}: retry with exact buffer sizes still overflowed ({n_cand}, {n_res})")
            cand_cap, res_cap = caps
            del cand, out
        raise AssertionError("unreachable")

    def cross_fold_duplicates(self, segs: Sequence, folds, min_score: float, flags: int = native.NF_ROWNORM,
                              max_results: int = 1 << 26, distributed: bool = False) -> Dict[str, torch.Tensor]:
        """Near-duplicate audit of a CV cohort: every pair of cases in DIFFERENT folds whose exact fp32 similarity
        (rows as ``cv_search_and_vote`` prepares them) is >= ``min_score`` -- the cases that put one patient's data on
        both sides of a split and inflate every CV number.  ``near_duplicates`` with ``folds``: returns each unordered
        pair once: ``i`` < ``j`` (caller row numbers, int64), ``score`` float32, ``fold_i``, ``fold_j``; sorted by i,
        then j."""
        return self.near_duplicates(segs, min_score, folds, flags, max_results, distributed)

    def near_duplicates(self, segs: Sequence, min_score: float, folds=None, flags: int = native.NF_ROWNORM,
                        max_results: int = 1 << 26, distributed: bool = False) -> Dict[str, torch.Tensor]:
        """Every pair of rows i < j of one cohort whose exact fp32 similarity is >= ``min_score``, each pair once and no
        row with itself -- whole-cohort deduplication.  Rows are prepared as ``cv_search_and_vote`` prepares them (one K1
        pass in the rescore layout with fp32 rows); ``emr2a_self_join`` computes only the upper triangle on the tensor
        cores and re-scores every candidate exactly, so the scores equal the ones ``range_search`` reports.  With
        ``folds`` only pairs of different folds count, and the rows are brought into fold order so that whole tiles of
        one fold are skipped.
        Returns ``i`` < ``j`` (caller row numbers, int64), ``score`` float32 and, with folds, ``fold_i`` / ``fold_j``
        (int64); sorted by i, then j.  More than ``max_results`` pairs (or more than 4 x ``max_results`` filter
        candidates on a GPU) raise ValueError.
        ``distributed=True``: under ``torchrun`` with an NCCL process group, every rank called with the same arrays
        (verified with checksums): each rank prepares the whole cohort, joins its band of query rows
        (``dist.self_join_ranges``, equal tensor-core work per rank) and the pair lists are all-gathered; every rank
        returns the same result, bit for bit equal to ``distributed=False``."""
        if not np.isfinite(min_score):
            raise ValueError(f"near_duplicates: min_score must be finite, got {min_score}")
        mats = [self._embedding(x)[0] for x in segs if x is not None]
        n = int(mats[0].shape[0])
        folds_t, perm = None, None
        if folds is not None:
            folds_t = self.to_device(folds, torch.uint8)
            if int(folds_t.shape[0]) != n:
                raise ValueError(f"near_duplicates: {int(folds_t.shape[0])} fold ids for {n} rows")
            perm = _fold_order(folds_t)
            if perm is not None:
                mats = [m.index_select(0, perm) for m in mats]
                folds_t = folds_t.index_select(0, perm)
        q0, q1, world = 0, n, 1
        if distributed:
            import torch.distributed as tdist
            from .dist import self_join_ranges
            world, rank = tdist.get_world_size(), tdist.get_rank()
            # cheap guard against ranks that were handed different cohorts
            sample = torch.arange(0, n, max(1, n // 61), device=self.device)[:64]
            sig = torch.stack([torch.tensor(float(n), device=self.device, dtype=torch.float64),
                               torch.tensor(float(sum(int(m.shape[1]) for m in mats)), device=self.device,
                                            dtype=torch.float64),
                               folds_t.double().sum() if folds_t is not None else torch.zeros((), device=self.device,
                                                                                              dtype=torch.float64)]
                              + [m.index_select(0, sample).double().sum() for m in mats])
            lo_sig, hi_sig = sig.clone(), sig.clone()
            tdist.all_reduce(lo_sig, op=tdist.ReduceOp.MIN)
            tdist.all_reduce(hi_sig, op=tdist.ReduceOp.MAX)
            if not torch.equal(lo_sig, hi_sig):
                raise ValueError("near_duplicates(distributed=True): the ranks were called with different cohorts "
                                 "(row count / dim / fold / row-sample checksums differ); every rank must pass the same "
                                 "arrays")
            counts = None if folds_t is None else torch.bincount(folds_t.long()).cpu().tolist()
            q0, q1 = self_join_ranges(n, counts, world)[rank]
        op = self.prepare(mats[0], mats[1] if len(mats) > 1 else None, 1.0, 1.0, flags, "rescore")
        if world == 1:
            pairs = self.self_join_prepared(op, min_score, folds_t, q0, q1, max_results)
        else:
            from .dist import _gather_varlen
            err, pairs = None, torch.zeros((0, 2), dtype=torch.int64, device=self.device)
            try:
                pairs = self.self_join_prepared(op, min_score, folds_t, q0, q1, max_results)
            except ValueError as e:             # every rank must take the same branch: the collectives below must match
                err = e
            failed = torch.tensor([0 if err is None else 1], dtype=torch.int64, device=self.device)
            tdist.all_reduce(failed, op=tdist.ReduceOp.MAX)
            if int(failed.item()):
                raise err if err is not None else ValueError("near_duplicates: another rank's band exceeded max_results")
            pairs = torch.cat(_gather_varlen(pairs, world))
            if int(pairs.shape[0]) > max_results:
                raise ValueError(f"near_duplicates: {int(pairs.shape[0])} pairs exceed max_results = {max_results}")
        return self_join_result(pairs, perm, folds_t, n)

    def self_join_prepared(self, op: Operand, min_score: float, folds=None, q_begin: int = 0, q_end: Optional[int] = None,
                           max_results: int = 1 << 26) -> torch.Tensor:
        """``emr2a_self_join`` on an operand prepared for the rescore arm with fp32 rows: the pairs i < j with
        q_begin <= i < q_end, fold[i] != fold[j] (``folds``, in the operand's row order), exact score >= min_score.
        Returns int64 [m, 2] (i, packed key of the exact score and j), in no particular order.  The first buffers hold
        one result per query row (the triangle finds each pair once) and the retry sizes them from the exact counts."""
        if op.f32 is None or op.hi is None or op.stats is None:
            raise ValueError("self_join needs an operand prepared for the rescore arm with fp32 rows (bf16 plane, stats)")
        n, D = op.n, op.dim
        q_end = n if q_end is None else int(q_end)
        q_begin = int(q_begin)
        if not 0 <= q_begin <= q_end <= n:
            raise ValueError(f"self_join: need 0 <= q_begin <= q_end <= n, got {q_begin}, {q_end}, {n}")
        if q_begin == q_end:
            return torch.zeros((0, 2), dtype=torch.int64, device=self.device)
        fold_sorted = False
        if folds is not None:
            folds = self.to_device(folds, torch.uint8)
            fold_sorted = _non_decreasing(folds)
        ws_bytes = int(self.lib.emr2a_self_join_workspace_bytes(n, D))
        ws = torch.empty((ws_bytes + 256,), dtype=torch.uint8, device=self.device)

        def call(cand, cand_cap, out, res_cap, counts):
            return self.lib.emr2a_self_join(
                op.f32.data_ptr(), _ld(op.f32), op.hi.data_ptr(), _ld(op.hi), n, D, q_begin, q_end, native.ptr(folds),
                int(fold_sorted), float(min_score), op.stats.data_ptr(), cand.data_ptr(), cand_cap, out.data_ptr(),
                res_cap, counts.data_ptr(), _round_up(ws.data_ptr(), 256), ws_bytes, self._stream())
        return self._pairs_with_retry(call, min(max_results, max(1 << 16, q_end - q_begin)), max_results, "self_join")

    # ----------------------------------------------- host-buffer (end-to-end) path
    def search_and_vote_host(self, db_segs_host: Sequence, q_segs_host: Sequence, db_labels, q_labels,
                             n_classes: int, k: int, db_flags: int = native.NF_ROWNORM,
                             q_flags: int = native.NF_ROWNORM, q_weights=(1.0, 1.0),
                             k_list: Sequence[int] = (1, 3, 5), precision: str = "auto",
                             chunk_rows: Optional[int] = None, row_offset: int = 0,
                             reduce_fn=None, gather_queries: bool = False) -> Dict[str, object]:
        """Same pipeline as ``search_and_vote`` for HOST-resident inputs (pinned CPU tensors or
        numpy): the database streams to the device in row chunks on a copy stream while the
        previous chunk is normalised and searched on the compute stream; per-chunk Top-K lists
        are merged by K3, K4 votes, and the results are copied back to the host.
        ``reduce_fn(keys) -> keys`` lets the multi-GPU caller all-gather + merge before the vote.
        ``gather_queries`` (multi-GPU, every rank holds the same host queries): a rank copies only its 1/world slice of
        the query rows over its host link and the slices are all-gathered over NVLink -- the replicated query copy is
        the one part of the step that does not shrink with the shard (41 MB per rank for C2: 1.8 ms on a 23 GB/s link).
        ``EMR2A_HOST_TAPER=1`` streams the tail of the database in shrinking chunks (``plan_chunks``).  It is off by
        default: the search of a chunk has a cost per QUERY (re-scoring, merge) that does not shrink with the chunk, so
        small tail chunks make the un-overlapped end of the step longer, not shorter (measured: e2e -2 %)."""
        def as_host(x):
            return torch.from_numpy(x) if isinstance(x, np.ndarray) else x
        db_host = [as_host(s) for s in db_segs_host if s is not None]
        q_host = [as_host(s) for s in q_segs_host if s is not None]
        n_db, n_q = int(db_host[0].shape[0]), int(q_host[0].shape[0])
        dim = sum(int(s.shape[1]) for s in db_host)
        prec = self.pick_precision(n_q, n_db, dim, k, precision)
        compute = torch.cuda.current_stream(self.device)
        copy = torch.cuda.Stream(self.device)
        h2d = 0
        if gather_queries:
            from .dist import gather_host_rows
            q_dev, q_bytes = gather_host_rows(q_host, self.device)
            h2d += q_bytes
        else:
            q_dev = [s.to(self.device, non_blocking=True) for s in q_host]
            h2d += sum(s.numel() * s.element_size() for s in q_host)
        qs = self.prepare(q_dev[0], q_dev[1] if len(q_dev) > 1 else None, q_weights[0], q_weights[1], q_flags, prec)
        if chunk_rows is None:       # ~128 MB of host rows per chunk: short pipeline fill/drain, PCIe stays saturated (measured)
            row_bytes = sum(int(s.shape[1]) * s.element_size() for s in db_host)
            chunk_rows = max(4096, (128 << 20) // max(row_bytes, 1))
        chunk_rows = max(256, min(chunk_rows, max(n_db, 1)))
        slots = [[torch.empty((chunk_rows, int(s.shape[1])), dtype=s.dtype, device=self.device) for s in db_host]
                 for _ in range(2)]
        for slot in slots:
            for b in slot:
                b.record_stream(copy)
        copied = [torch.cuda.Event(), torch.cuda.Event()]
        freed = [torch.cuda.Event(), torch.cuda.Event()]
        parts: List[torch.Tensor] = []
        n_chunks = 0
        taper = os.environ.get("EMR2A_HOST_TAPER", "0") == "1"
        for c, (lo, hi) in enumerate(plan_chunks(n_db, chunk_rows, min_rows=4096 if taper else chunk_rows)):
            sl = c % 2
            with torch.cuda.stream(copy):
                if c >= 2:
                    copy.wait_event(freed[sl])
                else:
                    copy.wait_stream(compute)
                for b, src in zip(slots[sl], db_host):
                    b[:hi - lo].copy_(src[lo:hi], non_blocking=True)
                copied[sl].record(copy)
            h2d += sum((hi - lo) * int(s.shape[1]) * s.element_size() for s in db_host)
            compute.wait_event(copied[sl])
            segs = [b[:hi - lo] for b in slots[sl]]
            db = self.prepare(segs[0], segs[1] if len(segs) > 1 else None, 1.0, 1.0, db_flags, prec,
                              defer_f32=self.defer_default(dim))
            parts.append(self.topk_search(qs, db, k, prec, idx_base=row_offset + lo))
            freed[sl].record(compute)
            n_chunks += 1
        keys = parts[0] if n_chunks == 1 else self.topk_merge(torch.stack(parts), k)
        if prec == "rescore":
            _, overflow = self.consume_status()
            if overflow:
                return self.search_and_vote_host(db_segs_host, q_segs_host, db_labels, q_labels, n_classes, k, db_flags,
                                                 q_flags, q_weights, k_list, "bf16x3", chunk_rows, row_offset, reduce_fn)
        if reduce_fn is not None:
            keys = reduce_fn(keys)
        db_labels = as_host(db_labels)
        q_labels = as_host(q_labels)
        h2d += db_labels.numel() * 4 + q_labels.numel() * 4
        res = self.vote_metrics(keys, db_labels, q_labels, n_classes, k_list=k_list)
        out: Dict[str, object] = {"precision": prec, "h2d_bytes": h2d}
        d2h = 0
        for name in ("top_idx", "top_scores", "top_labels", "pred_top1", "pred_vote", "pred_weighted",
                     "hit_counts", "vote_counts", "confusion", "group_sizes"):
            t = res[name].to("cpu", non_blocking=False)
            d2h += t.numel() * t.element_size()
            out[name] = t
        out["d2h_bytes"] = d2h
        return out


def _fold_order(folds: torch.Tensor) -> Optional[torch.Tensor]:
    """Stable permutation that sorts the rows by fold (None if they already are): the order in which the CV search
    skips whole tiles of a query's own fold."""
    if _non_decreasing(folds):
        return None
    return torch.argsort(folds.to(torch.int16), stable=True)


def _non_decreasing(v: torch.Tensor) -> bool:
    return bool((v[1:] >= v[:-1]).all().item()) if int(v.shape[0]) > 1 else True


def decode_keys(keys: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Packed keys (int64 storage, non-empty) -> (scores float32, global row indices int64), on the keys' device."""
    o = (keys >> 32) & 0xFFFFFFFF
    bits = torch.where(o >= 0x80000000, o - 0x80000000, 0xFFFFFFFF - o)
    bits = torch.where(bits >= 0x80000000, bits - (1 << 32), bits)           # as a signed 32-bit pattern
    return bits.to(torch.int32).view(torch.float32), 0xFFFFFFFF - (keys & 0xFFFFFFFF)


def csr_from_pairs(pairs: torch.Tensor, n_queries: int) -> Dict[str, torch.Tensor]:
    """(query, packed key) pairs int64 [n, 2], any order -> CSR by query; within a query by key descending, i.e.
    score descending, then index ascending (the tie rule of the packed keys)."""
    q, key = pairs[:, 0], pairs[:, 1]
    signed = key ^ (-(1 << 63))                       # unsigned key order as signed int64 order
    o1 = torch.argsort(signed, descending=True, stable=True)
    o = o1[torch.argsort(q[o1], stable=True)]
    q, key = q[o], key[o]
    scores, idx = decode_keys(key)
    counts = torch.bincount(q, minlength=n_queries) if q.numel() else torch.zeros(n_queries, dtype=torch.int64,
                                                                                   device=pairs.device)
    offsets = torch.zeros(n_queries + 1, dtype=torch.int64, device=pairs.device)
    offsets[1:] = torch.cumsum(counts, 0)
    return {"offsets": offsets, "idx": idx, "scores": scores}


def range_retry_caps(n_cand: int, n_res: int, cand_cap: int, res_cap: int, max_results: int
                     ) -> Optional[Tuple[int, int]]:
    """Buffer sizes for the one retry of a range search (None: the outputs are complete).  The counts of
    emr2a_range_search are exact; when the candidates overflowed nothing was re-scored and the results, a subset of
    the candidates, are bounded by their count.  Raises ValueError instead of sizing past ``max_results`` results or
    4 x ``max_results`` candidates."""
    if n_cand > 4 * max_results:
        raise ValueError(f"range_search: {n_cand} filter candidates exceed 4 x max_results = {4 * max_results}; "
                         "raise min_score or max_results")
    if n_cand > cand_cap:
        return n_cand, max(1, min(n_cand, max_results))
    if n_res > max_results:
        raise ValueError(f"range_search: {n_res} results exceed max_results = {max_results}")
    if n_res > res_cap:
        return cand_cap, n_res
    return None


def cross_fold_pairs(pairs: torch.Tensor, perm: Optional[torch.Tensor], folds: torch.Tensor) -> Dict[str, torch.Tensor]:
    """Self-join results (query, packed key) in fold order -> each unordered pair once, in caller row numbers:
    i < j, score, fold_i, fold_j, sorted by (i, j).  ``perm[r]`` = caller row of fold-ordered row r (None: identity)."""
    scores, b = decode_keys(pairs[:, 1])
    a = pairs[:, 0]
    fa, fb = folds[a].to(torch.int64), folds[b].to(torch.int64)
    if perm is not None:
        a, b = perm[a], perm[b]
    keep = a < b
    i, j, s, fi, fj = a[keep], b[keep], scores[keep], fa[keep], fb[keep]
    o = torch.argsort(i * (int(folds.shape[0]) + 1) + j)
    return {"i": i[o], "j": j[o], "score": s[o], "fold_i": fi[o], "fold_j": fj[o]}


def self_join_result(pairs: torch.Tensor, perm: Optional[torch.Tensor], folds: Optional[torch.Tensor], n: int
                     ) -> Dict[str, torch.Tensor]:
    """Self-join results (i, packed key of j) with i < j in the joined row order -> caller row numbers.  ``perm[r]`` =
    caller row of joined row r (None: identity); a < b does not imply perm[a] < perm[b], so every pair is normalised to
    (min, max).  Returns i < j, score, and fold_i / fold_j (of caller rows i and j) when ``folds`` (joined order) is
    given; sorted by (i, j)."""
    scores, b = decode_keys(pairs[:, 1])
    a = pairs[:, 0]
    res: Dict[str, torch.Tensor] = {}
    if folds is not None:
        fa, fb = folds[a].to(torch.int64), folds[b].to(torch.int64)
    if perm is not None:
        a, b = perm[a], perm[b]
    swap = a > b
    i, j = torch.where(swap, b, a), torch.where(swap, a, b)
    o = torch.argsort(i * (int(n) + 1) + j)
    res["i"], res["j"], res["score"] = i[o], j[o], scores[o]
    if folds is not None:
        res["fold_i"], res["fold_j"] = torch.where(swap, fb, fa)[o], torch.where(swap, fa, fb)[o]
    return res


def plan_chunks(n_rows: int, chunk_rows: int, min_rows: int = 4096) -> List[Tuple[int, int]]:
    """Row ranges of a streamed database: full chunks, then a tail that halves down to ``min_rows`` -- the search of
    the last chunk is the one piece of compute that cannot hide behind a copy, so it should be short."""
    out, lo = [], 0
    chunk_rows = max(int(chunk_rows), 1)
    min_rows = max(1, min(min_rows, chunk_rows // 2))          # every piece fits a chunk-sized staging slot
    while n_rows - lo > chunk_rows + chunk_rows // 2:
        out.append((lo, lo + chunk_rows))
        lo += chunk_rows
    rest = n_rows - lo
    while rest > 2 * min_rows:
        step = min(chunk_rows, (rest // 2 + 255) // 256 * 256)
        out.append((lo, lo + step))
        lo += step
        rest -= step
    if rest > 0:
        out.append((lo, n_rows))
    return out


class DatabaseIndex:
    """A database resident in HBM in the layout the search kernels consume (see ``Engine.build_index``)."""

    def __init__(self, engine: Engine, operand: Operand, labels: torch.Tensor, n_classes: int, flags: int, precision: str):
        self.engine, self.operand, self.labels = engine, operand, labels
        self.n_classes, self.flags, self.precision = n_classes, flags, precision

    @property
    def rows(self) -> int:
        return self.operand.n

    def _enqueue(self, q_segs: Sequence, q_labels, k: int, q_weights, q_flags: Optional[int], k_list: Sequence[int],
                 want_lists: bool) -> Dict[str, torch.Tensor]:
        """K1 (queries) -> K2 -> K4, stream-ordered, no host synchronisation; the rescore status stays on the device."""
        eng = self.engine
        prec = self.precision
        if prec == "rescore" and k > _RESCORE_MAX_K:
            raise ValueError(f"this index was built for the rescore arm (K <= {_RESCORE_MAX_K}); rebuild it with precision='bf16x3'")
        # Small batches: a query tile whose rows are partly out of bounds of the query matrix makes the TMA loads of
        # that tile markedly slower for some row counts (measured on B200, 1M x 1024 plane: Q = 1: 0.55-0.73 ms,
        # Q = 48: 0.56 ms, against 0.37-0.41 ms for 64 in-bounds rows).  Up to 256 queries the batch is therefore
        # filled to a multiple of 64 rows with copies of its last query; the copies' results are dropped before the vote.
        segs = [eng._embedding(x)[0] for x in q_segs if x is not None]
        n_q = int(segs[0].shape[0])
        pad = (-n_q) % 64 if (0 < n_q <= _QPAD_MAX and prec != "fp32") else 0
        if pad:
            segs = [torch.cat([t, t[-1:].expand(pad, int(t.shape[1]))]) for t in segs]
        qs = eng.prepare(segs[0], segs[1] if len(segs) > 1 else None, q_weights[0], q_weights[1],
                         self.flags if q_flags is None else q_flags, prec)
        keys = eng.topk_search(qs, self.operand, k, prec)
        if pad:
            keys = keys[:n_q]
            if eng.last_unverified is not None and prec == "rescore":
                eng.last_unverified = eng.last_unverified[:n_q]
        if q_labels is None:
            q_labels = torch.full((n_q,), -1, dtype=torch.int32, device=eng.device)
        res = eng.vote_metrics(keys, self.labels, q_labels, self.n_classes, k_list=k_list, want_lists=want_lists)
        res["keys"] = keys
        if prec == "rescore":
            res["status"] = eng.pop_status_tensor()
        return res

    @staticmethod
    def _check_status(res: Dict[str, torch.Tensor]) -> None:
        st = res.pop("status", None)
        if st is None:
            return
        st = st.cpu()
        if int(st[1]):
            raise Emr2aOverflow("rescore verification overflowed for this query batch; rebuild the index with "
                                "precision='bf16x3' for databases with very dense score neighbourhoods")
        res["unverified"] = int(st[0])

    def search(self, q_segs: Sequence, q_labels=None, k: int = 10, q_weights=(1.0, 1.0), q_flags: Optional[int] = None,
               k_list: Sequence[int] = (1, 3, 5), want_lists: bool = True) -> Dict[str, torch.Tensor]:
        """K1 on the queries (host or device arrays) -> K2 against the resident rows -> K4 vote.  Without
        ``q_labels`` the hit/vote counters are meaningless and only lists and predictions should be read."""
        res = self._enqueue(q_segs, q_labels, k, q_weights, q_flags, k_list, want_lists)
        self._check_status(res)
        return res

    def range_search(self, q_segs: Sequence, min_score: float, q_weights=(1.0, 1.0), q_flags: Optional[int] = None,
                     max_results: int = 1 << 26) -> Dict[str, torch.Tensor]:
        """``Engine.range_search`` against the resident rows: every row with exact score >= ``min_score``, as a CSR
        dict.  Needs an index built with ``precision='rescore'`` (the filter reads its bf16 plane and stats)."""
        op = self.operand
        if self.precision != "rescore" or op.hi is None or op.stats is None or (op.f32 is None and op.lazy is None):
            raise ValueError(f"range_search needs an index built with precision='rescore' (this one: {self.precision!r}); "
                             "rebuild it with build_index(..., precision='rescore')")
        eng = self.engine
        qs = eng.prepare(q_segs[0], q_segs[1] if len(q_segs) > 1 else None, q_weights[0], q_weights[1],
                         self.flags if q_flags is None else q_flags, "rescore")
        return eng.range_search_prepared(qs, op, min_score, max_results=max_results)

    def capture(self, n_queries: int, k: int = 10, q_weights=(1.0, 1.0), q_flags: Optional[int] = None,
                k_list: Sequence[int] = (1, 3, 5), want_lists: bool = True, seg_dims: Optional[Sequence[int]] = None
                ) -> "GraphedSearch":
        """Small-batch serving: the whole K1 -> K2 -> K4 sequence for batches of exactly ``n_queries`` queries captured
        in ONE CUDA graph (the ~10 launches of a batch are launch-bound below a few hundred queries)."""
        return GraphedSearch(self, n_queries, k, q_weights, q_flags, k_list, want_lists, seg_dims)


class GraphedSearch:
    """``DatabaseIndex.search`` for a fixed batch size as a CUDA graph.  Calling it copies the queries into the
    graph's static input buffers, replays the graph and returns the graph's static output tensors (overwritten by
    the next call)."""

    def __init__(self, index: DatabaseIndex, n_queries: int, k: int, q_weights, q_flags, k_list, want_lists, seg_dims):
        eng = index.engine
        if seg_dims is None:
            seg_dims = [index.operand.dim]
        if sum(int(d) for d in seg_dims) != index.operand.dim or not 1 <= len(seg_dims) <= 2:
            raise ValueError(f"capture: seg_dims {list(seg_dims)} do not add up to the index dimension {index.operand.dim}")
        self.index, self.n_queries = index, int(n_queries)
        self.q_in = [torch.zeros((self.n_queries, int(d)), dtype=torch.float32, device=eng.device) for d in seg_dims]
        self.labels_in = torch.full((self.n_queries,), -1, dtype=torch.int32, device=eng.device)
        args = (self.q_in, self.labels_in, k, q_weights, q_flags, list(k_list), want_lists)
        side = torch.cuda.Stream(eng.device)                 # warm-up off the capture stream (lazy module loads etc.)
        side.wait_stream(torch.cuda.current_stream(eng.device))
        with torch.cuda.stream(side):
            for t in self.q_in:
                t.normal_()                                  # all-zero queries would tie every score
            index._enqueue(*args)
        torch.cuda.current_stream(eng.device).wait_stream(side)
        eng._status_log.clear()
        l0 = eng.launches
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = index._enqueue(*args)
        self.launches_per_replay = eng.launches - l0
        eng.launches = l0

    def __call__(self, q_segs: Sequence, q_labels=None) -> Dict[str, torch.Tensor]:
        eng = self.index.engine
        if len(q_segs) != len(self.q_in):
            raise ValueError("graphed search: number of query segments differs from the captured one")
        for dst, src in zip(self.q_in, q_segs):
            src_t = torch.from_numpy(np.ascontiguousarray(src, dtype=np.float32)) if isinstance(src, np.ndarray) else src
            if tuple(src_t.shape) != tuple(dst.shape):
                raise ValueError(f"graphed search: query block {tuple(src_t.shape)} != captured {tuple(dst.shape)}")
            dst.copy_(src_t, non_blocking=True)
        if q_labels is not None:
            self.labels_in.copy_(eng.to_device(q_labels, torch.int32), non_blocking=True)
        self.graph.replay()
        eng.launches += self.launches_per_replay
        res = dict(self.out)
        self.index._check_status(res)
        return res


class Emr2aOverflow(RuntimeError):
    pass


_engines: Dict[int, Engine] = {}


def get_engine(device: Optional[torch.device] = None) -> Engine:
    if not torch.cuda.is_available():
        raise RuntimeError("emr2a_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    idx = torch.cuda.current_device() if device is None else torch.device(device).index or 0
    if idx not in _engines:
        _engines[idx] = Engine(torch.device("cuda", idx))
    return _engines[idx]


def unpack_keys(keys: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Host-side decode of packed keys (tests / debugging): returns (scores f32, indices int64, -1 = empty)."""
    k = keys.cpu().numpy().view(np.uint64)
    o = (k >> np.uint64(32)).astype(np.uint32)
    neg = (o & np.uint32(0x80000000)) == 0
    bits = np.where(neg, ~o, o ^ np.uint32(0x80000000)).astype(np.uint32)
    scores = bits.view(np.float32)
    idx = (np.uint64(0xFFFFFFFF) - (k & np.uint64(0xFFFFFFFF))).astype(np.int64)
    idx[k == 0] = -1
    scores = np.where(k == 0, np.float32(0), scores)
    return scores, idx
