"""Brute-force k=2 ratio-test matching through the C-ABI (nm_match_*)."""
from __future__ import annotations

import ctypes as C

from . import _lib
from ._lib import check
from .sift import _stream_ptr


def set_engine(engine: int) -> None:
    """0 = exact fp32 SIMT scan, 1 = tcgen05 candidate search + fp32 re-rank, -1 = auto."""
    check(_lib.load().nm_match_set_engine(engine), "nm_match_set_engine")


def get_engine() -> int:
    return _lib.load().nm_match_get_engine()


def _desc(t, name):
    """The C-ABI reads raw memory: contiguous cuda float32 (n, 128) or nothing."""
    import torch
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32 and t.dim() == 2 and t.shape[1] == 128):
        raise TypeError(f"{name}: expected a cuda float32 tensor of shape (n, 128), got {getattr(t, 'dtype', type(t))} "
                        f"{tuple(getattr(t, 'shape', ()))}")
    return t if t.is_contiguous() else t.contiguous()


def _i32(t, name, n):
    import torch
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.int32 and t.is_contiguous() and t.numel() == n):
        raise TypeError(f"{name}: expected a contiguous cuda int32 tensor of {n} elements")
    return t


def match(A, B, ambiguity: float = 0.8, match_io=None, want_distance: bool = False):
    """compute_sift_matches semantics (reference src/gpu/sift/siftfunctions.cu:15-40).
    A: (nA,128), B: (nB,128) cuda float32.  Returns match indices (int32, -1 = rejected),
    and the nA x nB squared-distance matrix when want_distance."""
    import torch
    A, B = _desc(A, "A"), _desc(B, "B")
    nA, nB = A.shape[0], B.shape[0]
    if match_io is None:
        match_io = torch.full((nA,), -1, dtype=torch.int32, device=A.device)
    _i32(match_io, "match_io", nA)
    dist = torch.empty((nA, nB), dtype=torch.float32, device=A.device) if want_distance else None
    check(_lib.load().nm_match_f32(C.c_void_p(A.data_ptr()), nA, C.c_void_p(B.data_ptr()), nB, ambiguity,
                                   C.c_void_p(match_io.data_ptr()),
                                   C.c_void_p(dist.data_ptr()) if dist is not None else None, _stream_ptr()), "nm_match_f32")
    return (match_io, dist) if want_distance else match_io


def match_top2(A, B, index_offset: int = 0):
    """Per-shard records (nA,4) float32: (d1, bits(i1+offset), d2, 0)."""
    import torch
    A = _desc(A, "A")
    B = _desc(B, "B") if B.shape[0] else B
    nA, nB = A.shape[0], B.shape[0]
    rec = torch.empty((nA, 4), dtype=torch.float32, device=A.device)
    check(_lib.load().nm_match_top2_f32(C.c_void_p(A.data_ptr()), nA, C.c_void_p(B.data_ptr()) if nB else None, nB,
                                        index_offset, C.c_void_p(rec.data_ptr()), _stream_ptr()), "nm_match_top2_f32")
    return rec


def merge_top2(recs, ambiguity: float = 0.8, match_io=None):
    """recs: (n_shards, nA, 4) records -> match indices."""
    import torch
    if not (recs.is_cuda and recs.dtype == torch.float32 and recs.dim() == 3 and recs.shape[2] == 4):
        raise TypeError("recs: expected a cuda float32 tensor of shape (n_shards, nA, 4)")
    recs = recs if recs.is_contiguous() else recs.contiguous()
    n_shards, nA = recs.shape[0], recs.shape[1]
    if match_io is None:
        match_io = torch.full((nA,), -1, dtype=torch.int32, device=recs.device)
    _i32(match_io, "match_io", nA)
    check(_lib.load().nm_match_merge_top2(C.c_void_p(recs.data_ptr()), n_shards, nA, ambiguity,
                                          C.c_void_p(match_io.data_ptr()), _stream_ptr()), "nm_match_merge_top2")
    return match_io


def match_pairs(desc, counts, ambiguity: float = 0.8, match_out=None, want_records: bool = False):
    """nm_match_pairs_f32: frame p matched to frame p + 1 for every p.  desc: (n_frames, capacity, 128) cuda float32
    (the layout of SiftBatch.results()["desc"]), counts: (n_frames,) cuda int32.  Returns match indices
    (n_frames - 1, capacity) int32 (-1 where unmatched / beyond the frame's count), optionally the exact records and
    the device counter of rows that needed the exact fallback scan.  No host synchronisation."""
    import torch
    assert desc.is_cuda and desc.dtype == torch.float32 and desc.is_contiguous() and desc.dim() == 3 and desc.shape[2] == 128
    n_frames, cap = desc.shape[0], desc.shape[1]
    _i32(counts, "counts", n_frames)
    if match_out is None:
        match_out = torch.full((n_frames - 1, cap), -1, dtype=torch.int32, device=desc.device)
    rec = torch.zeros((n_frames - 1, cap, 4), dtype=torch.float32, device=desc.device) if want_records else None
    fb = torch.zeros(1, dtype=torch.int32, device=desc.device) if want_records else None
    check(_lib.load().nm_match_pairs_f32(C.c_void_p(desc.data_ptr()), C.c_void_p(counts.data_ptr()), n_frames, cap, ambiguity,
                                         C.c_void_p(match_out.data_ptr()), C.c_void_p(rec.data_ptr()) if rec is not None else None,
                                         C.c_void_p(fb.data_ptr()) if fb is not None else None, _stream_ptr()), "nm_match_pairs_f32")
    return (match_out, rec, fb) if want_records else match_out


def span_links(n_frames: int, span: int) -> int:
    """Rows of the span layout over n_frames frames: the links (t, t + d), 1 <= d <= span, d-major (include/nm_b200.h)."""
    return span * n_frames - span * (span + 1) // 2


def link_row(n_frames: int, t: int, d: int) -> int:
    """Row of link (t, t + d) in the span layout."""
    return (d - 1) * n_frames - (d - 1) * d // 2 + t


def match_pairs_span(desc, counts, span, ambiguity: float = 0.8, match_out=None, want_records: bool = False):
    """nm_match_pairs_span_f32: match_pairs for every link (t, t + d), d <= span, of the span layout.  Returns match
    indices (span_links(n_frames, span), capacity) int32; row link_row(n, t, d) holds frame t's matches into frame t + d.
    Span 1 is match_pairs.  No host synchronisation."""
    import torch
    assert desc.is_cuda and desc.dtype == torch.float32 and desc.is_contiguous() and desc.dim() == 3 and desc.shape[2] == 128
    n_frames, cap = desc.shape[0], desc.shape[1]
    _i32(counts, "counts", n_frames)
    L = span_links(n_frames, span)
    if match_out is None:
        match_out = torch.full((max(L, 0), cap), -1, dtype=torch.int32, device=desc.device)
    rec = torch.zeros((L, cap, 4), dtype=torch.float32, device=desc.device) if want_records else None
    fb = torch.zeros(1, dtype=torch.int32, device=desc.device) if want_records else None
    check(_lib.load().nm_match_pairs_span_f32(C.c_void_p(desc.data_ptr()), C.c_void_p(counts.data_ptr()), n_frames, cap, span,
                                              ambiguity, C.c_void_p(match_out.data_ptr()),
                                              C.c_void_p(rec.data_ptr()) if rec is not None else None,
                                              C.c_void_p(fb.data_ptr()) if fb is not None else None, _stream_ptr()),
          "nm_match_pairs_span_f32")
    return (match_out, rec, fb) if want_records else match_out


def tc_probe(A, B, want_candidates: bool = False):
    """Diagnostics of the tensor-core engine (nm_match_tc_probe): exact records (nA,4), the number
    of rows whose exactness certificate failed (re-scanned by the exact engine), and optionally
    the candidate lists of the tcgen05 scan with the power-of-two scale that was applied."""
    import numpy as np
    import torch
    A, B = _desc(A, "A"), _desc(B, "B")
    nA, nB = A.shape[0], B.shape[0]
    rec = torch.empty((nA, 4), dtype=torch.float32, device=A.device)
    fb, nl, sc = C.c_int(-1), C.c_int(0), C.c_float(0)
    cs = np.zeros((8, nA, 4), np.float32) if want_candidates else None
    ci = np.zeros((8, nA, 4), np.int32) if want_candidates else None
    check(_lib.load().nm_match_tc_probe(C.c_void_p(A.data_ptr()), nA, C.c_void_p(B.data_ptr()), nB, C.c_void_p(rec.data_ptr()),
                                        C.byref(fb), cs.ctypes.data_as(C.c_void_p) if want_candidates else None,
                                        ci.ctypes.data_as(C.c_void_p) if want_candidates else None, C.byref(nl), C.byref(sc),
                                        _stream_ptr()), "nm_match_tc_probe")
    out = {"rec": rec, "fallback_rows": fb.value, "n_lists": nl.value, "scale": sc.value}
    if want_candidates:
        n = nl.value
        out["cand_scores"] = cs.reshape(-1)[: n * nA * 4].reshape(n, nA, 4)
        out["cand_index"] = ci.reshape(-1)[: n * nA * 4].reshape(n, nA, 4)
    return out
