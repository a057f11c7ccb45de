"""Registration after matching through the C-ABI (nm_align_points_f32, nm_ransac_*): the
reference's align_points / ransac_translation / ransac_similarity / ransac_homography
(src/gpu/kernels/ransac.h:8-22)."""
from __future__ import annotations

import ctypes as C

from . import _lib
from ._lib import check
from .sift import _stream_ptr

TRANSLATION, SIMILARITY, HOMOGRAPHY = 0, 1, 2
MOSAIC, TRANSFER = 0, 1          # residual of adjust_chain: NM_ADJUST_MOSAIC, NM_ADJUST_TRANSFER


def _p(t):
    return C.c_void_p(t.data_ptr())


def _f32(*ts):
    """The C-ABI reads raw memory: every coordinate array must be a contiguous cuda float32 tensor of one shape."""
    import torch
    shape = ts[0].shape
    for t in ts:
        if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.shape == shape):
            raise TypeError("expected contiguous cuda float32 tensors of equal shape")


def _int32(t, name):
    import torch
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.int32 and t.is_contiguous()):
        raise TypeError(f"{name}: expected a contiguous cuda int32 tensor (torch.nonzero / argmax give int64)")


def align_points(src_x, src_y, dst_x, dst_y, matches):
    """Correspondences (c_src_x, c_src_y, c_dst_x, c_dst_y): src[i] with dst[matches[i]], -1 where unmatched."""
    import torch
    _f32(src_x, src_y); _f32(dst_x, dst_y); _int32(matches, "matches")
    n = matches.shape[0]
    assert src_x.shape[0] == n
    out = [torch.empty(n, dtype=torch.float32, device=src_x.device) for _ in range(4)]
    check(_lib.load().nm_align_points_f32(_p(src_x), _p(src_y), _p(dst_x), _p(dst_y), *[_p(o) for o in out],
                                          _p(matches), n, _stream_ptr()), "nm_align_points_f32")
    return tuple(out)


def align_pairs_span(x, y, matches, counts, span):
    """nm_align_pairs_span_f32: the correspondences of every link of the span layout.  x, y: (n_frames, capacity) cuda
    float32 keypoint coordinates, matches: (L, capacity) int32 as match_pairs_span returns them, counts: (n_frames,) int32.
    Returns (c_src_x, c_src_y, c_dst_x, c_dst_y), each (L, capacity)."""
    import torch
    _f32(x, y); _int32(matches, "matches"); _int32(counts, "counts")
    n_frames, cap = x.shape
    L = matches.shape[0]
    assert tuple(matches.shape) == (span * n_frames - span * (span + 1) // 2, cap) and counts.numel() == n_frames
    out = [torch.empty((L, cap), dtype=torch.float32, device=x.device) for _ in range(4)]
    check(_lib.load().nm_align_pairs_span_f32(_p(x), _p(y), _p(matches), _p(counts), n_frames, cap, span, *[_p(o) for o in out],
                                              _stream_ptr()), "nm_align_pairs_span_f32")
    return tuple(out)


def ransac_hypotheses(kind, src_x, src_y, dst_x, dst_y, rand_list, inlier_threshold):
    """All hypotheses of a caller-supplied index list: (iterations, 9) homographies and inlier counts."""
    import torch
    _f32(src_x, src_y, dst_x, dst_y); _int32(rand_list, "rand_list")
    m = (1, 2, 4)[kind]
    iterations = rand_list.numel() // m
    H = torch.empty((iterations, 9), dtype=torch.float32, device=src_x.device)
    inl = torch.empty(iterations, dtype=torch.int32, device=src_x.device)
    check(_lib.load().nm_ransac_hypotheses_f32(kind, _p(src_x), _p(src_y), _p(dst_x), _p(dst_y), src_x.shape[0],
                                               _p(rand_list), iterations, inlier_threshold, _p(H), _p(inl),
                                               _stream_ptr()), "nm_ransac_hypotheses_f32")
    return H, inl


def ransac(kind, src_x, src_y, dst_x, dst_y, inlier_threshold, iterations, seed=0, homography=None):
    """Best model of `iterations` random hypotheses; no host synchronisation.  Returns (homography (9,) cuda,
    status (3,) cuda int32 = [ok, inliers, iteration])."""
    import torch
    _f32(src_x, src_y, dst_x, dst_y)
    if homography is None:
        homography = torch.zeros(9, dtype=torch.float32, device=src_x.device)
    status = torch.zeros(3, dtype=torch.int32, device=src_x.device)
    check(_lib.load().nm_ransac_f32(kind, _p(src_x), _p(src_y), _p(dst_x), _p(dst_y), src_x.shape[0], inlier_threshold,
                                    iterations, seed & 0xFFFFFFFFFFFFFFFF, _p(homography), _p(status), _stream_ptr()),
          "nm_ransac_f32")
    return homography, status


def ransac_batch(kind, src_x, src_y, dst_x, dst_y, counts, inlier_threshold, iterations, seed=0):
    """nm_ransac_batch_f32: src_x ... dst_y are (n_pairs, max_pts) cuda float32 (contiguous), counts (n_pairs,) cuda
    int32 or None.  Returns homographies (n_pairs, 9) and status (n_pairs, 3); pair p uses seed + p."""
    import torch
    _f32(src_x, src_y, dst_x, dst_y)
    if counts is not None:
        _int32(counts, "counts")
    n_pairs, max_pts = src_x.shape
    H = torch.zeros((n_pairs, 9), dtype=torch.float32, device=src_x.device)
    status = torch.zeros((n_pairs, 3), dtype=torch.int32, device=src_x.device)
    check(_lib.load().nm_ransac_batch_f32(kind, _p(src_x), _p(src_y), _p(dst_x), _p(dst_y), max_pts,
                                          _p(counts) if counts is not None else None, max_pts, n_pairs, inlier_threshold,
                                          iterations, seed & 0xFFFFFFFFFFFFFFFF, _p(H), _p(status), _stream_ptr()),
          "nm_ransac_batch_f32")
    return H, status


def refine_batch(kind, src_x, src_y, dst_x, dst_y, counts, H, status, inlier_threshold, rounds=2, out=None):
    """nm_ransac_refine_batch_f32: least-squares refits of the models H (n_pairs, 9) on their inlier sets, and the inlier
    masks.  Correspondences and counts as for ransac_batch; status (n_pairs, 3) cuda int32 as ransac_batch returns it, or
    None.  out = (H_out, status_out) writes there (they may be H and status: in place).  Returns (H (n_pairs, 9),
    status (n_pairs, 3) = [ok, inliers, refits kept], mask (n_pairs, max_pts) bool)."""
    import torch
    _f32(src_x, src_y, dst_x, dst_y)
    if counts is not None:
        _int32(counts, "counts")
    n_pairs, max_pts = src_x.shape
    if not (isinstance(H, torch.Tensor) and H.is_cuda and H.dtype == torch.float32 and H.is_contiguous()
            and tuple(H.shape) == (n_pairs, 9)):
        raise TypeError("H: expected a contiguous cuda float32 tensor of shape (n_pairs, 9)")
    if status is not None:
        _int32(status, "status")
        assert tuple(status.shape) == (n_pairs, 3)
    if out is None:
        H_out = torch.empty_like(H)
        st_out = torch.zeros((n_pairs, 3), dtype=torch.int32, device=src_x.device)
    else:
        H_out, st_out = out
        _f32(H_out, H); _int32(st_out, "status_out")
        assert tuple(st_out.shape) == (n_pairs, 3)
    mask = torch.empty((n_pairs, max_pts), dtype=torch.bool, device=src_x.device)
    check(_lib.load().nm_ransac_refine_batch_f32(kind, _p(src_x), _p(src_y), _p(dst_x), _p(dst_y), max_pts,
                                                 _p(counts) if counts is not None else None, max_pts, n_pairs,
                                                 inlier_threshold, _p(H), _p(status) if status is not None else None,
                                                 rounds, _p(H_out), _p(st_out), _p(mask), _stream_ptr()),
          "nm_ransac_refine_batch_f32")
    return H_out, st_out, mask


def refine(kind, src_x, src_y, dst_x, dst_y, H, status, inlier_threshold, rounds=2):
    """refine_batch for one pair: src_x ... dst_y (n,), H (9,), status (3,) or None.  Returns (H (9,), status (3,),
    mask (n,) bool)."""
    Hb, sb, mb = refine_batch(kind, src_x[None], src_y[None], dst_x[None], dst_y[None], None, H.reshape(1, 9),
                              None if status is None else status.reshape(1, 3), inlier_threshold, rounds)
    return Hb[0], sb[0], mb[0]


def adjust_chain(kind, src_x, src_y, dst_x, dst_y, counts, span, masks, H, link_status, frame_w, frame_h, inlier_threshold,
                 iterations=10, out=None, cost=MOSAIC, fixed=None):
    """nm_ransac_adjust_chain_fixed_f32 (arguments in the order of nm_ransac_adjust_chain_f32, then cost and fixed): joint
    least-squares adjustment of the poses of a window of n frames from the links of its span layout.  src_x ... dst_y
    (L, max_pts) and counts (L,) or None as for refine_batch; masks (L, max_pts) bool, H (L, 9) the link models and
    link_status (L, 3), as refine_batch returns them (rows 0 .. n-2 are the consecutive pairs).  inlier_threshold: the
    RANSAC rule that counts status[:, 1].  out = (H_out, status_out), (n - 1, 9) and (n - 1, 3): written there (they may
    be H[: n - 1] and link_status[: n - 1]).  Returns (H (n - 1, 9) pairwise models that nm_mosaic_place_f32 chains into
    the adjusted poses, status (n - 1, 3) = [frame p + 1 connected, inliers, LM steps accepted], chain (n, 9) float64
    frame -> frame-0 transforms, report (4,) float64 = [mean squared residual before, after (px^2), residual points,
    links used]).  cost: MOSAIC (the default, nm_ransac_adjust_chain_f32) measures a link's residual in frame-0 pixels,
    TRANSFER in the pixels of its target frame t + d, which does not reward shrinking the frames far from frame 0 (long
    windows of similarity or homography models).  With TRANSFER a point behind the target camera at the initial poses
    leaves the window unadjusted (report costs +inf).  fixed = (chain (n_fixed, 9) float64, conn (n_fixed,) int32 or None),
    cuda tensors, 1 <= n_fixed <= n - 1: frames 0 .. n_fixed-1 keep the poses chain[j] (any common frame: the rows are
    rebased on chain[0]) and only links reaching a later frame are used -- for example the last rows of the previous
    window's chain and its status[:, 0] as conn (entry 0 is ignored).  None: n_fixed = 1, the window on its own."""
    import torch
    _f32(src_x, src_y, dst_x, dst_y)
    if counts is not None:
        _int32(counts, "counts")
    L, max_pts = src_x.shape
    n = next((m for m in range(2, 1026) if span * m - span * (span + 1) // 2 == L), None) if span >= 1 else None
    if n is None:
        raise ValueError(f"{L} links do not form a span-{span} layout")
    if not (masks.is_cuda and masks.dtype == torch.bool and masks.is_contiguous() and tuple(masks.shape) == (L, max_pts)):
        raise TypeError("masks: expected a contiguous cuda bool tensor of shape (L, max_pts)")
    _int32(link_status, "link_status")
    if not (isinstance(H, torch.Tensor) and H.is_cuda and H.dtype == torch.float32 and H.is_contiguous()
            and tuple(H.shape) == (L, 9) and tuple(link_status.shape) == (L, 3)):
        raise TypeError("H, link_status: expected contiguous cuda tensors of shapes (L, 9) float32 and (L, 3) int32")
    if out is None:
        H_out = torch.empty((n - 1, 9), dtype=torch.float32, device=H.device)
        st_out = torch.empty((n - 1, 3), dtype=torch.int32, device=H.device)
    else:
        H_out, st_out = out
        _f32(H_out, H[: n - 1])
        _int32(st_out, "status_out")
        if tuple(st_out.shape) != (n - 1, 3):
            raise TypeError("status_out: expected shape (n - 1, 3)")
    n_fixed, fchain, fconn = 1, None, None
    if fixed is not None:
        fchain, fconn = fixed
        if not (isinstance(fchain, torch.Tensor) and fchain.is_cuda and fchain.dtype == torch.float64 and fchain.is_contiguous()
                and fchain.dim() == 2 and fchain.shape[1] == 9):
            raise TypeError("fixed chain: expected a contiguous cuda float64 tensor of shape (n_fixed, 9)")
        n_fixed = fchain.shape[0]
        if fconn is not None:
            _int32(fconn, "fixed conn")
            if tuple(fconn.shape) != (n_fixed,):
                raise TypeError("fixed conn: expected shape (n_fixed,)")
    chain = torch.empty((n, 9), dtype=torch.float64, device=H.device)
    report = torch.empty(4, dtype=torch.float64, device=H.device)
    check(_lib.load().nm_ransac_adjust_chain_fixed_f32(kind, cost, _p(src_x), _p(src_y), _p(dst_x), _p(dst_y), max_pts,
                                                       _p(counts) if counts is not None else None, max_pts, inlier_threshold, n,
                                                       span, frame_w, frame_h, _p(masks), _p(H), _p(link_status), n_fixed,
                                                       _p(fchain) if fchain is not None else None,
                                                       _p(fconn) if fconn is not None else None, iterations,
                                                       _p(H_out), _p(st_out), _p(chain), _p(report), _stream_ptr()),
          "nm_ransac_adjust_chain_fixed_f32")
    return H_out, st_out, chain, report
