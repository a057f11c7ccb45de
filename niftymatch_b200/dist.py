"""Multi-GPU partitioning of the hot path (one process per GPU, torch.distributed).

* SIFT detect+describe shards by FRAMES: each rank takes a contiguous range of the batch /
  stream (frame_range); there is no data-path collective (weak scaling).
* Brute-force matching against a large database shards the DATABASE rows: queries are
  replicated, every rank scans its shard and emits one 16-byte record per query
  (d1, i1_global, d2); the records are all-gathered (NCCL over NVLink/NVSwitch) and merged on
  every rank.  The merged result is bit-identical to the single-GPU result.
"""
from __future__ import annotations

from .ransac import MOSAIC


def shard_bounds(n: int, world: int, rank: int):
    """Contiguous range [lo, hi) of shard `rank` out of `world` over n items; the first
    n % world shards get one extra item."""
    q, r = divmod(n, world)
    lo = rank * q + min(rank, r)
    return lo, lo + q + (1 if rank < r else 0)


def frame_range(n_frames: int, world: int, rank: int, overlap: int = 0):
    """Frames of a batch / stream owned by `rank`.  overlap = 1 for consecutive-frame matching
    streams: every rank but the last also computes the first frame of the next range, so no
    descriptors have to cross GPUs (SURVEY.md 8e)."""
    lo, hi = shard_bounds(n_frames, world, rank)
    return lo, min(n_frames, hi + (overlap if rank + 1 < world else 0))


def match_sharded(A, B_shard, shard_offset: int, ambiguity: float = 0.8, group=None,
                  top2=None, merge=None):
    """Match replicated queries A against a row-sharded database.  `top2` / `merge` default to
    the CUDA entry points (nm_match_top2_f32 / nm_match_merge_top2); the CPU gloo tests pass the
    oracle's functions to exercise the same orchestration without a GPU."""
    import torch
    import torch.distributed as dist
    from .match import match_top2 as _top2, merge_top2 as _merge   # (the package attribute `match` is the function)
    top2 = top2 or _top2
    merge = merge or _merge
    rec = top2(A, B_shard, shard_offset)
    world = dist.get_world_size(group)
    n = rec.shape[0]
    allrec = torch.empty((world * n,) + tuple(rec.shape[1:]), dtype=rec.dtype, device=rec.device)
    dist.all_gather_into_tensor(allrec, rec.contiguous(), group=group)     # shard-major
    return merge(allrec.view((world, n) + tuple(rec.shape[1:])), ambiguity)


def stream_pairs(n_frames: int, world: int, rank: int):
    """Consecutive-frame pairs (t, t+1) owned by `rank` of a mosaicking stream (BASELINE.json
    configs[4]): its contiguous frame range plus one overlap frame, so no descriptors cross GPUs."""
    lo, hi = frame_range(n_frames, world, rank, overlap=1)
    return lo, hi, [(t, t + 1) for t in range(lo, hi - 1)]


def match_stream(sift_batch, frames, ambiguity: float = 0.8, world: int = 1, rank: int = 0, chunk: int = 16):
    """SIFT detect+describe on this rank's frames of a stream and match every frame to its
    successor.  frames: cuda float32 (n, h, w) holding the WHOLE stream (or at least this rank's
    range).  Returns {t: match indices of frame t into frame t+1} for the pairs this rank owns."""
    import torch
    from .match import match as _match
    n = frames.shape[0]
    lo, hi, pairs = stream_pairs(n, world, rank)
    out, prev = {}, None
    for c0 in range(lo, hi, chunk):
        c1 = min(hi, c0 + chunk)
        sift_batch.run(frames[c0:c1].contiguous())
        r = sift_batch.results()
        counts = r["counts"][: c1 - c0].tolist()
        descs = [r["desc"][i, : counts[i]].clone() for i in range(c1 - c0)]
        for i, d in enumerate(descs):
            t = c0 + i
            if prev is not None and prev[0] == t - 1:
                if prev[1].shape[0] and d.shape[0]:
                    out[t - 1] = _match(prev[1], d, ambiguity)
                else:
                    out[t - 1] = torch.full((prev[1].shape[0],), -1, dtype=torch.int32, device=frames.device)
            prev = (t, d)
    return out


def register_stream(sift_batch, frames, kind: int = 2, ambiguity: float = 0.8, inlier_threshold: float = 4.0,
                    iterations: int = 1024, seed: int = 0, world: int = 1, rank: int = 0, chunk: int = 16,
                    refine_rounds: int = 0):
    """BASELINE.json configs[4] with its consumer: SIFT on this rank's frames of a stream, every frame matched to
    its successor, correspondences aligned (align_points) and ONE batched RANSAC over all the rank's pairs.
    Returns (pairs, homographies (n_pairs, 9) cuda, status (n_pairs, 3) cuda); pair t -> t+1 maps frame t's
    coordinates to frame t+1's.  Pair t uses the seed `seed + t` (independent of the sharding).  refine_rounds > 0
    refits every model on its inliers (ransac.refine_batch, in place); status[:, 2] is then the refits kept."""
    import torch
    from .match import match as _match
    from .ransac import align_points, ransac_batch, refine_batch
    n = frames.shape[0]
    lo, hi, pairs = stream_pairs(n, world, rank)
    cap = sift_batch.capacity
    dev = frames.device
    npairs = len(pairs)
    c = [torch.full((max(npairs, 1), cap), -1.0, dtype=torch.float32, device=dev) for _ in range(4)]
    counts = torch.zeros(max(npairs, 1), dtype=torch.int32, device=dev)
    prev = None
    for c0 in range(lo, hi, chunk):
        c1 = min(hi, c0 + chunk)
        sift_batch.run(frames[c0:c1].contiguous())
        r = sift_batch.results()
        cnt = r["counts"][: c1 - c0].tolist()
        for i in range(c1 - c0):
            t = c0 + i
            cur = (t, r["desc"][i, : cnt[i]].clone(), r["x"][i, : cnt[i]].clone(), r["y"][i, : cnt[i]].clone())
            if prev is not None and prev[0] == t - 1 and prev[1].shape[0] and cur[1].shape[0]:
                m = _match(prev[1], cur[1], ambiguity)
                al = align_points(prev[2], prev[3], cur[2], cur[3], m)
                k = t - 1 - lo
                for a, b in zip(c, al):
                    a[k, : b.shape[0]] = b
                counts[k] = prev[1].shape[0]
            prev = cur
    if npairs == 0:
        return pairs, torch.zeros((0, 9), device=dev), torch.zeros((0, 3), dtype=torch.int32, device=dev)
    # one seed per PAIR INDEX of the whole stream, so a sharded run reproduces the single-rank run
    H, st = ransac_batch(kind, *c, counts, inlier_threshold, iterations, seed + lo)
    if refine_rounds > 0:
        refine_batch(kind, *c, counts, H, st, inlier_threshold, refine_rounds, out=(H, st))
    return pairs, H, st


class StreamRegistrar:
    """BASELINE.json configs[4] as ONE device-side launch sequence per chunk of frames: batched SIFT (nm_sift_run),
    every frame matched to its successor on the tcgen05 engine (nm_match_pairs_f32), correspondences aligned
    (nm_align_pairs_f32) and all pairs registered by one batched RANSAC (nm_ransac_batch_f32).  Keypoint counts never
    leave the device and nothing synchronises; consecutive chunks share one frame (recomputed), so no state is carried
    between chunks or between GPUs.  Pair t -> t + 1 draws with seed + t: the result does not depend on the chunking or
    on how the stream is sharded over ranks (frame_range(..., overlap=1)).  refine_rounds > 0 refits each chunk's models
    on their inliers in place (nm_ransac_refine_batch_f32) right after its RANSAC; status[:, 2] is then the refits kept.

    span > 1 (at most 8) registers every frame t of a chunk also to t + 2 ... t + span and adjusts the chunk's poses
    jointly: each chunk [c0, c1) is one adjustment window of the span layout (span min(span, c1 - c0 - 1)), run as
    match_pairs_span, align_pairs_span, one ransac_batch per d (link (t, d), t in stream coordinates, draws with seed +
    t + ((d - 1) << 40)), refine_batch on all links (rounds = refine_rounds, 0 = masks only) and adjust_chain, whose
    pairwise models and status [connected, inliers, LM steps accepted] are returned (status[:, 2] counts LM steps here,
    not refits kept; adjust_iterations bounds the LM builds per window; adjust_cost is adjust_chain's residual: MOSAIC,
    the default, or TRANSFER, which keeps long windows of similarity or homography models from contracting).  A frame
    that no usable link reaches keeps its predecessor's pose (status 0).  The result then depends on the window
    boundaries -- lo and the chunk size -- and on nothing else.  span = 1 calls nothing new.

    overlap O (1 <= O <= span; chunk >= O + 2 when O > 1) is the number of frames consecutive windows share: windows
    start at lo, then at the previous window's end minus O.  The first window of a call is unanchored; every later one
    holds its first O frames at the previous window's adjusted poses (adjust_chain(fixed=...): its last O chain rows,
    connected flags from its status) and writes only the pairs whose later frame is free.  With O = span every link (t, t + d) lies
    in the window where t + d is free, so no skip link is lost at a window boundary.  The extra cost is the SIFT and
    matching of O - 1 more frames per window.  O = 1 (the default) is the behaviour above.  Windows are anchored within
    one call on one rank only: the first window of each rank's range is unanchored, so ranks share no state and need
    no collective (run(..., resume=True) continues a call on the same registrar)."""

    def __init__(self, sift_batch, chunk=None, kind: int = 2, ambiguity: float = 0.8, inlier_threshold: float = 4.0,
                 iterations: int = 1024, seed: int = 0, refine_rounds: int = 0, span: int = 1, adjust_iterations: int = 10,
                 adjust_cost: int = MOSAIC, overlap: int = 1):
        import torch
        self.sb = sift_batch
        self.chunk = min(chunk or sift_batch.max_batch, sift_batch.max_batch)
        assert self.chunk >= 2 and sift_batch.capacity % 256 == 0
        self.kind, self.ambiguity, self.thr, self.iters, self.seed = kind, ambiguity, inlier_threshold, iterations, seed
        self.refine_rounds = refine_rounds
        assert 1 <= span <= 8
        self.span, self.adjust_iterations, self.adjust_cost = span, adjust_iterations, adjust_cost
        if not 1 <= overlap <= span:
            raise ValueError(f"overlap {overlap}: expected 1 <= overlap <= span ({span})")
        if overlap > 1 and self.chunk < overlap + 2:          # overlap 1 keeps the chunk >= 2 of unanchored windows
            raise ValueError(f"chunk {self.chunk} < overlap + 2 ({overlap + 2})")
        self.overlap = overlap
        self._tail = None        # end of the last run: (hi, chain rows, conn, its last overlap - 1 pairs and status)
        cap, n = sift_batch.capacity, self.chunk - 1
        dev = torch.device("cuda", torch.cuda.current_device())
        self.match = torch.empty((n, cap), dtype=torch.int32, device=dev)
        self.corr = [torch.empty((n, cap), dtype=torch.float32, device=dev) for _ in range(4)]

    def run(self, frames_of, lo: int, hi: int, resume: bool = False):
        """frames_of(t0, t1) -> frames [t0, t1) of the stream on the device: cuda float32 (t1 - t0, h, w), or BGRA video
        frames, cuda uint8 (t1 - t0, h, w, 4), whose grey conversion is fused into the base blur (nm_sift_run_bgra) --
        the same colour buffer then feeds the mosaic (mosaic.render_stream).  Registers every pair (t, t + 1) with
        lo <= t < hi - 1.  Returns (homographies (hi - lo - 1, 9), status (hi - lo - 1, 3)) on the device.
        resume=True appends to the previous call (a live session): lo must be that call's hi - overlap, the first window
        is anchored on the end of that call's last window, and the first overlap - 1 rows returned are that call's."""
        import ctypes as C
        import torch
        from . import _lib
        from ._lib import check
        from .sift import _stream_ptr
        lib = _lib.load()
        sb, cap = self.sb, self.sb.capacity
        O = self.overlap
        anchor = None                               # (chain rows, conn) the next window holds fixed
        if resume:
            if self._tail is None or lo != self._tail[0] - O or hi <= self._tail[0]:
                raise ValueError("resume: needs a previous call, lo = its hi - overlap and hi > its hi")
            anchor = self._tail[1:3] if O > 1 else None
        n_pairs = max(hi - lo - 1, 0)
        H = torch.zeros((max(n_pairs, 1), 9), dtype=torch.float32, device=self.match.device)
        st = torch.zeros((max(n_pairs, 1), 3), dtype=torch.int32, device=self.match.device)
        if n_pairs == 0:
            return H[:0], st[:0]
        if resume and O > 1:
            H[: O - 1], st[: O - 1] = self._tail[3], self._tail[4]
        r = sb.results()
        p = lambda t: C.c_void_p(t.data_ptr())
        c0 = lo
        while c0 < hi - 1:
            c1 = min(hi, c0 + self.chunk)
            n = c1 - c0
            chunk = frames_of(c0, c1)
            if chunk.dtype == torch.uint8 and chunk.dim() == 4 and chunk.shape[-1] == 4:
                sb.run_bgra(chunk)
            else:
                sb.run(chunk)
            k = c0 - lo
            if self.span > 1:
                # an anchored window writes the pairs of its free frames only: the first O - 1 are the last window's
                a = O - 1 if anchor is not None else 0
                out = (H[k: k + n - 1], st[k: k + n - 1]) if a == 0 else None
                Hw, Sw, chain, _ = adjust_window(r, n, min(self.span, n - 1), chunk.shape[2], chunk.shape[1], self.kind,
                                                 self.ambiguity, self.thr, self.iters, self.seed + c0, self.refine_rounds,
                                                 out=out, adjust_iterations=self.adjust_iterations,
                                                 adjust_cost=self.adjust_cost, fixed=anchor)
                if a:
                    H[k + a: k + n - 1], st[k + a: k + n - 1] = Hw[a:], Sw[a:]
                self._tail = (c1,)
                if O > 1:
                    anchor = (chain[n - O:], Sw[n - O - 1: n - 1, 0].clone(memory_format=torch.contiguous_format))
                    self._tail += anchor + (Hw[n - O:].clone(), Sw[n - O:].clone())
                if c1 >= hi:
                    break
                c0 = c1 - O
                continue
            self.match[: n - 1].fill_(-1)
            check(lib.nm_match_pairs_f32(p(r["desc"]), p(r["counts"]), n, cap, self.ambiguity, p(self.match), None, None,
                                         _stream_ptr()), "nm_match_pairs_f32")
            check(lib.nm_align_pairs_f32(p(r["x"]), p(r["y"]), p(self.match), p(r["counts"]), n, cap, *[p(c) for c in self.corr],
                                         _stream_ptr()), "nm_align_pairs_f32")
            check(lib.nm_ransac_batch_f32(self.kind, *[p(c) for c in self.corr], cap, p(r["counts"]), cap, n - 1, self.thr,
                                          self.iters, (self.seed + c0) & 0xFFFFFFFFFFFFFFFF, p(H[k:]), p(st[k:]), _stream_ptr()),
                  "nm_ransac_batch_f32")
            if self.refine_rounds > 0:
                check(lib.nm_ransac_refine_batch_f32(self.kind, *[p(c) for c in self.corr], cap, p(r["counts"]), cap, n - 1,
                                                     self.thr, p(H[k:]), p(st[k:]), self.refine_rounds, p(H[k:]), p(st[k:]),
                                                     None, _stream_ptr()), "nm_ransac_refine_batch_f32")
            self._tail = (c1,)
            c0 = c1 - 1
        return H[:n_pairs], st[:n_pairs]


def adjust_window(res, n, span, frame_w, frame_h, kind, ambiguity, inlier_threshold, iterations, seed, refine_rounds, out,
                  adjust_iterations: int = 10, adjust_cost: int = MOSAIC, fixed=None):
    """One adjustment window of StreamRegistrar(span > 1): frames 0 .. n-1 of the SIFT results `res` (SiftBatch.results())
    through the five public calls.  seed = the stream seed + the window's first frame.  Writes the window's n - 1 pairwise
    models and status into out = (H, status), or new tensors when out is None; returns adjust_chain's (H, status, chain,
    report).  adjust_cost and fixed: adjust_chain's cost (MOSAIC or TRANSFER) and fixed frames."""
    import torch
    from .match import match_pairs_span, link_row
    from .ransac import align_pairs_span, ransac_batch, refine_batch, adjust_chain
    counts = res["counts"][:n]
    m = match_pairs_span(res["desc"][:n], counts, span, ambiguity)
    corr = align_pairs_span(res["x"][:n], res["y"][:n], m, counts, span)
    HL, SL = [], []
    for d in range(1, span + 1):
        r0 = link_row(n, 0, d)
        Hd, Sd = ransac_batch(kind, *[c[r0: r0 + n - d] for c in corr], counts[: n - d], inlier_threshold, iterations,
                              seed + ((d - 1) << 40))
        HL.append(Hd)
        SL.append(Sd)
    link_counts = torch.cat([counts[: n - d] for d in range(1, span + 1)])
    HL, SL, mask = refine_batch(kind, *corr, link_counts, torch.cat(HL), torch.cat(SL), inlier_threshold, refine_rounds)
    return adjust_chain(kind, *corr, link_counts, span, mask, HL, SL, frame_w, frame_h, inlier_threshold, adjust_iterations, out=out,
                        cost=adjust_cost, fixed=fixed)
