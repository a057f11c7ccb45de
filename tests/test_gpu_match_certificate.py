"""The tensor-core matcher's certificate and every exact path behind it (nm_match_tc.cu, nm_match.cu).

1. The certificate's assumption, restated in float64 (tests/match_cert_ref.py): no column outside the candidate lists
   scores above thr + eta/2 (soundness), on every input family and at the sizes where the scan changes shape (seed
   pass, splits, re-rank rounds, 256-row query blocks).  The candidates' own error is measured in test_gpu_match.py
   (test_tc_accumulation_error_within_certificate_margin, test_tc_accumulation_error_on_input_families).
2. Near-tie clusters that no certificate can pass, so that each fallback path runs with a known number of rows:
   scan_rows_small_kernel (<= 256 listed rows), scan_exact_kernel<false, true> (longer lists, grid-stride loop),
   a non-zero index offset, and the in-warp exact scan of the batched pair matcher.
3. The ratio rule's edge values (column-0 start value, a ratio of exactly the ambiguity, min2 == 0, one database row)
   through every engine and every copy of the rule."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from niftymatch_b200 import synth  # noqa: E402
from niftymatch_b200.match import link_row, span_links  # noqa: E402
from tests import match_cert_ref as mcr  # noqa: E402

gpu = pytest.mark.gpu

NB_SIZES = [2, 4, 5, 10, 11, 65, 129, 3968, 3969, 10113, 40000]
NA_SIZES = [1, 255, 256, 257, 513]
CLUSTER = 40                     # rows per near-tie cluster: more than the 4 a list keeps, in every list they reach


@pytest.fixture(scope="module")
def nm():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import niftymatch_b200 as nm
    nm.load()
    try:
        nm.set_engine(1)
    except nm.NmError:
        pytest.skip("tensor-core engine unavailable on this device")
    nm.set_engine(-1)
    return nm


def _cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _top2_true(oracle, A, B, offset=0):
    rec = np.zeros((len(A), 4), np.float32)
    oracle.lib.orc_match_top2_true(_p(A), len(A), _p(B), len(B), offset, _p(rec))
    return rec


def _bits(rec):
    return np.ascontiguousarray(rec, np.float32).view(np.uint32)[..., :3]


# ---- 1. the certificate's assumption ------------------------------------------------------------------------------
def test_threshold_sizes_cover_every_seed_regime():
    """The sizes of test_certificate_sound_at_threshold_sizes reach every regime of the host's seed-pass formula:
    off (< 32 database tiles), the 4-tile floor, in between, and the 16-tile cap."""
    seeds = [mcr.seed_tiles(n) for n in NB_SIZES]
    assert 0 in seeds and 4 in seeds and 16 in seeds and any(4 < s < 16 for s in seeds), seeds
    assert mcr.seed_tiles(3968) == 0 and mcr.seed_tiles(3969) == 4 and mcr.seed_tiles(10113) == 5
    assert (40000 + 127) // 128 // 16 > 16


@gpu
@pytest.mark.parametrize("fam", mcr.FAMILIES)
def test_certificate_sound_on_input_families(nm, oracle, fam):
    """(a) on the benchmark's descriptors, real SIFT descriptors and the adversarial operands; records bitwise equal
    to the oracle's true top-2."""
    A, B = mcr.family(fam, nm, torch)
    pr = nm.tc_probe(_cu(A), _cu(B), want_candidates=True)
    r = mcr.certificate_ratios(A, B, pr)
    print(f"{fam}: {len(A)} x {len(B)}, {pr['n_lists']} lists, {pr['fallback_rows']} fallback rows; worst non-candidate "
          f"(S - thr) / (eta/2) {mcr.log2_str(r['sound'])}, candidate error {mcr.log2_str(r['cand'])} of eta/2, "
          f"{mcr.log2_str(r['cand_rel'])} of |a^|^2 + |b^|^2")
    assert r["sound"] <= 1.0, r
    assert np.array_equal(_bits(pr["rec"].cpu().numpy()), _bits(_top2_true(oracle, A, B)))


@gpu
@pytest.mark.parametrize("nB", NB_SIZES)
def test_certificate_sound_at_threshold_sizes(nm, oracle, nB):
    """(a) and (b) where the scan changes shape: the seed pass off / on / capped (nB 3968, 3969, 10113, 40000), the two
    re-rank rounds of 4 and 10 candidates and the all-evaluated shortcut (nB 2 .. 11), partial tiles and halves (65,
    129), and 1 .. 3 query blocks of 256 rows.  The split count is checked against the host's formula."""
    n_sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = synth.descriptors(nB, 500 + nB)
    Bt = _cu(B)
    worst = {"sound": -np.inf, "cand": 0.0}
    for nA in NA_SIZES:
        A = synth.descriptors(nA, 600 + nA, planted_from=B)
        pr = nm.tc_probe(_cu(A), Bt, want_candidates=True)
        assert pr["n_lists"] == 2 * mcr.tc_splits(nA, nB, n_sms), (nA, nB, pr["n_lists"])
        r = mcr.certificate_ratios(A, B, pr)
        assert r["sound"] <= 1.0 and r["cand"] <= 1.0, (nA, nB, r)
        assert np.array_equal(_bits(pr["rec"].cpu().numpy()), _bits(_top2_true(oracle, A, B))), (nA, nB)
        worst = {k: max(worst[k], r[k]) for k in worst}
    print(f"nB {nB} (seed tiles {mcr.seed_tiles(nB)}): worst (S - thr) / (eta/2) {mcr.log2_str(worst['sound'])}, "
          f"candidate error {mcr.log2_str(worst['cand'])} of eta/2")


# ---- 2. forced certificate failures -------------------------------------------------------------------------------
def _near(c16, s, n, rng):
    """n pairwise different float32 rows that all round to the fp16 row c16 (scaled units) at scale s: every nonzero
    component moves by less than a quarter of its fp16 spacing.  Their tensor-core scores tie, their fp32 distances
    do not."""
    mag = np.abs(c16)
    ulp = np.where(mag >= mcr.F16_MIN_NORMAL, 2.0 ** (np.floor(np.log2(np.maximum(mag, mcr.F16_MIN_NORMAL))) - 10), 0.0)
    rows = ((c16 + ulp * rng.uniform(-0.24, 0.24, (n, 128))) / s).astype(np.float32)
    assert (mcr.fp16_scaled(rows, s) == c16).all()
    return rows


def _plant(B, at, s, rng):
    """Replaces B[at : at + CLUSTER] by a near-tie cluster around B[at]'s fp16 row; returns the centre."""
    c16 = mcr.fp16_scaled(B[at:at + 1], s)[0]
    B[at:at + CLUSTER] = _near(c16, s, CLUSTER, rng)
    return c16


def _cluster_problem(nA, nB, K, seed):
    """synth descriptors with three clusters in the database (one at the last rows) and K queries near them; one
    element of database row 0 sets the scale, so that the clusters cannot change it."""
    rng = np.random.default_rng(seed)
    B = synth.descriptors(nB, seed)
    A = synth.descriptors(nA, seed + 1, planted_from=B)
    B[0, 0] = 1.5 * max(A.max(), B.max())            # sets the scale; row 0 is in no cluster
    s = mcr.tc_scale(A, B)
    centres = [_plant(B, at, s, rng) for at in (7, nB // 2 + 3, nB - CLUSTER)]
    for q in range(K):
        A[q] = _near(centres[q % 3], s, 1, rng)[0]
    assert mcr.tc_scale(A, B) == s
    return A, B


def _slack(n_other):
    return max(4, n_other // 50)


@gpu
@pytest.mark.parametrize("K,nA,nB", [(1, 300, 1037), (256, 256, 3001), (257, 257, 3001), (5000, 6000, 5003)])
def test_forced_fallback_rows(nm, oracle, K, nA, nB):
    """K cluster queries fail the certificate: 256 is the last list length of scan_rows_small_kernel, 257 the first of
    scan_exact_kernel<false, true>, 5000 runs its grid-stride loop over 32 x 64 rows three times; nB is no multiple of
    64 or 256 (chunk and split tails; 5003 also has the seed pass).  Records bitwise equal to the oracle's."""
    A, B = _cluster_problem(nA, nB, K, 40 + K)
    pr = nm.tc_probe(_cu(A), _cu(B))
    fb = pr["fallback_rows"]
    if nA == K:
        assert fb == K, fb
    else:
        assert K <= fb <= K + _slack(nA - K), fb
    assert np.array_equal(_bits(pr["rec"].cpu().numpy()), _bits(_top2_true(oracle, A, B)))


@gpu
@pytest.mark.parametrize("K", [1, 257])
def test_forced_fallback_with_index_offset(nm, oracle, K):
    """The same through match_top2 with a shard offset on the tensor-core engine: both fallback kernels add the offset
    (the records carry global database indices)."""
    A, B = _cluster_problem(K, 3001, K, 90 + K)
    off = 123457
    nm.set_engine(1)
    try:
        rec = nm.match_top2(_cu(A), _cu(B), index_offset=off).cpu().numpy()
        fb = nm.tc_probe(_cu(A), _cu(B))["fallback_rows"]
    finally:
        nm.set_engine(-1)
    assert fb == K, fb
    assert np.array_equal(_bits(rec), _bits(_top2_true(oracle, A, B, off)))


def _pair_frames(cap=2048):
    """Five frames, clusters planted so that pair p has K_p = (whole frame, 1, 300, 0) queries near a cluster of
    frame p + 1: frame 0 is entirely near frame 1's cluster (at frame-local rows 0..39, so column 0 is the best one),
    frame 1 row 100 near frame 2's cluster (its last rows), frame 2 rows 100..399 near frame 3's (rows 500..539)."""
    counts = [cap, 1337, 1501, 999, 1100]
    rng = np.random.default_rng(17)
    desc = (rng.random((len(counts), cap, 128)) * 300).astype(np.float32)         # stale rows beyond the counts
    prev = None
    for f, c in enumerate(counts):
        desc[f, :c] = synth.descriptors(c, 700 + f, planted_from=prev)
        prev = desc[f, :c]
    desc[4, 0, 0] = 1.5 * desc[:, :1100].max()                                     # sets the scale, in no cluster
    s = mcr.tc_scale(np.concatenate([desc[f, :c] for f, c in enumerate(counts)]), np.zeros((1, 128), np.float32))
    c1 = _plant(desc[1], 0, s, rng)
    c2 = _plant(desc[2], counts[2] - CLUSTER, s, rng)
    c3 = _plant(desc[3], 500, s, rng)
    desc[0, :counts[0]] = _near(c1, s, counts[0], rng)
    desc[1, 100] = _near(c2, s, 1, rng)[0]
    desc[2, 100:400] = _near(c3, s, 300, rng)
    assert mcr.tc_scale(np.concatenate([desc[f, :c] for f, c in enumerate(counts)]), np.zeros((1, 128), np.float32)) == s
    return desc, counts, counts[0] + 1 + 300


@gpu
@pytest.mark.parametrize("span", [1, 3])
def test_forced_fallback_in_pair_matcher(nm, span):
    """match_pairs / match_pairs_span on frames with planted clusters: the in-warp exact scan of pairs_rerank_kernel
    runs for at least the planted rows, and every link's records and indices equal one exact-engine call per link."""
    desc, counts, planted = _pair_frames()
    n, cap = len(counts), desc.shape[1]
    dd, cc = _cu(desc), torch.tensor(counts, dtype=torch.int32, device="cuda")
    L = span_links(n, span)
    init = torch.full((L, cap), 55, dtype=torch.int32, device="cuda")
    if span == 1:
        m, rec, fb = nm.match_pairs(dd, cc, 0.8, match_out=init.clone(), want_records=True)
    else:
        m, rec, fb = nm.match_pairs_span(dd, cc, span, 0.8, match_out=init.clone(), want_records=True)
    torch.cuda.synchronize()
    m, rec, fb = m.cpu().numpy(), rec.cpu().numpy(), int(fb.item())
    assert fb >= planted, (fb, planted)
    if span == 1:
        assert fb <= planted + _slack(sum(counts[:-1]) - planted), (fb, planted)
    nm.set_engine(0)
    try:
        for d in range(1, span + 1):
            for t in range(n - d):
                row = link_row(n, t, d)
                nA, nB = counts[t], counts[t + d]
                At, Bt = dd[t, :nA], dd[t + d, :nB]
                r2 = nm.match_top2(At, Bt).cpu().numpy()
                assert np.array_equal(_bits(rec[row, :nA]), _bits(r2)), (t, d)
                ref = nm.match(At, Bt, 0.8, match_io=init[row, :nA].clone()).cpu().numpy()
                assert np.array_equal(m[row, :nA], ref), (t, d)
                assert (m[row, nA:] == 55).all(), (t, d)
    finally:
        nm.set_engine(-1)


# ---- 3. the ratio rule's edge values ------------------------------------------------------------------------------
def _rule_rows():
    """Rows whose records sit on the ratio rule's edges; returns A, B and the expected indices (start value 55).
      q0: best column 0 at d1 = 0.85 * 2139095040, true d2 = 2.4995e9: the start value 2139095040.0f is min2, so the
          row is rejected, although d1 / d2 < 0.8
      q1: d1 = 4, d2 = 5: fdiv_rn gives exactly 0.8f and the strict < rejects it
      q2: two database rows at distance 0: min2 == 0 keeps the previous value
      q3: best column 0 at distance 0: matched
      q4: an ordinary match (column 2)."""
    z = np.zeros(128, np.float32)
    e = np.eye(128, dtype=np.float32)
    P, R = z + 5000.0, z + 4800.0
    B = np.stack([z + 3769.0, z + 4419.0, P + 2 * e[0], P + e[0] + 2 * e[1], R, R])
    A = np.stack([z, P, R, B[0], P + 2 * e[0] + 0.5 * e[5]])
    return A, B, np.array([-1, -1, 55, 0, 2], np.int32)


def _single_row():
    z = np.zeros(128, np.float32)
    B = np.stack([z + 3769.0])
    A = np.stack([z, B[0], B[0] + 10.0 * np.eye(128, dtype=np.float32)[0]])
    return A, B, np.array([-1, 0, 0], np.int32)


def test_rule_rows_sit_on_the_edges(oracle):
    """The oracle sees the edges the rows are built for: the column-0 start value decides q0, q1's ratio is exactly
    0.8f, q2's second distance is 0, and one database row keeps min2 at the start value."""
    A, B, want = _rule_rows()
    rec = _top2_true(oracle, A, B)
    d1, d2 = rec[:, 0], rec[:, 2]
    assert rec[0, 1].view(np.int32) == 0 and d1[0] / np.float32(2139095040.0) >= 0.8 and d1[0] / d2[0] < 0.8
    assert d1[1] == 4.0 and d2[1] == 5.0 and np.float32(4.0) / np.float32(5.0) == np.float32(0.8)
    assert d1[2] == 0.0 and d2[2] == 0.0
    assert np.array_equal(oracle.match(A, B, 0.8, match_io=np.full(len(A), 55, np.int32)), want)
    A1, B1, want1 = _single_row()
    assert np.array_equal(oracle.match(A1, B1, 0.8, match_io=np.full(len(A1), 55, np.int32)), want1)


@gpu
@pytest.mark.parametrize("case", ["edges", "single_row"])
def test_ratio_rule_edges_in_every_engine(nm, oracle, case):
    """The edge rows through engine 0 and 1 (merge_kernel), match_top2 over 3 shards + merge_top2 (global column 0 in
    shard 0), match_pairs / match_pairs_span (pairs_rerank_kernel, frame-local column 0) and nm_dist2_f32 +
    nm_set_matches_f32 (set_matches_kernel): the same indices as the oracle."""
    import niftymatch_b200._lib as L
    A, B, want = _rule_rows() if case == "edges" else _single_row()
    nA, nB = len(A), len(B)
    init = np.full(nA, 55, np.int32)
    mo = oracle.match(A, B, 0.8, match_io=init)
    assert np.array_equal(mo, want)
    At, Bt = _cu(A), _cu(B)
    for eng in (0, 1):
        nm.set_engine(eng)
        try:
            assert np.array_equal(nm.match(At, Bt, 0.8, match_io=_cu(init)).cpu().numpy(), mo), eng
            if nB >= 3:
                bounds = [0, 2, 4, nB]                                   # global column 0 in shard 0
                recs = torch.stack([nm.match_top2(At, Bt[lo:hi].contiguous(), lo) for lo, hi in zip(bounds, bounds[1:])])
                orc_recs = np.stack([_top2_true(oracle, A, np.ascontiguousarray(B[lo:hi]), lo)
                                     for lo, hi in zip(bounds, bounds[1:])])
                assert np.array_equal(_bits(recs.cpu().numpy()), _bits(orc_recs)), eng
                m_orc = init.copy()
                oracle.lib.orc_merge_top2(_p(orc_recs), 3, nA, C.c_float(0.8), _p(m_orc))
                assert np.array_equal(m_orc, mo)
                assert np.array_equal(nm.merge_top2(recs.contiguous(), 0.8, match_io=_cu(init)).cpu().numpy(), mo), eng
        finally:
            nm.set_engine(-1)
    # batched pair matcher: frames A, B, A, B (every link starts at frame-local column 0)
    cap = 256
    frames = [A, B, A, B]
    desc = np.zeros((4, cap, 128), np.float32)
    for f, X in enumerate(frames):
        desc[f, :len(X)] = X
    dd, cc = _cu(desc), torch.tensor([len(X) for X in frames], dtype=torch.int32, device="cuda")
    for span in (1, 3):
        Lk = span_links(4, span)
        out = torch.full((Lk, cap), 55, dtype=torch.int32, device="cuda")
        m = (nm.match_pairs(dd, cc, 0.8, match_out=out) if span == 1 else
             nm.match_pairs_span(dd, cc, span, 0.8, match_out=out)).cpu().numpy()
        for d in range(1, span + 1):
            for t in range(4 - d):
                Xa, Xb = frames[t], frames[t + d]
                ref = oracle.match(Xa, Xb, 0.8, match_io=np.full(len(Xa), 55, np.int32))
                assert np.array_equal(m[link_row(4, t, d), :len(Xa)], ref), (span, t, d)
    # compat operators: A dim-major in, D^T out, then set_matches on the materialised matrix
    lib = L.load()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    A_T = _cu(np.ascontiguousarray(A.T))
    D_T = torch.empty((nB, nA), dtype=torch.float32, device="cuda")
    assert lib.nm_dist2_f32(C.c_void_p(A_T.data_ptr()), nA, C.c_void_p(Bt.data_ptr()), nB, 128, C.c_void_p(D_T.data_ptr()), st) == 0
    D = D_T.t().contiguous()
    m = _cu(init)
    assert lib.nm_set_matches_f32(C.c_void_p(D.data_ptr()), nA, nB, nB, C.c_void_p(m.data_ptr()), C.c_float(0.8), st) == 0
    assert np.array_equal(m.cpu().numpy(), mo)
