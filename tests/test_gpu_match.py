"""GPU suite: brute-force k=2 ratio-test matching through the C-ABI."""
import ctypes as C
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from niftymatch_b200 import synth  # noqa: E402
from tests import match_cert_ref as mcr  # noqa: E402
from tests._util import GOLDEN  # noqa: E402


@pytest.fixture(scope="module")
def nm():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import niftymatch_b200 as nm
    nm.load()
    return nm


def _cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _engines(nm):
    e = [0]
    try:
        nm.set_engine(1)
        e.append(1)
    except nm.NmError:
        pass
    nm.set_engine(-1)
    return e


def test_match_vs_reference_golden(nm):
    g = np.load(os.path.join(GOLDEN, "match_200x250.npz"))
    for eng in _engines(nm):
        nm.set_engine(eng)
        m = nm.match(_cu(g["A"]), _cu(g["B"]), 0.8, match_io=_cu(g["m0"]))
        assert np.array_equal(m.cpu().numpy(), g["m"]), f"engine {eng}"
    nm.set_engine(-1)
    m, D = nm.match(_cu(g["A"]), _cu(g["B"]), 0.8, match_io=_cu(g["m0"]), want_distance=True)
    assert np.array_equal(D.cpu().numpy(), g["D"]), "distance matrix not bitwise equal to the reference's"
    assert np.array_equal(m.cpu().numpy(), g["m"])


@pytest.mark.parametrize("nA,nB", [(1, 1), (1, 2), (3, 1), (64, 64), (65, 129), (500, 700), (1000, 37), (2048, 2048)])
def test_match_vs_oracle(nm, oracle, nA, nB):
    B = synth.descriptors(nB, 100 + nB)
    A = synth.descriptors(nA, 200 + nA, planted_from=B)
    mo = oracle.match(A, B, 0.8)
    for eng in _engines(nm):
        nm.set_engine(eng)
        m = nm.match(_cu(A), _cu(B), 0.8)
        assert np.array_equal(m.cpu().numpy(), mo), f"engine {eng}"
    nm.set_engine(-1)


def test_compat_matcher_operators(nm, oracle):
    """transpose + compute_brute_force_distance (A dim-major in, D^T out) + get_sift_matches,
    as compute_sift_matches chains them (reference siftfunctions.cu:15-40)."""
    import niftymatch_b200._lib as L
    lib = L.load()
    B = synth.descriptors(150, 7)
    A = synth.descriptors(90, 8, planted_from=B)
    At, Bt = _cu(A), _cu(B)
    A_T = torch.empty((128, 90), dtype=torch.float32, device="cuda")
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.nm_transpose_f32(C.c_void_p(A_T.data_ptr()), C.c_void_p(At.data_ptr()), 128, 90, st) == 0
    assert np.array_equal(A_T.cpu().numpy(), A.T)
    D_T = torch.empty((150, 90), dtype=torch.float32, device="cuda")
    assert lib.nm_dist2_f32(C.c_void_p(A_T.data_ptr()), 90, C.c_void_p(Bt.data_ptr()), 150, 128, C.c_void_p(D_T.data_ptr()), st) == 0
    mo, Do = oracle.match(A, B, 0.8, want_distance=True)
    assert np.array_equal(D_T.cpu().numpy().T, Do)
    D = D_T.t().contiguous()
    m = torch.full((90,), -1, dtype=torch.int32, device="cuda")
    assert lib.nm_set_matches_f32(C.c_void_p(D.data_ptr()), 90, 150, 150, C.c_void_p(m.data_ptr()), 0.8, st) == 0
    assert np.array_equal(m.cpu().numpy(), mo)


@pytest.mark.parametrize("shards", [2, 3, 8])
def test_sharded_records_merge_bit_identical(nm, oracle, shards):
    """Database sharding emulated on one GPU: per-shard records + merge == unsharded result
    (the N>1 collective path all-gathers exactly these records)."""
    from niftymatch_b200.dist import shard_bounds
    B = synth.descriptors(1000, 31)
    A = synth.descriptors(600, 32, planted_from=B)
    At = _cu(A)
    single = nm.match(At, _cu(B), 0.8).cpu().numpy()
    recs = []
    for s in range(shards):
        lo, hi = shard_bounds(len(B), shards, s)
        recs.append(nm.match_top2(At, _cu(B[lo:hi]), lo))
    m = nm.merge_top2(torch.stack(recs).contiguous(), 0.8).cpu().numpy()
    assert np.array_equal(m, single)
    assert np.array_equal(m, oracle.match(A, B, 0.8))


def test_invalid_arguments_return_codes(nm):
    import niftymatch_b200._lib as L
    lib = L.load()
    a = torch.zeros((4, 128), device="cuda")
    m = torch.zeros(4, dtype=torch.int32, device="cuda")
    assert lib.nm_match_f32(None, 4, C.c_void_p(a.data_ptr()), 4, 0.8, C.c_void_p(m.data_ptr()), None, None) == -1
    assert lib.nm_match_f32(C.c_void_p(a.data_ptr()), 0, C.c_void_p(a.data_ptr()), 4, 0.8, C.c_void_p(m.data_ptr()), None, None) == -1
    assert lib.nm_blur_f32(C.c_void_p(a.data_ptr()), C.c_void_p(a.data_ptr()), None, 4, 4, C.c_void_p(a.data_ptr()), 46, None) == -1


def test_large_match_properties(nm, oracle):
    """20k x 20k: planted rows must match their source; a row subset is checked against the
    oracle exactly."""
    n = 20000
    B = synth.descriptors(n, 2)
    A = synth.descriptors(n, 1, planted_from=B)
    m = nm.match(_cu(A), _cu(B), 0.8).cpu().numpy()
    sub = np.arange(0, n, 313)
    mo = oracle.match(np.ascontiguousarray(A[sub]), B, 0.8)
    assert np.array_equal(m[sub], mo)
    assert (m >= 0).sum() > 0.15 * n


# ---- tensor-core engine (tcgen05 candidate search + exact re-rank + certificate) ---------
def _need_tc(nm):
    try:
        nm.set_engine(1)
    except nm.NmError:
        pytest.skip("tensor-core engine unavailable on this device")
    nm.set_engine(-1)


@pytest.mark.parametrize("nA,nB", [(1, 1), (7, 130), (256, 128), (300, 1000), (1000, 37), (4096, 8192), (9000, 20000)])
def test_tc_records_bitwise_equal_exact_engine(nm, nA, nB):
    """The tcgen05 engine must return the SAME records (d1, i1, d2 bit patterns) as the exact fp32
    scan: candidates come from fp16 tensor-core scores, the values from the reference's fp32
    arithmetic, and rows whose certificate fails are re-scanned exactly."""
    _need_tc(nm)
    B = synth.descriptors(nB, 300 + nB)
    A = synth.descriptors(nA, 400 + nA, planted_from=B)
    At, Bt = _cu(A), _cu(B)
    nm.set_engine(0)
    ref = nm.match_top2(At, Bt)
    nm.set_engine(-1)
    pr = nm.tc_probe(At, Bt)
    assert torch.equal(pr["rec"].view(torch.int32), ref.view(torch.int32))
    assert 0 <= pr["fallback_rows"] <= max(4, nA // 50), pr["fallback_rows"]


def test_tc_engine_hard_cases(nm, oracle):
    """Inputs built to stress the certificate: exact duplicates in the database (ties -> lowest
    index), all-equal rows, a huge dynamic range, zero vectors.  Indices must equal the oracle's."""
    _need_tc(nm)
    rng = np.random.RandomState(5)
    nB, nA = 3000, 700
    B = synth.descriptors(nB, 77)
    B[100:200] = B[0:100]                      # duplicates: ties must resolve to the lower index
    B[500] = 0.0
    B[501:520] = B[501]                        # 19 identical rows
    B[600:700] *= 1e-4                         # tiny rows (fp16 subnormal range after scaling)
    B[700:710] *= 50.0                         # large rows set the global scale
    A = synth.descriptors(nA, 78, planted_from=B)
    A[0:50] = B[100:150]                       # exact copies of duplicated rows: d1 = d2 = 0
    A[50] = 0.0
    A[51:60] = B[501] + rng.randn(9, 128).astype(np.float32) * 0.01
    A[60:70] = B[600:610]
    mo = oracle.match(A, B, 0.8)
    nm.set_engine(1)
    m = nm.match(_cu(A), _cu(B), 0.8).cpu().numpy()
    nm.set_engine(0)
    m0 = nm.match(_cu(A), _cu(B), 0.8).cpu().numpy()
    nm.set_engine(-1)
    assert np.array_equal(m0, mo)
    assert np.array_equal(m, mo)


def _candidate_error(nm, fam):
    """Candidate score errors of the tensor-core scan on one input family (tests/match_cert_ref.py)."""
    _need_tc(nm)
    Ah, Bh = mcr.family(fam, nm, torch)
    pr = nm.tc_probe(_cu(Ah), _cu(Bh), want_candidates=True)
    r = mcr.certificate_ratios(Ah, Bh, pr)
    print(f"{fam}: {len(Ah)} x {len(Bh)}, candidate error {mcr.log2_str(r['cand_rel'])} of |a^|^2 + |b^|^2, "
          f"{mcr.log2_str(r['cand'])} of eta/2")
    assert r["cand"] <= 1.0, r
    return r


def test_tc_accumulation_error_within_certificate_margin(nm):
    """The certificate assumes |S_tensor - S_exact| <= eta / 2 = 2^-18 (|a^|^2 + |b^|^2max) + 2^-17 for the fp32
    accumulation of the fp16 products (nm_match_tc.cu).  Measure it on the candidates against a float64 restatement,
    on the benchmark's descriptors (3000 x 7000 synth.descriptors)."""
    r = _candidate_error(nm, "synth")
    assert r["cand_rel"] < 2.0 ** -20, r          # 4x below what the certificate budgets


@pytest.mark.parametrize("fam", [f for f in mcr.FAMILIES if f != "synth"])
def test_tc_accumulation_error_on_input_families(nm, fam):
    """The same measurement on real SIFT descriptors and on adversarial operands, held to the budget itself with the
    column's own norm: |S_tensor - S_exact| <= 2^-18 (|a^|^2 + |b^_j|^2) + 2^-17."""
    r = _candidate_error(nm, fam)
    assert r["cand_col"] <= 1.0, r


def test_tc_matches_exact_at_scale(nm):
    """40k x 60k: match indices of the two engines must be identical."""
    _need_tc(nm)
    B = synth.descriptors(60000, 2)
    A = synth.descriptors(40000, 1, planted_from=B)
    At, Bt = _cu(A), _cu(B)
    nm.set_engine(1)
    m1 = nm.match(At, Bt, 0.8)
    nm.set_engine(0)
    m0 = nm.match(At, Bt, 0.8)
    nm.set_engine(-1)
    assert torch.equal(m0, m1)
    assert int((m1 >= 0).sum()) > 5000


def test_match_sharded_default_path_single_rank_nccl(nm, oracle):
    """match_sharded with its default CUDA entry points and a real NCCL all-gather (world size 1 here;
    the N > 1 orchestration is covered by tests/test_dist_gloo.py and bench.py --gpus N)."""
    import torch.distributed as dist
    from niftymatch_b200.dist import match_sharded
    created = False
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29533")
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
        created = True
    try:
        B = synth.descriptors(1500, 41)
        A = synth.descriptors(900, 42, planted_from=B)
        m = match_sharded(_cu(A), _cu(B), 0, 0.8).cpu().numpy()
        assert np.array_equal(m, oracle.match(A, B, 0.8))
    finally:
        if created:
            dist.destroy_process_group()


def test_full_size_100k_engines_agree_and_planted_rows_match(nm):
    """BASELINE.json configs[3] at full size on one GPU: 100k x 100k.  The tensor-core engine and the
    exact fp32 engine must return identical indices, and every planted query (a database row plus
    small noise) must match the row it was planted from."""
    _need_tc(nm)
    n = 100000
    Bh = synth.descriptors(n, 2)
    Ah = synth.descriptors(n, 1, planted_from=Bh)
    At, Bt = _cu(Ah), _cu(Bh)
    nm.set_engine(1)
    m1 = nm.match(At, Bt, 0.8)
    nm.set_engine(0)
    m0 = nm.match(At, Bt, 0.8)
    nm.set_engine(-1)
    assert torch.equal(m0, m1)
    # recover the planting (same construction as synth.descriptors)
    k = int(n * 0.2)
    rows = (synth.uniform(1, 14, k) * n).astype(np.int64)
    src = (synth.uniform(1, 15, k) * n).astype(np.int64)
    last = {}
    for r, s_ in zip(rows, src):
        last[int(r)] = int(s_)                      # later plantings overwrite earlier ones
    mm = m1.cpu().numpy()
    rr = np.fromiter(last.keys(), dtype=np.int64)
    ss = np.fromiter(last.values(), dtype=np.int64)
    hit = mm[rr] == ss
    assert hit.mean() > 0.999, hit.mean()


def test_unaligned_descriptor_pointers(nm, oracle):
    """Descriptor blocks that start at a 4-byte (not 16-byte) aligned address, e.g. a slice of a larger
    buffer: the call must still succeed (exact engine) and agree with the oracle."""
    B = synth.descriptors(2500, 51)
    A = synth.descriptors(2000, 52, planted_from=B)
    bufA = torch.zeros(A.size + 1, dtype=torch.float32, device="cuda")
    bufB = torch.zeros(B.size + 1, dtype=torch.float32, device="cuda")
    bufA[1:] = _cu(A).reshape(-1)
    bufB[1:] = _cu(B).reshape(-1)
    At, Bt = bufA[1:].view(2000, 128), bufB[1:].view(2500, 128)
    assert At.data_ptr() % 16 == 4
    nm.set_engine(1) if 1 in _engines(nm) else None
    m = nm.match(At, Bt, 0.8).cpu().numpy()
    nm.set_engine(-1)
    assert np.array_equal(m, oracle.match(A, B, 0.8))


def test_batched_pair_matching_equals_per_pair_calls(nm):
    """nm_match_pairs_f32 (frame p -> p + 1 for a whole batch, all sizes on the device, tcgen05 engine) against one
    nm_match_f32 call (exact engine) per pair: match indices AND the (d1, i1, d2) records must be bitwise equal.
    Frames: planted true matches, counts that are not multiples of the 128-row tiles, a one-descriptor frame, an empty
    frame in the middle (both of its pairs stay unmatched), stale rows beyond the counts, a duplicated database row
    (min2 == 0: the entry keeps its previous value, match.cu:107), a frame matched against a copy of itself."""
    cap = 2048
    counts = [1500, 1337, 1, 0, 900, 2048, 700, 700]
    n = len(counts)
    rng = np.random.default_rng(11)
    desc = (rng.random((n, cap, 128)) * 300).astype(np.float32)          # rows beyond the counts: stale values, must be ignored
    prev = None
    for f, c in enumerate(counts):
        if c == 0:
            prev = None
            continue
        d = synth.descriptors(c, 100 + f, planted_from=prev) if prev is not None and len(prev) else synth.descriptors(c, 100 + f)
        desc[f, :c] = d
        prev = d
    desc[7, :700] = desc[6, :700]                                        # identical frames: d1 == 0 everywhere
    desc[5, 11] = desc[5, 10]; desc[4, 3] = desc[5, 10]                  # query 3 of frame 4: two database rows at distance 0
    dd, cc = _cu(desc), torch.tensor(counts, dtype=torch.int32, device="cuda")
    init = torch.full((n - 1, cap), 55, dtype=torch.int32, device="cuda")
    m, rec, fb = nm.match_pairs(dd, cc, 0.8, match_out=init.clone(), want_records=True)
    torch.cuda.synchronize()
    m, rec = m.cpu().numpy(), rec.cpu().numpy()
    nm.set_engine(0)
    try:
        for p in range(n - 1):
            nA, nB = counts[p], counts[p + 1]
            assert (m[p, nA:] == 55).all(), p                            # rows beyond the count untouched
            if nA == 0 or nB == 0:
                assert (m[p] == 55).all(), p
                continue
            ref = nm.match(dd[p, :nA], dd[p + 1, :nB], 0.8, match_io=init[p, :nA].clone()).cpu().numpy()
            r2 = nm.match_top2(dd[p, :nA], dd[p + 1, :nB]).cpu().numpy()
            assert np.array_equal(m[p, :nA], ref), (p, np.nonzero(m[p, :nA] != ref)[0][:10])
            assert np.array_equal(rec[p, :nA].view(np.uint32)[:, :3], r2.view(np.uint32)[:, :3]), p
    finally:
        nm.set_engine(-1)
    assert m[4, 3] == 55                                                 # min2 == 0: left as it was
    assert (m[0, :1500] >= 0).sum() > 150
    self_match = m[6, :700]                                              # identical frames: every row finds itself,
    assert (self_match == np.arange(700))[self_match != 55].all() and (self_match == 55).sum() <= 4   # bar duplicated rows (min2 == 0)
    assert int(fb.item()) < 200                                          # the exact fallback is the exception
