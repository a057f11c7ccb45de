"""Float64 restatement of the tensor-core matcher's certificate (niftymatch_b200/csrc/nm_match_tc.cu) and the input
families it is measured on.  Test infrastructure only.

The scan keeps the 4 best fp16 tensor-core scores S = a^.b^ - |b^|^2/2 per row and list (a^ = fp16(s a),
b^ = fp16(s b), s the power-of-two scale); the re-rank trusts that every accumulated score is within eta/2 of the exact
one, eta = 2^-17 (|a^|^2 + |b^|^2max) + 2^-16.  `certificate_ratios` measures both halves of that assumption against
S computed here in float64 from the same fp16 operands:
  (a) soundness: a column in none of the row's lists has S_exact <= thr + eta/2, thr = max over lists of the 4th-best
      score -- otherwise the scan dropped a column that could be nearer than the certified second distance;
  (b) accuracy: every candidate's score is within eta/2 of S_exact."""
from __future__ import annotations

import numpy as np

from niftymatch_b200 import synth

F16_MIN_NORMAL = 2.0 ** -14


def tc_scale(A, B):
    """tc_scale_from_max: max |x| over A and B = f 2^e, f in [0.5, 1)  ->  s = 2^(8 - e), scaled values in [128, 256)."""
    mx = float(max(np.abs(A).max(initial=0.0), np.abs(B).max(initial=0.0)))
    if not mx > 0.0:
        return 1.0
    _, e = np.frexp(np.float32(mx))
    return float(2.0 ** min(max(8 - int(e), -100), 100))


def fp16_scaled(X, s):
    """fp16(s x) as float64 (numpy's float32 -> float16 conversion rounds to nearest even, as __float2half_rn)."""
    return (X.astype(np.float32) * np.float32(s)).astype(np.float16).astype(np.float64)


def seed_tiles(nB):
    """tc_run's seed pass: database tiles (128 rows) scanned first, 0 below 32 tiles, else clamp(tiles / 16, 4, 16)."""
    t = (nB + 127) // 128
    return 0 if t < 32 else min(max(t // 16, 4), 16)


def tc_splits(nA, nB, n_sms):
    """tc_pick_splits over the main scan's tiles: the candidate lists are 2 per split."""
    rowblocks, tiles = (nA + 255) // 256, (nB + 127) // 128 - seed_tiles(nB)
    best, best_eff = 1, -1.0
    for s in range(1, max(1, min(tiles // 2, 4)) + 1):
        per = -(-tiles // s)
        if -(-tiles // per) != s:
            continue
        units = rowblocks * s
        waves = -(-units // n_sms)
        eff = units / (waves * n_sms) + (1e-3 if s >= 2 else 0.0)
        if eff > best_eff + 1e-9:
            best, best_eff = s, eff
    return best


def certificate_ratios(A, B, probe, block=1024):
    """Worst ratios of the two halves of the certificate's assumption over all rows of a probe (nm.tc_probe(...,
    want_candidates=True)).  Returns a dict:
      sound   max over rows and non-candidate columns j < nB of (S_exact - thr) / (eta / 2); <= 1 is sound
      cand    max over candidates j < nB of |score - S_exact| / (eta / 2); <= 1 is within the budget
      cand_rel max over candidates of |score - S_exact| / (|a^|^2 + |b^_j|^2), the figure DESIGN.md 4.3 quotes
      cand_col max over candidates of |score - S_exact| / (2^-18 (|a^|^2 + |b^_j|^2) + 2^-17): eta / 2 with the
               column's own norm in place of the database maximum, which a large row elsewhere would inflate."""
    nA, nB = len(A), len(B)
    s = probe["scale"]
    assert s == tc_scale(A, B), (s, tc_scale(A, B))
    a16, b16 = fp16_scaled(A, s), fp16_scaled(B, s)
    na2, nb2 = (a16 ** 2).sum(1), (b16 ** 2).sum(1)
    bmax2 = float((B.astype(np.float64) ** 2).sum(1).max()) * s * s * (1.0 + 2.0 ** -9)
    eta_half = 0.5 * (np.ldexp(na2 + bmax2, -17) + 2.0 ** -16)
    cs = probe["cand_scores"].astype(np.float64)             # [lists][nA][4]
    ci = probe["cand_index"]
    thr = cs[:, :, 3].max(0)
    sound, cand, cand_rel, cand_col = -np.inf, 0.0, 0.0, 0.0
    for r0 in range(0, nA, block):
        r1 = min(nA, r0 + block)
        S = a16[r0:r1] @ b16.T - 0.5 * nb2[None, :]
        rows = np.arange(r1 - r0)
        picked = []
        for l in range(ci.shape[0]):
            for k in range(4):
                j = ci[l, r0:r1, k]
                ok = (j >= 0) & (j < nB)
                rr, jj = rows[ok], j[ok]
                picked.append((rr, jj))
                if len(rr):
                    err = np.abs(cs[l, r0:r1, k][ok] - S[rr, jj])
                    cand = max(cand, float((err / eta_half[r0 + rr]).max()))
                    nsum = na2[r0 + rr] + nb2[jj]
                    cand_rel = max(cand_rel, float((err / nsum).max()))
                    cand_col = max(cand_col, float((err / (np.ldexp(nsum, -18) + 2.0 ** -17)).max()))
        for rr, jj in picked:                                 # candidates (the seed's are in every list) leave the
            S[rr, jj] = -np.inf                               # soundness check
        sound = max(sound, float(((S.max(1) - thr[r0:r1]) / eta_half[r0:r1]).max()))
    return {"sound": sound, "cand": cand, "cand_rel": cand_rel, "cand_col": cand_col}


def log2_str(x):
    return f"2^{np.log2(x):.2f}" if x > 0 else f"{x:.3g} (<= 0)"


# ---- input families ----------------------------------------------------------------------------------------------
def fam_synth():
    """The benchmark's descriptor statistics (synth.descriptors), 20 % of the queries planted."""
    B = synth.descriptors(7000, 12)
    return synth.descriptors(3000, 11, planted_from=B), B


def fam_sift(nm, torch):
    """Real SIFT descriptors: two overlapping 1920x1080 crops of one synth.scene, frame 0 against frame 1."""
    w, h = 1920, 1080
    base = synth.scene(w + 48, h + 32, synth.SEED_BASE + 5)
    frames = np.stack([base[0:h, 0:w], base[23:23 + h, 37:37 + w]])
    P = nm.SiftParams(w, h)
    P._peak_threshold = 2.0
    sb = nm.SiftBatch(P, 2, 16384)
    try:
        sb.run(torch.from_numpy(np.ascontiguousarray(frames)).cuda())
        torch.cuda.synchronize()
        r = sb.results()
        n0, n1 = int(r["counts"][0].item()), int(r["counts"][1].item())
        A = r["desc"][0, :n0].cpu().numpy().copy()
        B = r["desc"][1, :n1].cpu().numpy().copy()
    finally:
        sb.close()
    assert min(n0, n1) > 1000, (n0, n1)
    return A, B


def _odd_mantissas(rng, shape):
    """fp16 mantissas 1 + m/1024 with m odd: every product keeps low bits that an aligned or truncated sum drops."""
    return 1.0 + (2 * rng.integers(0, 512, shape) + 1) / 1024.0


def fam_coherent(nA=256, nB=32, seed=1):
    """Per 16-element k block one dominant product plus fifteen products 2^-10 .. 2^-22 of it, odd low bits, all of one
    sign: the errors of aligning or truncating the small products add up instead of cancelling.  The dominant
    operands are near 200 (scale 1); the small ones split the exponent between query and database, so that both stay
    normal fp16 numbers."""
    rng = np.random.default_rng(seed)

    def rows(n, side):
        X = np.empty((n, 128))
        for blk in range(8):
            X[:, 16 * blk] = 128.0 * _odd_mantissas(rng, n)
            for k in range(1, 16):
                e = min(9 + k, 22)                                   # product 2^-e of the dominant one, e = 10 .. 22
                ea = (e + 1) // 2 if side == 0 else e // 2
                X[:, 16 * blk + k] = 128.0 * 2.0 ** -ea * _odd_mantissas(rng, n)
        return X.astype(np.float16).astype(np.float32)

    return rows(nA, 0), rows(nB, 1)


def fam_near_equal(nA=256, nB=32, seed=2):
    """a ~ b: queries are database rows plus noise near the fp16 resolution, or database rows halved (a^.b^ =
    |b^|^2/2 exactly, so S = 0 while the fp16 part of the sum reaches |b^|^2/2 and the norm slab cancels it)."""
    rng = np.random.default_rng(seed)
    B = (128.0 + 127.0 * rng.random((nB, 128))).astype(np.float32)
    src = rng.integers(0, nB, nA)
    A = B[src].astype(np.float64)
    half = np.arange(nA) % 2 == 1
    A[half] *= 0.5
    A[~half] += rng.normal(0.0, 0.1, (int((~half).sum()), 128))
    return A.astype(np.float32), B


def fam_equal_components(nA=256, nB=32, seed=3):
    """All-equal components: every product of a row pair is the same number, so rounding errors are all alike."""
    rng = np.random.default_rng(seed)
    va = (128.0 * _odd_mantissas(rng, nA)).astype(np.float16).astype(np.float32)
    vb = (128.0 * _odd_mantissas(rng, nB)).astype(np.float16).astype(np.float32)
    vb[0] = 255.875
    return np.repeat(va[:, None], 128, 1), np.repeat(vb[:, None], 128, 1)


def fam_mixed_signs(nA=256, nB=32, seed=4):
    """Mixed signs: large products of alternating sign, so the dot product is a small difference of large partial
    sums; queries are database rows with some signs flipped."""
    rng = np.random.default_rng(seed)
    sign = np.where(np.arange(128) % 2 == 0, 1.0, -1.0)
    B = (sign * (128.0 + 127.0 * rng.random((nB, 128)))).astype(np.float32)
    A = B[rng.integers(0, nB, nA)].astype(np.float64)
    flip = rng.random(A.shape) < 0.5
    A[flip] *= -1.0
    return A.astype(np.float32), B


def fam_tiny_tail(nA=256, nB=32, seed=5):
    """One database row sets the scale at 255; every other row is 2^-8 .. 2^-14 below it, so that after scaling the
    rows and their norm slab reach the fp16 subnormal range (the absolute 2^-16 of eta)."""
    rng = np.random.default_rng(seed)
    e = rng.integers(8, 15, nB)
    B = 255.0 * 2.0 ** -e[:, None] * rng.random((nB, 128))
    B[0] = 0.0
    B[0, 0] = 255.0
    eA = rng.integers(8, 15, nA)
    A = B[rng.integers(1, nB, nA)] + 255.0 * 2.0 ** -eA[:, None] * rng.normal(0.0, 0.05, (nA, 128))
    return A.astype(np.float32), B.astype(np.float32)


ADVERSARIAL = {"coherent": fam_coherent, "near_equal": fam_near_equal, "equal_components": fam_equal_components,
               "mixed_signs": fam_mixed_signs, "tiny_tail": fam_tiny_tail}


def family(name, nm=None, torch=None):
    if name == "synth":
        return fam_synth()
    if name == "sift":
        return fam_sift(nm, torch)
    return ADVERSARIAL[name]()


FAMILIES = ["synth", "sift"] + list(ADVERSARIAL)
