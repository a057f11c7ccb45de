"""Bring-up / timing of the tensor-core matcher engine against the exact fp32 engine (GPU box).
Usage: python tools/tc_bringup.py [big]"""
import ctypes as C
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import niftymatch_b200 as nm  # noqa: E402
from niftymatch_b200 import synth, _lib  # noqa: E402

lib = _lib.load()


def probe(A, B):
    rec = torch.empty((A.shape[0], 4), dtype=torch.float32, device="cuda")
    fb = C.c_int(-1)
    rc = lib.nm_match_tc_probe(C.c_void_p(A.data_ptr()), A.shape[0], C.c_void_p(B.data_ptr()), B.shape[0],
                               C.c_void_p(rec.data_ptr()), C.byref(fb), None, None, None, None,
                               C.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return rc, rec, fb.value


def accumulation_error(nA=3000, nB=7000):
    """max |S_tensor - S_exact| / (|a^|^2 + |b^|^2) over the candidates the scan kept."""
    Bh = synth.descriptors(nB, 12)
    Ah = synth.descriptors(nA, 11, planted_from=Bh)
    A, B = torch.from_numpy(Ah).cuda(), torch.from_numpy(Bh).cuda()
    rec = torch.empty((nA, 4), dtype=torch.float32, device="cuda")
    fb, nl, sc = C.c_int(-1), C.c_int(0), C.c_float(0)
    cs = np.zeros((8, nA, 4), np.float32)
    ci = np.zeros((8, nA, 4), np.int32)
    rc = lib.nm_match_tc_probe(C.c_void_p(A.data_ptr()), nA, C.c_void_p(B.data_ptr()), nB, C.c_void_p(rec.data_ptr()),
                               C.byref(fb), cs.ctypes.data_as(C.c_void_p), ci.ctypes.data_as(C.c_void_p), C.byref(nl),
                               C.byref(sc), C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, rc
    n = nl.value
    cs = cs.reshape(-1)[: n * nA * 4].reshape(n, nA, 4)
    ci = ci.reshape(-1)[: n * nA * 4].reshape(n, nA, 4)
    a16 = (Ah * sc.value).astype(np.float16).astype(np.float64)
    b16 = (Bh * sc.value).astype(np.float16).astype(np.float64)
    na2, nb2 = (a16 ** 2).sum(1), (b16 ** 2).sum(1)
    worst = 0.0
    for l in range(n):
        for k in range(4):
            idx = ci[l, :, k]
            ok = (idx >= 0) & (idx < nB)
            rows = np.nonzero(ok)[0]
            j = idx[ok]
            s_exact = (a16[rows] * b16[j]).sum(1) - 0.5 * nb2[j]
            err = np.abs(cs[l, rows, k].astype(np.float64) - s_exact) / (na2[rows] + nb2[j])
            worst = max(worst, float(err.max()))
    print(f"accumulation error: lists={n} scale={sc.value} max |dS|/(|a|^2+|b|^2) = {worst:.3e} = 2^{np.log2(worst):.1f}", flush=True)
    return worst


def check(nA, nB, seed=0):
    Bh = synth.descriptors(nB, 2 + seed)
    Ah = synth.descriptors(nA, 1 + seed, planted_from=Bh)
    A, B = torch.from_numpy(Ah).cuda(), torch.from_numpy(Bh).cuda()
    nm.set_engine(0)
    ref = nm.match_top2(A, B)
    torch.cuda.synchronize()
    rc, rec, fb = probe(A, B)
    same = torch.equal(rec.view(torch.int32), ref.view(torch.int32)) if rc == 0 else False
    bad = -1
    if rc == 0 and not same:
        bad = int((rec.view(torch.int32) != ref.view(torch.int32)).any(dim=1).sum().item())
    print(f"nA={nA} nB={nB}: rc={rc} fallback_rows={fb} records_equal={same} differing_rows={bad}", flush=True)
    if rc == 0 and not same and bad > 0:
        idx = (rec.view(torch.int32) != ref.view(torch.int32)).any(dim=1).nonzero()[:4, 0]
        for i in idx.tolist():
            print("   row", i, "tc", rec[i].tolist(), rec[i].view(torch.int32)[1].item(), "exact", ref[i].tolist(), ref[i].view(torch.int32)[1].item())
    nm.set_engine(-1)
    return same


def timeit(fn, n=5):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


if __name__ == "__main__":
    print("cc", lib.nm_device_cc())
    ok = True
    for nA, nB in [(256, 128), (256, 512), (300, 1000), (1, 1), (5, 3), (1000, 37), (2048, 2048), (4096, 8192), (20000, 30000)]:
        ok &= check(nA, nB)
    print("ALL EQUAL" if ok else "MISMATCH")
    accumulation_error()
    if ok and len(sys.argv) > 1:
        n = 100000
        Bh = synth.descriptors(n, 2)
        Ah = synth.descriptors(n, 1, planted_from=Bh)
        A, B = torch.from_numpy(Ah).cuda(), torch.from_numpy(Bh).cuda()
        nm.set_engine(1)
        m1 = nm.match(A, B, 0.8)
        ms = timeit(lambda: nm.match(A, B, 0.8))
        print(f"tc engine 100k x 100k: {ms:.3f} ms  {n * n / ms / 1e6:.1f} Gpairs/s  {n * n * 256 / ms / 1e9:.1f} TFLOP/s (256 flop/pair)")
        rc, rec, fb = probe(A, B)
        print("fallback rows at 100k x 100k:", fb)
        nm.set_engine(0)
        m0 = nm.match(A, B, 0.8)
        print("indices equal to exact engine:", torch.equal(m0, m1), "matched", int((m1 >= 0).sum()))
        nm.set_engine(-1)
