"""GPU: the tcgen05 3xTF32 GEMM (gemm_tf32x3.cu) against a float64 reference -- fp32-level accuracy
(1e-5 relative, an order tighter than the layer bar) at the layer's shapes, ragged edges included; strided operands
through the C-ABI, exact integer products, bit-identical results whatever the persistent grid, and the rank-counting
epilogue at ragged entity counts."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from relationprediction_b200 import _lib, ops
from relationprediction_b200.decoders.bilinear_diag import BilinearDiag
from conftest import ROOT
from test_gpu_rank import make_known, reference_ranks

pytestmark = pytest.mark.gpu


def rel(a, b):
    return float((a.double() - b).abs().max() / b.abs().max())


@pytest.mark.parametrize("M,N,K", [(128, 128, 32), (128, 128, 128), (256, 256, 64), (14541, 500, 500),
                                   (1000, 512, 512), (77, 8, 8), (300, 200, 200), (129, 132, 36),
                                   (5000, 24, 40),
                                   # many tiles per persistent CTA (one / two / sixteen k-blocks per tile)
                                   (100000, 512, 512), (40000, 132, 32), (30000, 24, 40)])
@pytest.mark.parametrize("b_is_nk", [False, True])
def test_gemm_tf32x3_matches_float64(M, N, K, b_is_nk):
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N)
    A = torch.randn(M, K, device="cuda", generator=g)
    B = torch.randn(*((N, K) if b_is_nk else (K, N)), device="cuda", generator=g)
    ref = A.double() @ (B.double().T if b_is_nk else B.double())
    C = ops.gemm_tf32x3(A, B, b_is_nk=b_is_nk)
    assert torch.isfinite(C).all()
    assert rel(C, ref) < 1e-5, rel(C, ref)
    # accumulate form
    C0 = torch.randn(M, N, device="cuda", generator=g)
    C1 = ops.gemm_tf32x3(A, B, b_is_nk=b_is_nk, out=C0.clone(), accumulate=True)
    assert rel(C1, ref + C0.double()) < 1e-5


def test_gemm_tf32x3_is_tighter_than_single_tf32_and_handles_scales():
    g = torch.Generator(device="cuda").manual_seed(1)
    A = torch.randn(2048, 512, device="cuda", generator=g) * 1e3
    B = torch.randn(512, 512, device="cuda", generator=g) * 1e-3
    ref = A.double() @ B.double()
    assert rel(ops.gemm_tf32x3(A, B), ref) < 1e-5


@pytest.mark.parametrize("K,M,N", [(128, 128, 128), (1000, 128, 128), (14541, 500, 500), (50000, 512, 512),
                                   (33, 8, 8), (4097, 132, 36), (3000, 2500, 500), (100, 200, 24)])
def test_gemm_tn_tf32x3_matches_float64(K, M, N):
    g = torch.Generator(device="cuda").manual_seed(K + M)
    A = torch.randn(K, M, device="cuda", generator=g)
    B = torch.randn(K, N, device="cuda", generator=g)
    ref = A.double().T @ B.double()
    C = ops.gemm_tn_tf32x3(A, B)
    assert torch.isfinite(C).all()
    assert rel(C, ref) < 1e-5, rel(C, ref)
    C0 = torch.randn(M, N, device="cuda", generator=g)
    C1 = ops.gemm_tn_tf32x3(A, B, out=C0.clone(), accumulate=True)
    assert rel(C1, ref + C0.double()) < 1e-5


def _p(t):
    return ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def padded(rows, cols, ld, fill, g):
    """A [rows, ld] buffer whose first `cols` columns are random and whose padding holds `fill`."""
    buf = torch.full((rows, ld), fill, device="cuda")
    buf[:, :cols] = torch.randn(rows, cols, device="cuda", generator=g)
    return buf


@pytest.mark.parametrize("b_is_nk", [False, True])
@pytest.mark.parametrize("accumulate", [False, True])
def test_nt_gemm_strided_operands_through_the_c_abi(b_is_nk, accumulate):
    """rgcn_gemm_tf32x3 with lda > K, ldb > K (or N) and ldc > N, as the basis layer calls it (lda = 2 d B): the
    NaN padding of A and B must never be read and the padding of C must come back bit for bit."""
    lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(11)
    M, N, K = 300, 132, 100                   # K is not a multiple of the 32-wide k-block
    lda, ldc = K + 32, N + 20
    ldb = K + 12 if b_is_nk else N + 8
    A = padded(M, K, lda, float("nan"), g)
    B = padded(N, K, ldb, float("nan"), g) if b_is_nk else padded(K, N, ldb, float("nan"), g)
    C = padded(M, N, ldc, 0.0, g)
    C[:, N:] = torch.randn(M, ldc - N, device="cuda", generator=g)
    C0 = C.clone()
    ws = torch.empty(2 * N * K, device="cuda")
    rc = lib.rgcn_gemm_tf32x3(_p(A), lda, _p(B), ldb, int(b_is_nk), _p(C), ldc, M, N, K, int(accumulate), _p(ws),
                              ws.numel() * 4, _stream())
    _lib.check(rc, "rgcn_gemm_tf32x3")
    torch.cuda.synchronize()
    Bd = B[:, :K].double() if b_is_nk else B[:, :N].double()
    ref = A[:, :K].double() @ (Bd.T if b_is_nk else Bd)
    if accumulate:
        ref = ref + C0[:, :N].double()
    assert torch.isfinite(C).all()
    assert rel(C[:, :N], ref) < 1e-5, rel(C[:, :N], ref)
    assert torch.equal(C[:, N:].view(torch.int32), C0[:, N:].view(torch.int32))


@pytest.mark.parametrize("accumulate", [False, True])
def test_tn_gemm_strided_operands_through_the_c_abi(accumulate):
    """rgcn_gemm_tn_tf32x3 with lda > M, ldb > N, ldc > N (the basis backward's dV = Agg^T G reads Agg with
    lda = 2 d B); split-K over 1000 rows."""
    lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(12)
    M, N, K = 256, 132, 1000
    lda, ldb, ldc = M + 8, N + 12, N + 4
    A = padded(K, M, lda, float("nan"), g)
    B = padded(K, N, ldb, float("nan"), g)
    C = torch.randn(M, ldc, device="cuda", generator=g)
    C0 = C.clone()
    rc = lib.rgcn_gemm_tn_tf32x3(_p(A), lda, _p(B), ldb, _p(C), ldc, M, N, K, int(accumulate), _stream())
    _lib.check(rc, "rgcn_gemm_tn_tf32x3")
    torch.cuda.synchronize()
    ref = A[:, :M].double().T @ B[:, :N].double()
    if accumulate:
        ref = ref + C0[:, :N].double()
    assert torch.isfinite(C).all()
    assert rel(C[:, :N], ref) < 1e-5, rel(C[:, :N], ref)
    assert torch.equal(C[:, N:].view(torch.int32), C0[:, N:].view(torch.int32))


# (M, N, K): 10 / 9 / 16 / 9 tiles of 128 x 128; one, two and sixteen 32-wide k-blocks against the 3-stage ring
GRID_SHAPES = [(640, 256, 32), (384, 384, 64), (1000, 132, 512), (300, 260, 544)]
GRIDS = ["1", "2", "3", "5", None, "64"]


@pytest.mark.parametrize("M,N,K", GRID_SHAPES)
@pytest.mark.parametrize("accumulate", [False, True])
def test_persistent_nt_gemm_is_bit_identical_for_every_grid(M, N, K, accumulate, monkeypatch):
    """Each tile is computed by one CTA in a fixed k order, so the number of persistent CTAs (RGCN_GEMM_CTAS, read
    on every launch) changes which CTA and which TMEM accumulator set / barrier phase a tile gets, never a bit."""
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    A = torch.randn(M, K, device="cuda", generator=g)
    B = torch.randn(K, N, device="cuda", generator=g)
    C0 = torch.randn(M, N, device="cuda", generator=g)
    results = []
    for ctas in GRIDS:
        if ctas is None:
            monkeypatch.delenv("RGCN_GEMM_CTAS", raising=False)
        else:
            monkeypatch.setenv("RGCN_GEMM_CTAS", ctas)
        results.append(ops.gemm_tf32x3(A, B, out=C0.clone(), accumulate=accumulate))
    ref = A.double() @ B.double() + (C0.double() if accumulate else 0)
    assert rel(results[0], ref) < 1e-5
    for ctas, C in zip(GRIDS[1:], results[1:]):
        assert torch.equal(C.view(torch.int32), results[0].view(torch.int32)), "grid %s differs from grid 1" % ctas


def test_rank_epilogue_is_identical_for_every_grid(monkeypatch):
    rng = np.random.RandomState(5)
    V, d, n = 1000, 64, 300                           # 3 x 8 tiles
    codes = rng.normal(0, 0.3, (V, d)).astype(np.float32)
    relt = rng.normal(0, 1, (V, d)).astype(np.float32)
    X = np.stack([rng.randint(0, V, n), rng.randint(0, V, n), rng.randint(0, V, n)], 1).astype(np.int32)
    mask = torch.as_tensor(BilinearDiag.known_bit_mask(make_known(rng, X, V, 1), V), device="cuda")
    ranker = ops.DistMultRanker(torch.as_tensor(codes, device="cuda"), torch.as_tensor(relt, device="cuda"))
    Xt = torch.as_tensor(X, device="cuda")
    out = []
    for ctas in GRIDS:
        if ctas is None:
            monkeypatch.delenv("RGCN_GEMM_CTAS", raising=False)
        else:
            monkeypatch.setenv("RGCN_GEMM_CTAS", ctas)
        raw, filt = ranker.rank(Xt, 1, mask)
        out.append((raw.cpu().numpy(), filt.cpu().numpy()))
    for ctas, (raw, filt) in zip(GRIDS[1:], out[1:]):
        np.testing.assert_array_equal(raw, out[0][0], err_msg="raw ranks, grid %s" % ctas)
        np.testing.assert_array_equal(filt, out[0][1], err_msg="filtered ranks, grid %s" % ctas)


@pytest.mark.parametrize("amax,bmax,K", [(2 ** 20, 3, 4), (2 ** 18, 15, 4), (2 ** 18, 3, 16), (2 ** 14, 15, 64)])
def test_integer_products_are_exact(amax, bmax, K):
    """|A| < amax needs both the hi and the lo part of the split (more than 11 significant bits), B is exact in
    TF32, and K |A| |B| < 2^24 keeps every partial sum an exact fp32 integer: C must EQUAL the float64 product.  A
    dropped or doubled MMA, or a wrong hi/lo split, changes the result by at least 1."""
    assert K * (amax - 1) * bmax < 2 ** 24
    g = torch.Generator(device="cuda").manual_seed(amax + K)
    M, N = 300, 132
    A = torch.randint(-amax + 1, amax, (M, K), device="cuda", generator=g).float()
    B = torch.randint(-bmax, bmax + 1, (K, N), device="cuda", generator=g).float()
    ref = A.double() @ B.double()
    for b_is_nk in (False, True):
        C = ops.gemm_tf32x3(A, B.T.contiguous() if b_is_nk else B, b_is_nk=b_is_nk)
        assert torch.equal(C.double(), ref), float((C.double() - ref).abs().max())
    At = torch.randint(-amax + 1, amax, (K, 256), device="cuda", generator=g).float()
    Bt = torch.randint(-bmax, bmax + 1, (K, N), device="cuda", generator=g).float()
    C = ops.gemm_tn_tf32x3(At, Bt)
    assert torch.equal(C.double(), At.double().T @ Bt.double())


@pytest.mark.parametrize("K", [4, 8, 12, 28, 36])
@pytest.mark.parametrize("N", [4, 132])
@pytest.mark.parametrize("b_is_nk", [False, True])
def test_single_row_and_short_contractions(K, N, b_is_nk):
    g = torch.Generator(device="cuda").manual_seed(K * 1000 + N)
    A = torch.randn(1, K, device="cuda", generator=g)
    B = torch.randn(*((N, K) if b_is_nk else (K, N)), device="cuda", generator=g)
    ref = A.double() @ (B.double().T if b_is_nk else B.double())
    C = ops.gemm_tf32x3(A, B, b_is_nk=b_is_nk)
    assert C.shape == (1, N) and torch.isfinite(C).all()
    assert rel(C, ref) < 1e-5, rel(C, ref)


@pytest.mark.parametrize("V", [1025, 1023, 129, 159])
@pytest.mark.parametrize("ctas", ["1", None])
def test_rank_epilogue_ragged_entity_count(V, ctas, monkeypatch):
    """V % 32 in {1, 31}: the last 32-column chunk of the known mask is partial.  Some gold entities sit in that
    chunk, and every bit PAST V in the last mask word is set: those columns do not exist and must not count."""
    if ctas is not None:
        monkeypatch.setenv("RGCN_GEMM_CTAS", ctas)
    rng = np.random.RandomState(V)
    d, n = 64, 200
    codes = (rng.randint(-1, 2, (V, d)) * (rng.uniform(size=(V, d)) < 0.05)).astype(np.float32)
    relt = rng.randint(-1, 2, (V, d)).astype(np.float32)
    X = np.stack([rng.randint(0, V, n), rng.randint(0, V, n), rng.randint(0, V, n)], 1).astype(np.int32)
    last = (V // 32) * 32
    X[::3, 2] = rng.randint(last, V, len(X[::3]))       # gold objects in the last, partial chunk
    X[::7, 2] = V - 1
    ranker = ops.DistMultRanker(torch.as_tensor(codes, device="cuda"), torch.as_tensor(relt, device="cuda"))
    known = make_known(rng, X, V, 1)
    mask = BilinearDiag.known_bit_mask(known, V).view(np.uint32).copy()
    if V % 32:
        mask[:, -1] |= np.uint32((0xFFFFFFFF << (V % 32)) & 0xFFFFFFFF)   # stray bits past V
    raw, filt = ranker.rank(torch.as_tensor(X, device="cuda"), 1, torch.as_tensor(mask.view(np.int32), device="cuda"))
    ref_raw, ref_filt = reference_ranks(codes, relt, X, 1, known, sigmoid=False)
    np.testing.assert_array_equal(raw.cpu().numpy(), ref_raw)
    np.testing.assert_array_equal(filt.cpu().numpy(), ref_filt)


def test_tn_gemm_with_prefetch_distance_2_in_a_child_process():
    """k_gemm_tn_tf32x3<2> runs only with RGCN_GEMM_PF=2, which the library reads once per process: a child process
    runs one TN product with it under torch.profiler and reports the kernel it saw and the error against float64."""
    code = r"""
import json, sys
sys.path[:0] = [%r, %r]
import torch
from relationprediction_b200 import ops
from test_gpu_kernel_matrix import traced_kernels
g = torch.Generator(device="cuda").manual_seed(7)
A = torch.randn(4097, 132, device="cuda", generator=g)
B = torch.randn(4097, 36, device="cuda", generator=g)
C, names = traced_kernels(lambda: ops.gemm_tn_tf32x3(A, B))
ref = A.double().T @ B.double()
err = float((C.double() - ref).abs().max() / ref.abs().max())
print(json.dumps({"names": sorted(names), "err": err, "finite": bool(torch.isfinite(C).all())}))
""" % (ROOT, os.path.join(ROOT, "tests"))
    env = dict(os.environ, RGCN_GEMM_PF="2")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code]
    res = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    out = json.loads(res.stdout.strip().splitlines()[-1])
    assert "k_gemm_tn_tf32x3<2>" in out["names"] and "k_gemm_tn_tf32x3<3>" not in out["names"], out["names"]
    assert out["finite"] and out["err"] < 1e-5, out
