"""GPU: the tcgen05 GEMM with the split A operand in tensor memory (default) vs the shared-memory operand path
(D3F_TC_A_SMEM=1). Both paths issue the same MMAs in the same order into the same accumulator rotation, so their
outputs are bit-identical -- except in tc_gemm_kernel<64,2,0>, which rotates over 2 accumulators instead of 4 with A
in TMEM and is held to float64 instead.

Which instantiation a shape reaches (tc_gemm.cu, launch_tc): BN = 32 / 64 / 128 from N (64 for N > 64 when K <= 256
and M >= 8192); one stage and one accumulator for <= 4 k-chunks on > 592 output tiles (BN <= 64); two stages for
<= 4 k-chunks or, at BN <= 64, > 148 output tiles; otherwise the deep ring (3 stages at BN = 128, else 4)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def both_paths(monkeypatch, fn):
    monkeypatch.setenv("D3F_TC_A_SMEM", "0")
    new = fn()
    monkeypatch.setenv("D3F_TC_A_SMEM", "1")
    old = fn()
    monkeypatch.setenv("D3F_TC_A_SMEM", "0")
    return new, old


@pytest.fixture
def co(cuda, monkeypatch):
    from d3feat_b200 import convolution_ops
    monkeypatch.setattr(convolution_ops, "USE_TENSOR_CORES", True)
    monkeypatch.setenv("D3F_TC_STREAM", "0")
    return convolution_ops


@pytest.mark.parametrize("K", [32, 64])
def test_tmem_operand_layout_identity_and_permutation(cuda, co, monkeypatch, K):
    """One 128-row tile, X @ I and X @ P (P a column permutation), so that a wrong TMEM layout of A (lane = row,
    column = k) shows up as a wrong element. With X exact in TF32 (11 significant bits: lo = 0) the product is exact
    and checks the hi columns. For general X the tensor core reads lo as TF32 too, so X @ I = hi + tf32(lo) is within
    2^-21 |x| of x, while a misplaced lo column would be off by ~2^-12 |x|."""
    rng = np.random.default_rng(K)
    perm = rng.permutation(K)
    p = np.zeros((K, K), np.float32)
    p[perm, np.arange(K)] = 1.0
    eye, tp = t(np.eye(K, dtype=np.float32), cuda), t(p, cuda)
    x = (np.round(rng.normal(size=(128, K)) * 256) / 256).astype(np.float32)
    tx = t(x, cuda)
    assert np.array_equal(co.unary_convolution(tx, eye).cpu().numpy(), x)
    assert np.array_equal(co.unary_convolution(tx, tp).cpu().numpy(), x[:, perm])
    x = rng.normal(size=(128, K)).astype(np.float32)
    tx = t(x, cuda)
    for w, ref in ((eye, x), (tp, x[:, perm])):
        out = co.unary_convolution(tx, w).cpu().numpy()
        assert np.all(np.abs(out.astype(np.float64) - ref) <= 2.0 ** -21 * np.abs(ref))


# (M, K, N, instantiation): every <BN, STAGES, ACC> with row tails (M % 128 != 0) and K tails (K % 32 != 0)
SAME_ROTATION = [
    (80001, 64, 32, "<32,1,1>"), (80001, 100, 32, "<32,1,1> K tail"),
    (40003, 128, 128, "<64,1,1>"), (80001, 36, 64, "<64,1,1> K tail"),
    (20001, 480, 32, "<32,2,0>"), (30001, 68, 32, "<32,2,0> K tail"),
    (1001, 128, 256, "<128,2,0>"), (999, 100, 200, "<128,2,0> K tail"),
    (1001, 512, 256, "<128,3,0>"), (777, 1000, 300, "<128,3,0> K tail"),
    (1001, 480, 32, "<32,4,0>"), (1001, 452, 20, "<32,4,0> K tail"),
    (1001, 960, 64, "<64,4,0>"), (3333, 196, 48, "<64,4,0> K tail"),
]


@pytest.mark.parametrize("M,K,N,variant", SAME_ROTATION)
def test_tmem_operand_bit_identical(cuda, co, monkeypatch, M, K, N, variant):
    rng = np.random.default_rng(M + K + N)
    x = t(rng.normal(size=(M, K)).astype(np.float32), cuda)
    w = t((rng.normal(size=(K, N)) / np.sqrt(K)).astype(np.float32), cuda)
    scale = t(rng.uniform(0.5, 1.5, N).astype(np.float32), cuda)
    shift = t(rng.normal(size=N).astype(np.float32), cuda)
    res = t(rng.normal(size=(M, N)).astype(np.float32), cuda)
    new, old = both_paths(monkeypatch, lambda: co.unary_convolution(x, w))
    assert torch.equal(new, old), variant
    new, old = both_paths(monkeypatch, lambda: co.unary_convolution(x, w, epilogue=(scale, shift, 0.2), residual=res))
    assert torch.equal(new, old), variant
    # device-side row count below the launch capacity: the rows past it are not written by either path
    rows = torch.tensor([M - 300], dtype=torch.int32, device=cuda)
    new, old = both_paths(monkeypatch, lambda: co.unary_convolution(x, w, rows=rows)[: M - 300])
    assert torch.equal(new, old), variant


@pytest.mark.parametrize("M,K", [(20001, 960), (20001, 2048)])
def test_tmem_operand_two_accumulators_vs_float64(cuda, co, monkeypatch, M, K):
    """<64,2,0> with A in TMEM rotates over 2 accumulators (4 with A in shared memory): all-positive data, where the
    tensor pipe's truncating accumulate biases every partial sum the same way (~1.1e-8 K / kAcc relative)."""
    rng = np.random.default_rng(K)
    x = rng.uniform(0, 1, size=(M, K)).astype(np.float32)
    w = rng.uniform(0, 1, size=(K, 64)).astype(np.float32)
    ref = x.astype(np.float64) @ w.astype(np.float64)
    new, old = both_paths(monkeypatch, lambda: co.unary_convolution(t(x, cuda), t(w, cuda)).cpu().numpy())
    for out in (new, old):
        assert np.abs(out - ref).max() <= 3e-5 * np.abs(ref).max()


@pytest.mark.parametrize("N,C1,C2,Cout", [(5000, 32, 64, 128), (3001, 64, 128, 256), (700, 512, 1024, 2048),
                                          (60001, 32, 64, 32)])
def test_tmem_operand_pair_gemm(cuda, co, monkeypatch, N, C1, C2, Cout):
    """[x1 | x2] along K: the k-chunks switch source matrix at C1."""
    rng = np.random.default_rng(N + C1)
    x1, x2 = (t(rng.normal(size=(N, c)).astype(np.float32), cuda) for c in (C1, C2))
    w1, w2 = (t((rng.normal(size=(c, Cout)) / np.sqrt(c)).astype(np.float32), cuda) for c in (C1, C2))
    a1, a2 = ((t(rng.uniform(0.5, 1.5, Cout).astype(np.float32), cuda), t(rng.normal(size=Cout).astype(np.float32), cuda))
              for _ in range(2))
    new, old = both_paths(monkeypatch, lambda: co.unary_pair_convolution(x1, w1, a1, x2, w2, a2, 0.2))
    assert torch.equal(new, old)


@pytest.mark.parametrize("Cin,Cout,Nq", [(256, 256, 300), (512, 512, 150), (128, 128, 700), (64, 32, 2500)])
def test_tmem_operand_kpconv_split_k_and_row_map(cuda, co, monkeypatch, Cin, Cout, Nq):
    """KPConv contractions: split-K for the small deep layers (< 96 output tiles, >= 16 k-chunks), and the
    row map of a permuted query order (the epilogue scatters the rows back)."""
    rng = np.random.default_rng(Cin + Nq)
    q = rng.uniform(0, 0.2, (Nq, 3)).astype(np.float32)     # dense: most neighbours inside the extent
    H = 24
    idx = rng.integers(0, Nq + 1, (Nq, H)).astype(np.int32)      # index Nq: the shadow neighbour
    f = rng.normal(size=(Nq, Cin)).astype(np.float32)
    Kp = rng.normal(size=(15, 3)).astype(np.float32) * 0.05
    W = (rng.normal(size=(15, Cin, Cout)) * np.sqrt(2.0 / Cout)).astype(np.float32)
    args = [t(a, cuda) for a in (q, q, idx, f, Kp, W)]
    perm = t(rng.permutation(Nq).astype(np.int32), cuda)
    for order in (None, perm):
        new, old = both_paths(monkeypatch, lambda: co.KPConv_ops(*args, 0.1, "linear", "sum", query_order=order))
        assert torch.equal(new, old)
