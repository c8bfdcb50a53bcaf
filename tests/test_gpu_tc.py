"""GPU tests of the tcgen05 (tensor-core) decoder-output kernel: operand-view self-tests against
float64 matmuls, then the fused training / scoring kernels against the exact-fp32 CUDA-core kernel."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _selftest(mode, A, Bm, dshape, split):
    from aaerec_b200 import _native as N
    D = torch.full(dshape, float("nan"), device="cuda")
    N.call("aae_tc_selftest", mode, N.ptr(A), N.ptr(Bm), N.ptr(D), split, None)
    torch.cuda.synchronize()
    return D.cpu().double()


@pytest.mark.parametrize("split,tol", [(3, 3e-6), (1, 3e-3)])
def test_tc_operand_views(split, tol):
    g = torch.Generator().manual_seed(0)
    # mode 1: K-major A [128,104], K-major B [32,104]
    A = torch.randn(128, 104, generator=g)
    Bm = torch.randn(32, 104, generator=g)
    D = _selftest(1, A.cuda(), Bm.cuda(), (128, 32), split)
    want = A.double() @ Bm.double().t()
    assert (D - want).abs().max() / want.abs().max() < tol
    # mode 2 (G2 form): A [128,32] from TMEM, B [112,32] K-major in smem with padded strides
    A = torch.randn(128, 32, generator=g)
    Bm = torch.randn(112, 32, generator=g)
    D = _selftest(2, A.cuda(), Bm.cuda(), (128, 112), split)
    want = A.double() @ Bm.double().t()
    assert (D - want).abs().max() / want.abs().max() < tol
    # mode 3 (G3 form): A [128,128] from TMEM, B [32,128] K-major in smem with padded strides
    A = torch.randn(128, 128, generator=g)
    Bm = torch.randn(32, 128, generator=g)
    D = _selftest(3, A.cuda(), Bm.cuda(), (128, 32), split)
    want = A.double() @ Bm.double().t()
    assert (D - want).abs().max() / want.abs().max() < tol


def _run_train(impl, B, V, H=100, seed=0, steps=2, wscale=0.1, bshift=0.0):
    from aaerec_b200 import _native as N
    from aaerec_b200.synth import synth_sets
    g = torch.Generator().manual_seed(seed)
    dev = "cuda"
    W = ((torch.rand(V, H, generator=g) * 2 - 1) * wscale).to(dev)
    b = (torch.rand(V, generator=g) * 0.2 - 0.1 + bshift).to(dev)
    mW, vW = torch.zeros_like(W), torch.zeros_like(W)
    mb, vb = torch.zeros_like(b), torch.zeros_like(b)
    X = synth_sets(B, V, 9, seed=seed + 1)
    ip = torch.as_tensor(X.indptr.astype(np.int32), device=dev)
    ii = torch.as_tensor(X.indices.astype(np.int32), device=dev)
    state = torch.zeros(48, dtype=torch.uint8, device=dev)
    N.call("aae_step_state_init", N.ptr(state), 1e-3, 1e-3, 0, None)
    out = []
    for s in range(steps):
        h2 = torch.relu(torch.randn(B, H, generator=g)).to(dev) * (1.0 + s)
        dh2 = torch.zeros(B, H, device=dev)
        loss = torch.zeros(1, dtype=torch.float64, device=dev)
        N.call("aae_step_tick", N.ptr(state), None)
        N.call("aae_dec_out_train", N.ptr(h2), B, H, N.ptr(W), N.ptr(b), N.ptr(mW), N.ptr(vW), N.ptr(mb), N.ptr(vb),
               0, V, N.ptr(ip), N.ptr(ii), float(B) * V, N.ptr(state), N.ptr(dh2), N.ptr(loss), impl, None)
        torch.cuda.synchronize()
        out.append((loss.item(), dh2.cpu().double()))
    return out, W.cpu().double(), b.cpu().double(), mW.cpu().double(), vW.cpu().double()


def _rel(a, b):
    return float((a - b).norm() / b.norm())


@pytest.mark.parametrize("B,V", [(100, 3200), (128, 1000), (37, 777), (1, 64), (100, 20000)])
def test_tc_train_matches_fp32_kernel(B, V):
    ref, Wr, br, mr, vr = _run_train(0, B, V)
    got, Wg, bg, mg, vg = _run_train(1, B, V)
    for (lr, dr), (lg, dg) in zip(ref, got):
        assert abs(lg - lr) / abs(lr) < 2e-6
        assert _rel(dg, dr) < 2e-5
    assert _rel(Wg, Wr) < 2e-6 and _rel(bg, br) < 2e-6
    assert _rel(mg, mr) < 2e-5 and _rel(vg, vr) < 4e-5


@pytest.mark.parametrize("B,V,H,impl", [(100, 3200, 100, 3), (100, 40000, 100, 1), (64, 5000, 64, 1), (50, 3000, 116, 1),
                                        (104, 9000, 100, 1), (100, 4733, 100, 1)])
def test_tc_train_variants_match_fp32_kernel(B, V, H, impl):
    """impl 3 = the one-tile-at-a-time kernel; impl 1 = pipelined kernel (compile-time and run-time n_hidden,
    many tiles per CTA, ragged last tile) or its fallback when the shape is outside the pipelined envelope."""
    ref, Wr, br, mr, vr = _run_train(0, B, V, H=H, steps=3)
    got, Wg, bg, mg, vg = _run_train(impl, B, V, H=H, steps=3)
    for (lr, dr), (lg, dg) in zip(ref, got):
        assert abs(lg - lr) / abs(lr) < 2e-6
        assert _rel(dg, dr) < 2e-5
    assert _rel(Wg, Wr) < 2e-6 and _rel(bg, br) < 2e-6
    assert _rel(mg, mr) < 2e-5 and _rel(vg, vr) < 4e-5


@pytest.mark.parametrize("wscale,bshift", [(0.5, 0.0), (0.4, -14.0), (0.15, -22.0)])
def test_tc_train_wide_logits_match_fp32_kernel(wscale, bshift):
    """Logits far outside (-16, 16): deep-negative values (everyday a few dozen steps into training; they stay on the
    tensor-core kernel's fast paths), values >= 16 and positives (ATen's clamped edge formulas, per element)."""
    B, V = 100, 6400
    ref, Wr, br, mr, vr = _run_train(0, B, V, steps=2, wscale=wscale, bshift=bshift)
    got, Wg, bg, mg, vg = _run_train(1, B, V, steps=2, wscale=wscale, bshift=bshift)
    for (lr, dr), (lg, dg) in zip(ref, got):
        assert abs(lg - lr) / abs(lr) < 5e-6
        assert _rel(dg, dr) < 2e-5
    assert _rel(Wg, Wr) < 2e-6 and _rel(bg, br) < 2e-6
    assert _rel(mg, mr) < 2e-5 and _rel(vg, vr) < 4e-5


def test_tc_single_tf32_is_close_but_not_parity():
    ref, Wr, *_ = _run_train(0, 100, 3200)
    got, Wg, *_ = _run_train(2, 100, 3200)
    assert abs(got[0][0] - ref[0][0]) / ref[0][0] < 1e-3
    assert _rel(got[0][1], ref[0][1]) < 5e-3


@pytest.mark.parametrize("B,V", [(100, 3200), (300, 1000), (5, 77)])
def test_tc_scores_match_fp32_kernel(B, V):
    from aaerec_b200 import _native as N
    H = 100
    g = torch.Generator().manual_seed(3)
    W = (torch.rand(V, H, generator=g) - 0.5).cuda()
    b = (torch.rand(V, generator=g) - 0.5).cuda()
    h2 = torch.relu(torch.randn(B, H, generator=g)).cuda()
    outs = []
    for impl in (0, 1, 3):
        o = torch.zeros(B, V, device="cuda")
        N.call("aae_dec_out_scores", N.ptr(h2), B, H, N.ptr(W), N.ptr(b), V, 0, N.ptr(o), V, impl, None)
        torch.cuda.synchronize()
        outs.append(o.cpu().double())
    want = h2.cpu().double() @ W.cpu().double().t() + b.cpu().double()
    assert (outs[0] - want).abs().max() < 2e-5
    assert (outs[1] - want).abs().max() < 2e-5
    assert torch.equal(outs[2], outs[1])   # impl 3 scores as impl 1
