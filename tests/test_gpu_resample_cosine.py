"""GPU (-m gpu): the fused resample2d -> cosine-similarity op (SURVEY row f4; external_function.py:275-279) and the
``PerceptualCorrectness`` loss built on it.

Oracles:
  * the CPU oracle's resample2d (forward and backward) composed with the cosine in numpy (float64 chain rule written out below);
  * the UNFUSED composition on the GPU: ``F.cosine_similarity(gfla_b200.Resample2d(...)(x, flow), target)`` with torch autograd;
  * the loss and flow gradients the reference's own ``PerceptualCorrectness`` class computed with the same feature extractor
    (tests/golden/reference_perceptual.npz).
Tolerances: fp32 1e-5 relative to the largest magnitude of the compared tensor, fp64 1e-11.
"""

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
EPS = 1e-8


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def host(t):
    return np.ascontiguousarray(t.detach().cpu().numpy())


@pytest.fixture(scope="module")
def F_():
    import gfla_b200
    from gfla_b200 import _lib
    _lib.check(_lib.lib().gfla_device_check(), "device check")
    return gfla_b200.functional


def _cos_chain(v, t, gcos):
    """cos = sum_c (v/max(|v|,eps)) (t/max(|t|,eps)) over axis 1 and its gradients, in float64"""
    v, t, gcos = v.astype(np.float64), t.astype(np.float64), gcos.astype(np.float64)
    nv, nt = np.sqrt((v * v).sum(1)), np.sqrt((t * t).sum(1))
    a, b = np.maximum(nv, EPS), np.maximum(nt, EPS)
    dot = (v * t).sum(1)
    cos = dot / (a * b)
    k1 = gcos / (a * b)
    k2v = np.where(nv > EPS, gcos * dot / (a * a * b * np.where(nv > 0, nv, 1.0)), 0.0)
    k2t = np.where(nt > EPS, gcos * dot / (a * b * b * np.where(nt > 0, nt, 1.0)), 0.0)
    gv = k1[:, None] * t - k2v[:, None] * v
    gt = k1[:, None] * v - k2t[:, None] * t
    return cos, gv, gt


@pytest.mark.parametrize("dt", [np.float32, np.float64])
@pytest.mark.parametrize("cfg", [(4, 1, 2.0), (2, 1, 5.0), (4, 2, 2.0), (6, 1, 1.5)])
def test_resample2d_cosine_vs_oracle(F_, oracle_lib, dt, cfg):
    ks, dil, sigma = cfg
    rng = np.random.default_rng(ks * 10 + dil)
    B, C, Hi, Wi, H, W = 2, 9, 15, 37, 13, 35          # ragged 32x4 tiles, source larger than the flow grid
    a = rng.standard_normal((B, C, Hi, Wi)).astype(dt)
    tgt = rng.standard_normal((B, C, H, W)).astype(dt)
    in2 = np.concatenate([rng.uniform(-6, 6, (B, 2, H, W)), np.full((B, 1, H, W), sigma)], 1).astype(dt)
    gcos = rng.standard_normal((B, H, W)).astype(dt)

    cos, stats = F_.resample2d_cosine_fwd(cu(a), cu(in2), cu(tgt), ks, dil, EPS)
    warped = oracle_lib.resample2d_fwd(a, in2, ks, dil)
    ref_cos, gv, gt = _cos_chain(warped, tgt, gcos)
    t = 1e-5 if dt == np.float32 else 1e-11
    np.testing.assert_allclose(host(cos), ref_cos, rtol=t, atol=t)
    np.testing.assert_allclose(host(stats)[:, 1], np.sqrt((warped.astype(np.float64) ** 2).sum(1)), rtol=t, atol=t)

    g1, g2, g3 = F_.resample2d_cosine_bwd(cu(a), cu(in2), cu(tgt), stats, cu(gcos), ks, dil, EPS, need_input1=True, need_target=True)
    o1, o2 = oracle_lib.resample2d_bwd(a, in2, gv.astype(dt), ks, dil)
    t = 2e-5 if dt == np.float32 else 1e-10
    np.testing.assert_allclose(host(g3), gt, rtol=t, atol=t * max(1.0, float(np.abs(gt).max())))
    np.testing.assert_allclose(host(g1), o1, rtol=t, atol=t * max(1.0, float(np.abs(o1).max())))
    np.testing.assert_allclose(host(g2), o2, rtol=10 * t, atol=10 * t * max(1.0, float(np.abs(o2).max())))
    # the flow-only backward (what the loss uses) gives the same grad_input2 and touches nothing else
    n1, n2, n3 = F_.resample2d_cosine_bwd(cu(a), cu(in2), cu(tgt), stats, cu(gcos), ks, dil, EPS)
    assert n1 is None and n3 is None
    assert torch.equal(n2, g2)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_resample2d_cosine_module_equals_unfused_composition(dtype):
    """value and all three gradients against torch autograd through the unfused modules, incl. zero feature vectors (both clamps)"""
    import gfla_b200
    torch.manual_seed(4)
    B, C, H, W = 2, 16, 20, 40
    x = torch.randn(B, C, H, W, device=DEV, dtype=dtype)
    tg = torch.randn(B, C, H, W, device=DEV, dtype=dtype)
    x[:, :, 3:9, 5:30] = 0          # warped vector exactly zero where the taps fall inside this block
    tg[:, :, 10:12, :] = 0          # zero target vectors
    flow = (torch.rand(B, 2, H, W, device=DEV, dtype=dtype) * 6 - 3)
    leaves = [[t.clone().requires_grad_() for t in (x, flow, tg)] for _ in range(2)]
    ref = F.cosine_similarity(gfla_b200.Resample2d(4, 1, sigma=2)(leaves[0][0], leaves[0][1]), leaves[0][2], dim=1, eps=EPS)
    ours = gfla_b200.Resample2dCosine(4, 1, sigma=2, eps=EPS)(leaves[1][0], leaves[1][1], leaves[1][2])
    assert ours.shape == ref.shape == (B, H, W)
    t = 1e-5 if dtype == torch.float32 else 1e-11
    assert (ours - ref).abs().max().item() <= t
    assert (ref == 0).any()                                       # the degenerate pixels are really exercised
    g = torch.randn_like(ref)
    ref.backward(g)
    ours.backward(g)
    for (r, o, name) in zip(leaves[0], leaves[1], ("input1", "flow", "target")):
        scale = max(1.0, r.grad.abs().max().item())
        assert torch.isfinite(o.grad).all(), name
        assert (r.grad - o.grad).abs().max().item() <= 20 * t * scale, name


def test_resample2d_cosine_backward_skips_unrequested_gradients():
    import gfla_b200
    torch.manual_seed(1)
    x = torch.randn(1, 8, 16, 16, device=DEV)                    # VGG features of data: no grad
    tg = torch.randn(1, 8, 16, 16, device=DEV)
    flow = torch.zeros(1, 2, 16, 16, device=DEV, requires_grad=True)
    from gfla_b200 import _lib
    n0 = _lib.lib().gfla_debug_launch_count()
    gfla_b200.Resample2dCosine(4, 1, sigma=2)(x, flow, tg).sum().backward()
    assert _lib.lib().gfla_debug_launch_count() - n0 == 2        # one kernel forward, one backward: no scatter pass
    assert flow.grad is not None and torch.isfinite(flow.grad).all()


def test_perceptual_correctness_equals_reference_class():
    """the reference's PerceptualCorrectness (external_function.py:222-284) with its Resample2d(4, 1, sigma=2) against
    gfla_b200.PerceptualCorrectness on the fused op: same feature extractor, same loss, same flow gradients, with and without
    a mask.  The reference class's values (its resample op on the reference's kernel bodies) are stored in
    tests/golden/reference_perceptual.npz by tests/golden/make_golden.py."""
    import gfla_b200
    from conftest import FixedFeatures, load_golden, perceptual_inputs
    ref = load_golden("reference_perceptual")
    ours = gfla_b200.PerceptualCorrectness(vgg=FixedFeatures()).to(DEV).eval()
    target, source, mask, flows = perceptual_inputs(DEV)
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        for name, m in (("nomask", None), ("mask", mask)):
            want = ref[f"resample_{name}"]
            fb = [f.clone().requires_grad_() for f in flows]
            lb = ours(target, source, fb, [2, 3], m)
            la = float(want["loss"])
            assert abs(la - float(lb)) <= 1e-5 * max(1.0, abs(la))
            lb.backward()
            for i, b in enumerate(fb):
                a = torch.from_numpy(want[f"grad{i}"]).to(DEV)
                assert a.abs().max().item() > 0
                assert (a - b.grad).abs().max().item() <= 1e-4 * max(1e-6, a.abs().max().item())
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
