"""gfla_b200.AffineRegularizationLoss (SURVEY section 8 row f3) against the reference's literal composition
(external_function.py:61-69) evaluated on the CPU with the oracle's block_extractor / local_attn_reshape."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import gfla_b200
from gfla_b200.losses import affine_residual_kernel


def _literal_loss(flow, kz, O):
    """the reference's __call__ / calculate_loss, op for op; the two custom ops come from the oracle"""
    b, _, h, w = flow.shape
    x = torch.arange(w).view(1, -1).expand(h, -1).to(flow.dtype)
    y = torch.arange(h).view(-1, 1).expand(-1, w).to(flow.dtype)
    grid = flow + torch.stack([x, y], 0).unsqueeze(0)
    weights = torch.from_numpy(affine_residual_kernel(kz)).view(kz * kz, kz, kz).unsqueeze(1).to(flow.dtype)
    total = 0.0
    for comp in (0, 1):
        g = grid[:, comp:comp + 1].contiguous()
        results = F.conv2d(g, weights)
        hb, wb = results.shape[2:]
        kernels_new = torch.from_numpy(O.attn_reshape_fwd(results.numpy(), kz))
        f = np.zeros((b, 2, hb, wb), dtype=results.numpy().dtype) + float(int(kz / 2))
        grid_h = torch.from_numpy(O.block_extract_fwd(g.numpy(), f, kz))
        result = F.avg_pool2d(grid_h * kernels_new, kz, kz)
        total = total + torch.mean(result) * kz ** 2
    return float(total)


def test_kernel_is_the_affine_fit_residual():
    for kz in (3, 4, 5):
        m = affine_residual_kernel(kz)
        assert m.shape == (kz * kz, kz * kz) and np.allclose(m, m.T)
        i, j = np.meshgrid(np.arange(kz), np.arange(kz), indexing="ij")
        for p in (i.ravel(), j.ravel(), np.ones(kz * kz), 2.5 * i.ravel() - 0.75 * j.ravel() + 3):   # affine windows cost nothing
            assert abs(p @ m @ p) < 1e-9
        assert np.allclose(m @ m, m)                     # K^T K = I - P is itself a projection


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("kz", [3, 4, 5])
def test_affine_regularization_matches_literal_composition(oracle_lib, kz, dtype):
    torch.manual_seed(kz)
    flow = (torch.randn(2, 2, 13, 17, dtype=dtype) * 3).contiguous()
    got = float(gfla_b200.AffineRegularizationLoss(kz)(flow))
    want = _literal_loss(flow, kz, oracle_lib)
    tol = 1e-10 if dtype == torch.float64 else 2e-4     # fp32: p^T M p cancels coordinates of size ~17 down to the residual
    assert abs(got - want) <= tol * max(1.0, abs(want)), (got, want)


def test_affine_regularization_gradient_and_multi_level():
    torch.manual_seed(0)
    flow = torch.randn(1, 2, 7, 8, dtype=torch.float64, requires_grad=True)
    loss_fn = gfla_b200.AffineRegularizationLoss(3)
    assert torch.autograd.gradcheck(lambda t: loss_fn(t), (flow,), atol=1e-6, rtol=1e-4)
    # an affine flow field is free of charge, whatever its size
    h, w = 9, 11
    yy, xx = torch.meshgrid(torch.arange(h, dtype=torch.float64), torch.arange(w, dtype=torch.float64), indexing="ij")
    affine = torch.stack([0.3 * xx - 0.2 * yy + 1.0, 0.1 * xx + 0.5 * yy - 2.0]).unsqueeze(0)
    assert float(gfla_b200.AffineRegularizationLoss(5)(affine)) < 1e-9
    # MultiAffineRegularizationLoss: descending layer keys, one flow field per level (external_function.py:12-28)
    multi = gfla_b200.MultiAffineRegularizationLoss({"2": 5, "3": 3})
    f3, f2 = torch.randn(1, 2, 8, 8, dtype=torch.float64), torch.randn(1, 2, 16, 16, dtype=torch.float64)
    want = gfla_b200.AffineRegularizationLoss(3)(f3) + gfla_b200.AffineRegularizationLoss(5)(f2)
    assert abs(float(multi([f3, f2])) - float(want)) < 1e-12


def test_perceptual_correctness_bilinear_branch_equals_reference_class():
    """gfla_b200.PerceptualCorrectness vs the reference's class (external_function.py:222-320) on CPU through the
    ``use_bilinear_sampling`` branch, which needs no custom op: everything around the fused resample -> cosine op
    (correlation, max, loss map, mask handling, layer bookkeeping) is pinned here; the fused branch is pinned on the GPU
    (tests/test_gpu_resample_cosine.py).  The reference class's loss and flow gradients on these inputs, with the same
    feature extractor, are stored in tests/golden/reference_perceptual.npz by tests/golden/make_golden.py."""
    from conftest import FixedFeatures, load_golden, perceptual_inputs
    ref = load_golden("reference_perceptual")
    ours = gfla_b200.PerceptualCorrectness(vgg=FixedFeatures()).eval()
    target, source, mask, flows = perceptual_inputs()
    for name, m in (("nomask", None), ("mask", mask)):
        want = ref[f"bilinear_{name}"]
        fb = [f.clone().requires_grad_() for f in flows]
        lb = ours(target, source, fb, [2, 3], m, True)
        assert abs(float(want["loss"]) - lb.item()) <= 1e-6
        lb.backward()
        for i, b in enumerate(fb):
            a = torch.from_numpy(want[f"grad{i}"])
            assert a.abs().max().item() > 1e-5
            assert (a - b.grad).abs().max().item() <= 1e-6 * max(1.0, a.abs().max().item())
