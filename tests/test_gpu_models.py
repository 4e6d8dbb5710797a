"""GPU (-m gpu): the reference's OWN generators / losses (snapshot baseline/_ref, byte-identical files) running
on this library -- BASELINE configs 4 and 5 at test size, SURVEY rows f2/f3.

  * one PoseGenerator / FaceGenerator forward with the fused ExtractorAttn equals the literal reference op chain
    (reference ExtractorAttn class on the unfused ops), and -- where the library was built -- the chain on the
    reference's own CUDA kernels recompiled for sm_100a;
  * the INTEGRATION.md recipe (`.bfloat16().to(memory_format=channels_last)`) reaches the tcgen05 tile kernels in
    forward AND backward (the flow is bf16 there: it is widened to fp32, ADVICE r1);
  * AffineRegularizationLoss on the GPU: the op-free rewrite in losses.py vs the reference class's stored values.
The generator tests need the reference's own network sources and skip without them.
"""

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(autouse=True)
def _no_tf32():
    """fused vs literal split the FC conv differently; with TF32 convolutions (torch's default) that alone is a 5e-4 difference"""
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


@pytest.fixture(scope="module")
def BM():
    import bench_models
    if bench_models.reference_root() is None:
        pytest.skip("baseline/_ref snapshot of the reference generators not present")
    return bench_models


def _pose_inputs(b, dtype=torch.float32, fmt=torch.contiguous_format):
    g = torch.Generator(device="cpu").manual_seed(3)
    mk = lambda c: torch.randn(b, c, 256, 256, generator=g).to(DEV, dtype).contiguous(memory_format=fmt)
    return mk(3), mk(18), mk(18)


def _build(BM, arm, kind, dtype=torch.float32, cl=False):
    Pose, Face = BM.load_generators(arm)
    torch.manual_seed(11)
    net = Pose(**BM.POSE_KW) if kind == "pose" else Face(**BM.FACE_KW)
    net.init_weights("orthogonal", gain=0.5)       # larger than the reference's 0.02 so flows / masks are not degenerate
    net = net.to(DEV, dtype)
    return net.to(memory_format=torch.channels_last) if cl else net


def test_pose_generator_fused_equals_literal_and_reference_cuda(BM):
    x = _pose_inputs(2)
    outs = {}
    for arm in ("fused", "literal", "refcuda"):
        try:
            net = _build(BM, arm, "pose")
        except FileNotFoundError:
            continue
        with torch.no_grad():
            img, flows, masks = net(*x)
        outs[arm] = (img, flows)
        assert type(net.target.attn0).__module__ == ("gfla_b200.extractor_attn" if arm == "fused" else "model.networks.base_function")
    assert "fused" in outs and "literal" in outs
    scale = max(1.0, outs["literal"][0].abs().max().item())
    assert (outs["fused"][0] - outs["literal"][0]).abs().max().item() <= 1e-4 * scale
    assert any(f.abs().max().item() > 0.05 for f in outs["literal"][1])       # the flow fields actually displace
    if "refcuda" in outs:
        assert (outs["fused"][0] - outs["refcuda"][0]).abs().max().item() <= 1e-4 * scale


def test_pose_generator_backward_fused_equals_literal(BM):
    x = _pose_inputs(1)
    grads = {}
    for arm in ("fused", "literal"):
        net = _build(BM, arm, "pose")
        img, flows, masks = net(*x)
        (img.mean() + sum(f.pow(2).mean() for f in flows)).backward()
        grads[arm] = {n: p.grad.clone() for n, p in net.named_parameters() if p.grad is not None}
    assert grads["fused"].keys() == grads["literal"].keys() and len(grads["fused"]) > 50
    rel = []
    for n, g in grads["literal"].items():
        err, ref = (grads["fused"][n] - g).norm().item(), g.norm().item()
        rel.append(err / (ref + 1e-12))
        assert err <= 5e-2 * ref + 1e-7, (n, err, ref)      # fp32 atomics / summation order, amplified through ~40 layers + instance norms
    rel.sort()
    assert rel[len(rel) // 2] <= 5e-3, rel[len(rel) // 2]   # ... while the typical parameter agrees to a fraction of a percent


def test_face_generator_fused_equals_literal(BM):
    g = torch.Generator(device="cpu").manual_seed(5)
    mk = lambda *s: torch.randn(*s, generator=g).to(DEV)
    x = [mk(1, 2, 16, 256, 256), mk(1, 3, 256, 256), mk(1, 16, 256, 256), None, None]
    outs = {}
    for arm in ("fused", "literal"):
        net = _build(BM, arm, "face").eval()
        with torch.no_grad():
            imgs, _, _, _ = net(*x)
        outs[arm] = torch.stack(imgs)
    assert (outs["fused"] - outs["literal"]).abs().max().item() <= 1e-4 * max(1.0, outs["literal"].abs().max().item())


def test_bf16_channels_last_generator_reaches_the_tile_kernels(BM):
    """INTEGRATION.md recipe: every ExtractorAttn level must launch the tcgen05 forward AND backward kernels"""
    from torch.profiler import ProfilerActivity, profile
    net = _build(BM, "fused", "pose", torch.bfloat16, cl=True)
    x = _pose_inputs(2, torch.bfloat16, torch.channels_last)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        img, flows, masks = net(*x)
        assert flows[0].dtype == torch.bfloat16            # the network really hands us a bf16 flow
        img.float().mean().backward()
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages()]
    fwd = [n for n in names if "k_local_attn_fwd_strip" in n or "k_local_attn_fwd_tc" in n]
    bwd = [n for n in names if "k_local_attn_bwd" in n and "_tc" in n or "k_local_attn_bwd_fused" in n]
    slow = [n for n in names if "gfla::k_local_attn_fwd<" in n or "gfla::k_local_attn_bwd<" in n]
    assert fwd and bwd, names
    assert not slow, slow                                    # no fall-back to the CUDA-core gather kernels
    assert torch.isfinite(img.float()).all()
    assert all(p.grad is None or torch.isfinite(p.grad.float()).all() for p in net.parameters())


@pytest.mark.parametrize("kz", [3, 5])
def test_affine_regularization_loss_gpu_vs_reference_class(kz):
    """the reference's AffineRegularizationLoss (external_function.py:31-77) vs losses.AffineRegularizationLoss on the GPU
    (no custom op at all): value and gradient.  The reference class's values, with its two custom ops on the reference's
    kernel bodies, are stored in tests/golden/reference_losses.npz by tests/golden/make_golden.py."""
    import gfla_b200
    from conftest import load_golden
    ref = load_golden("reference_losses")[f"kz{kz}"]
    flow = (torch.randn(2, 2, 32, 32, generator=torch.Generator().manual_seed(kz)) * 3).to(DEV).requires_grad_()
    ours = gfla_b200.AffineRegularizationLoss(kz)(flow)
    want = float(ref["loss"])
    assert abs(want - float(ours)) <= 2e-4 * max(1.0, abs(want))
    ours.backward()
    g = torch.from_numpy(ref["loss_grad"]).to(DEV)
    assert (g - flow.grad).abs().max().item() <= 2e-4 * max(1e-3, g.abs().max().item())
