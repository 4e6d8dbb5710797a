import hashlib
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on the B200 box)")


def sha256(a):
    """digest of an array's dtype, shape and values, standing in for a golden array that is compared exactly: equal
    digests mean np.array_equal(..., equal_nan=True) (-0.0 is hashed as 0.0 and every NaN as the same NaN)"""
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.array(np.nan, a.dtype), a + a.dtype.type(0))
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def sample_index(numel, n=1024):
    """the fixed positions (sorted, into the C-order flattening) at which a full-size golden output is stored"""
    return np.sort(np.random.default_rng(numel).integers(0, numel, n))


def golden_grad_out(seed, shape, dtype):
    """the incoming gradient of a golden case that stores a seed instead of the array"""
    return np.random.default_rng(seed).standard_normal(shape).astype(dtype)


class FixedFeatures(torch.nn.Module):
    """stands in for VGG19 in the PerceptualCorrectness comparisons: seeded 3x3 convolutions at the resolutions of
    relu3_1 (1/4) and relu4_1 (1/8), the two layers those comparisons use"""

    def __init__(self, seed=0):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.register_buffer("w3", torch.randn(32, 3, 3, 3, generator=g) / 3)
        self.register_buffer("w4", torch.randn(64, 32, 3, 3, generator=g) / 17)

    def forward(self, x):
        f = torch.nn.functional
        r3 = f.softplus(f.conv2d(f.avg_pool2d(x, 4), self.w3, padding=1))
        return {"relu3_1": r3, "relu4_1": f.softplus(f.conv2d(f.avg_pool2d(r3, 2), self.w4, padding=1))}


def perceptual_inputs(device="cpu"):
    """-> target, source, mask, [flow at 1/8, flow at 1/4]: the inputs of the PerceptualCorrectness comparisons"""
    g = torch.Generator().manual_seed(1)
    B = 2
    target, source = torch.rand(B, 3, 64, 64, generator=g), torch.rand(B, 3, 64, 64, generator=g)
    mask = (torch.rand(B, 1, 64, 64, generator=g) > 0.4).float()
    flows = [torch.randn(B, 2, 8, 8, generator=g) * 1.5, torch.randn(B, 2, 16, 16, generator=g) * 2.5]
    return target.to(device), source.to(device), mask.to(device), [f.to(device) for f in flows]


def load_golden(name):
    """-> {case: {key: array}} from tests/golden/<name>.npz; a case with `grad_out_seed` gets its `grad_out` rebuilt"""
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    cases = {}
    for full in z.files:
        case, key = full.split("/", 1)
        cases.setdefault(case, {})[key] = z[full]
    for c in cases.values():
        if "grad_out_seed" in c:
            c["grad_out"] = golden_grad_out(int(c["grad_out_seed"]), tuple(c["grad_out_shape"]), c["source"].dtype)
    return cases


@pytest.fixture(scope="session")
def oracle_lib():
    import oracle.oracle as orc
    orc.build()          # gcc is in the image on both boxes; _ref only where the reference exists
    return orc.Oracle()


@pytest.fixture(scope="session")
def ref_lib():
    import oracle.oracle as orc
    if not orc.have_ref():
        pytest.skip("oracle/_ref not built (needs /root/reference)")
    return orc.Ref(threads=1)
