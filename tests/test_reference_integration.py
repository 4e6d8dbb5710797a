"""CPU: the reference's OWN network code (base_function.py, generator.py) imports and constructs on top of this
package's shims -- i.e. pose/face/shapenet generators call the ops unchanged (north_star).  That test needs a checkout
of the reference and skips without one; the loss constants are checked against values stored from the reference."""
import os
import subprocess
import sys

import pytest

from conftest import ROOT

REF = "/root/reference"

SCRIPT = r"""
import sys, warnings
warnings.simplefilter("ignore")
sys.path.insert(0, %r)
import gfla_b200
gfla_b200.compat.install(reference_root=%r, fuse_extractor_attn=%s)
from model.networks.generator import PoseGenerator, FaceGenerator
import model.networks.base_function as bf
g = PoseGenerator(image_nc=3, structure_nc=18, ngf=64, img_f=512, layers=3, num_blocks=2, use_spect=False,
                  attn_layer=[2, 3], norm='instance', activation='LeakyReLU', extractor_kz={'2': 5, '3': 3})   # pose_model.py:62-64
attn = [getattr(g.target, 'attn%%d' %% i) for i in range(2)]
print(type(attn[0]).__module__, type(attn[0].extractor).__module__, type(attn[0].reshape).__module__)
print(sorted(k for k in g.state_dict() if 'attn0.fully_connect_layer' in k))
print(attn[0].kernel_size, attn[1].kernel_size)
f = FaceGenerator(image_nc=3, structure_nc=16, ngf=64, img_f=512, layers=3, num_blocks=2, use_spect=False,
                  attn_layer=[2, 3], norm='instance', activation='LeakyReLU', extractor_kz={'2': 5, '3': 3})   # face_model.py:78-80
print(sum(p.numel() for p in f.parameters()) > 0)
"""


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "model", "networks")), reason="reference checkout not present")
@pytest.mark.parametrize("fuse", [True, False])
def test_reference_generators_build_on_our_ops(fuse):
    out = subprocess.run([sys.executable, "-c", SCRIPT % (ROOT, REF, fuse)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = out.stdout.strip().splitlines()
    mod_attn, mod_ex, mod_rs = lines[0].split()
    assert mod_ex == "gfla_b200.block_extractor" and mod_rs == "gfla_b200.local_attn_reshape"
    assert mod_attn == ("gfla_b200.extractor_attn" if fuse else "model.networks.base_function")
    # checkpoint compatibility: same parameter names either way (base_function.py:799-803)
    assert lines[1] == str(['target.attn0.fully_connect_layer.0.bias', 'target.attn0.fully_connect_layer.0.weight',
                            'target.attn0.fully_connect_layer.2.bias', 'target.attn0.fully_connect_layer.2.weight'])
    assert lines[2] == "3 5"       # attn_layer=2,3 with kernel_size 2=5,3=3: level 3 (first built) k=3, level 2 k=5
    assert lines[3] == "True"


def test_regularization_loss_constants_match_the_reference_class():
    """the reference's AffineRegularizationLoss itself needs a GPU (its two custom ops); its constants and grid do not.
    What its class computes (kernel per kz, flow2grid of a seeded flow, MultiAffineRegularizationLoss's layer order and
    kernel sizes) is stored in tests/golden/reference_losses.npz by tests/golden/make_golden.py."""
    import numpy as np
    import torch
    import gfla_b200
    from conftest import load_golden
    ref = load_golden("reference_losses")
    for kz in (3, 4, 5):
        want = torch.from_numpy(ref[f"kz{kz}"]["kernel"])
        ours = gfla_b200.AffineRegularizationLoss(kz)
        assert tuple(ours.kernel.shape) == tuple(want.shape)
        assert float((want - ours.kernel).abs().max()) < 1e-12
        flow = torch.from_numpy(ref[f"kz{kz}"]["flow"])
        assert np.array_equal(ours.flow2grid(flow).numpy(), ref[f"kz{kz}"]["grid"])
    m = ref["multi"]
    o = gfla_b200.MultiAffineRegularizationLoss({"2": 5, "3": 3})
    assert o.layers == [str(x) for x in m["layers"]] and [o.method_dic[k].kz for k in o.layers] == list(m["kz"])
