"""Drop-in for model/networks/resample2d_package/resample2d.py."""
import torch
from torch.autograd import Function
from torch.nn.modules.module import Module

from . import functional as F_


def _features(t):
    """16-bit channels_last feature maps stay as they are (the channels-last kernels read them in place); anything else
    is made contiguous, as the reference's module does"""
    if t.dtype in F_._HALF and t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last):
        return t
    return t.contiguous()


def _input2(input1, flow, sigma):
    """input2 = cat(flow, sigma plane) (resample2d.py:51-52) in the dtype the kernels take it in: fp32 next to bf16 / fp16
    features (F_.flow_f32), input1's own dtype next to fp32 / fp64 ones (a bf16 generator's flow into an fp32 VGG).
    Autograd casts the flow gradient back to the flow's dtype."""
    flow = F_.flow_f32(input1, flow)
    if flow.dtype != input1.dtype and input1.dtype not in F_._HALF:
        flow = flow.to(input1.dtype)
    plane = torch.full((flow.size(0), 1, flow.size(2), flow.size(3)), sigma, dtype=flow.dtype, device=flow.device)
    return torch.cat((flow, plane), 1)


def _is_features(t):
    return t.is_contiguous() or (t.dtype in F_._HALF and t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last))


class Resample2dFunction(Function):
    """reference: resample2d.py:6-39.  input2 carries (dx, dy, sigma)."""

    @staticmethod
    def forward(ctx, input1, input2, kernel_size=2, dilation=1):
        assert _is_features(input1)          # contiguous; bf16 / fp16 may also be channels_last
        assert input2.is_contiguous()
        ctx.save_for_backward(input1, input2)
        ctx.kernel_size = kernel_size
        ctx.dilation = dilation
        return F_.resample2d_fwd(input1, input2, kernel_size, dilation)

    @staticmethod
    def backward(ctx, grad_output):
        input1, input2 = ctx.saved_tensors
        grad_input1, grad_input2 = F_.resample2d_bwd(input1, input2, grad_output, ctx.kernel_size, ctx.dilation)
        return grad_input1, grad_input2, None, None


class Resample2d(Module):
    """reference: resample2d.py:41-53.

    One deliberate difference: the reference builds ``self.sigma`` with
    ``.cuda()`` inside ``__init__`` (resample2d.py:47), which needs a GPU at
    construction time and pins the module to device 0; here sigma is kept as a
    Python float and materialised on the input's device in ``forward``."""

    def __init__(self, kernel_size=2, dilation=1, sigma=5):
        super(Resample2d, self).__init__()
        self.kernel_size = kernel_size
        self.dilation = dilation
        self.sigma = float(sigma)

    def forward(self, input1, input2):
        input1_c = _features(input1)
        return Resample2dFunction.apply(input1_c, _input2(input1_c, input2, self.sigma), self.kernel_size, self.dilation)


class Resample2dCosineFunction(Function):
    """cosine_similarity(Resample2dFunction(input1, input2), target, dim=1, eps) as ONE op each way (SURVEY row f4;
    external_function.py:275-279).  The warped tensor is neither written nor saved: the backward rebuilds each channel of it
    in registers.  Gradients are produced only for the inputs that ask for one -- in the reference's loss that is the flow."""

    @staticmethod
    def forward(ctx, input1, input2, target, kernel_size=2, dilation=1, eps=1e-8):
        assert _is_features(input1)
        assert input2.is_contiguous()
        target = _features(target)
        cos, stats = F_.resample2d_cosine_fwd(input1, input2, target, kernel_size, dilation, eps)
        ctx.save_for_backward(input1, input2, target, stats)
        ctx.cfg = (kernel_size, dilation, eps)
        return cos

    @staticmethod
    def backward(ctx, grad_cos):
        input1, input2, target, stats = ctx.saved_tensors
        ks, dil, eps = ctx.cfg
        g1, g2, gt = F_.resample2d_cosine_bwd(input1, input2, target, stats, grad_cos, ks, dil, eps,
                                              need_input1=ctx.needs_input_grad[0], need_target=ctx.needs_input_grad[2])
        return g1, g2, gt, None, None, None


class Resample2dCosine(Module):
    """``Resample2dCosine(ks, dil, sigma)(source, flow, target)`` == ``F.cosine_similarity(Resample2d(ks, dil, sigma)(source, flow),
    target)`` -> [B,H,W]."""

    def __init__(self, kernel_size=2, dilation=1, sigma=5, eps=1e-8):
        super(Resample2dCosine, self).__init__()
        self.kernel_size = kernel_size
        self.dilation = dilation
        self.sigma = float(sigma)
        self.eps = float(eps)

    def forward(self, input1, input2, target):
        input1_c = _features(input1)
        return Resample2dCosineFunction.apply(input1_c, _input2(input1_c, input2, self.sigma), target, self.kernel_size, self.dilation,
                                              self.eps)
