"""Fused local attention and a drop-in ``ExtractorAttn``.

Reference: model/networks/base_function.py:790-818.  The module keeps the
reference's constructor, attribute names and ``state_dict`` keys
(``fully_connect_layer.{0,2}.{weight,bias}``) so reference checkpoints load
unchanged; what changes is how ``forward`` runs:

    reference                                   here
    ---------                                   ----
    block_source = extractor(source, flow)      same (needed as conv input)
    block_target = extractor(target, 0)         NOT materialised: its conv == a stride-1 conv of `target`
                                                with replicate padding (see _logits)
    attn = fc(cat(block_target, block_source))  conv -> act -> conv produce LOGITS;
           ... ending in Softmax(dim=1)         the softmax is folded into the fused kernel
    attn = reshape(attn, k)                     --
    out  = avg_pool2d(attn * block_source,k,k)  LocalAttnFunction(source, flow, logits): one kernel,
                                                never touches the [B,C,kH,kW] product again
"""
import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.autograd import Function

from . import functional as F_
from .block_extractor import BlockExtractor
from .local_attn_reshape import LocalAttnReshape


class LocalAttnFunction(Function):
    """(source [B,C,Hs,Ws], flow [B,2,H,W], logits [B,k*k,H,W]) -> out [B,C,H,W]

    out = avg_pool2d(LocalAttnReshape(softmax(logits, 1)) * BlockExtractor(k)(source, flow), k, k)
    """

    @staticmethod
    def forward(ctx, source, flow_field, logits, kernel_size, algo="auto"):
        assert flow_field.is_contiguous() and logits.is_contiguous()
        ctx.save_for_backward(source, flow_field, logits)
        ctx.kernel_size = kernel_size
        ctx.algo = algo
        return F_.local_attn_fwd(source, flow_field, logits, kernel_size, algo=algo)

    @staticmethod
    def backward(ctx, grad_output):
        source, flow_field, logits = ctx.saved_tensors
        gs, gf, gl = F_.local_attn_bwd(source, flow_field, logits, grad_output, ctx.kernel_size, algo=ctx.algo)
        return gs, gf, gl, None, None


def _keep_format(t):
    """contiguous NCHW stays, channels_last stays (the fast layout for the tile kernels); anything else -> NCHW"""
    if t.is_contiguous() or (t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last)):
        return t
    return t.contiguous()


_flow_f32 = F_.flow_f32


def local_attention(source, flow_field, logits, kernel_size, algo="auto"):
    return LocalAttnFunction.apply(_keep_format(source), _flow_f32(source, flow_field).contiguous(), logits.contiguous(),
                                   kernel_size, algo)


class ExtractorAttn(nn.Module):
    """Drop-in for base_function.py:790-818 (same ctor, same parameters)."""

    def __init__(self, feature_nc, kernel_size=4, nonlinearity=nn.LeakyReLU(), softmax=None):
        super(ExtractorAttn, self).__init__()
        self.kernel_size = kernel_size
        hidden_nc = 128
        self.fused_softmax = softmax is not None           # reference: `softmax=True` -> nn.Softmax(dim=1)
        softmax = nonlinearity if softmax is None else nn.Softmax(dim=1)

        self.extractor = BlockExtractor(kernel_size=kernel_size)
        self.reshape = LocalAttnReshape()
        self.fully_connect_layer = nn.Sequential(
            nn.Conv2d(2 * feature_nc, hidden_nc, kernel_size=kernel_size, stride=kernel_size, padding=0),
            nonlinearity,
            nn.Conv2d(hidden_nc, kernel_size * kernel_size, kernel_size=1, stride=1, padding=0),
            softmax,)

    def _logits(self, source, target, flow_field):
        """conv(k, stride k) over cat(block_target, block_source), then act, then the 1x1 conv (no softmax).

        The target half never needs its block tensor: BlockExtractor with a zero flow copies, for output
        position (y*k+i, x*k+j), target[clamp(y+i-k//2), clamp(x+j-k//2)] (integer taps: weights 1 and 0,
        block_extractor_kernel.cu:62-82), so a kernel-k stride-k convolution over it IS an ordinary kernel-k
        stride-1 convolution of `target` with replicate padding (k//2 before, k-1-k//2 after) using the first
        C input channels of the same weight.  Only block_source (flow-dependent, bilinear) is materialised.
        """
        conv1 = self.fully_connect_layer[0]
        k, c = self.kernel_size, source.shape[1]
        block_source = self.extractor(source, flow_field)
        x = F.conv2d(block_source, conv1.weight[:, c:], None, stride=k)
        lo, hi = k // 2, k - 1 - k // 2
        x = x + F.conv2d(F.pad(target, (lo, hi, lo, hi), mode="replicate"), conv1.weight[:, :c], conv1.bias)
        for layer in list(self.fully_connect_layer)[1:-1]:      # nonlinearity, 1x1 conv; not the softmax
            x = layer(x)
        return x, block_source

    def forward(self, source, target, flow_field, mask=None):
        """Reference signature (source, target, flow_field).  Optional `mask` [B,1,H,W]: also apply the caller's
        blend `target*(1-mask) + result*mask` (generator.py:130) -- fused into the kernel's store when no
        gradient is needed (inference), composed with torch ops otherwise."""
        logits, block_source = self._logits(source, target, flow_field)
        if self.fused_softmax:
            if mask is None:
                return local_attention(source, flow_field, logits, self.kernel_size)
            needs_grad = torch.is_grad_enabled() and any(t.requires_grad for t in (source, target, flow_field, logits, mask))
            if needs_grad:
                out_attn = local_attention(source, flow_field, logits, self.kernel_size)
                return target * (1 - mask) + out_attn * mask
            src = _keep_format(source)
            fmt = torch.channels_last if (not src.is_contiguous()) else torch.contiguous_format
            return F_.local_attn_blend_fwd(src, _flow_f32(src, flow_field).contiguous(), logits.contiguous(),
                                           target.contiguous(memory_format=fmt), mask.to(source.dtype), self.kernel_size)
        assert mask is None, "mask blend is only fused for the softmax variant"
        # softmax=None in the reference means "apply the nonlinearity instead": keep the literal composition
        attn_param = self.reshape(self.fully_connect_layer[-1](logits), self.kernel_size)
        return torch.nn.functional.avg_pool2d(attn_param * block_source, self.kernel_size, self.kernel_size)

    def hook_attn_param(self, source, target, flow_field):
        logits, block_source = self._logits(source, target, flow_field)
        if self.fused_softmax:
            result, probs = F_.local_attn_fwd(_keep_format(source), _flow_f32(source, flow_field).contiguous(), logits.contiguous(),
                                              self.kernel_size, return_probs=True)
            return probs, result
        attn_param_ = self.fully_connect_layer[-1](logits)
        attn_param = self.reshape(attn_param_, self.kernel_size)
        return attn_param_, torch.nn.functional.avg_pool2d(attn_param * block_source, self.kernel_size, self.kernel_size)
