"""Thin torch-tensor front end of the C ABI: pointer / size / stream plumbing only.

Every function here checks what the reference's autograd Functions check
(contiguity asserts: block_extractor.py:9-10, local_attn_reshape.py:9,
resample2d.py:10-11; `df == 2`: block_extractor.py:16; `ds == k*k`:
local_attn_reshape.py:13; CPU tensors -> NotImplementedError:
block_extractor.py:23-24, local_attn_reshape.py:20-21) and then hands raw
device pointers to libgfla_warp.so on the caller's current stream.
"""
from __future__ import annotations

import torch

from . import _lib

_DT = {torch.float32: _lib.GFLA_F32, torch.float64: _lib.GFLA_F64,
       torch.bfloat16: _lib.GFLA_BF16, torch.float16: _lib.GFLA_F16}


def _dt(t: torch.Tensor) -> int:
    try:
        return _DT[t.dtype]
    except KeyError:
        raise TypeError(f"unsupported dtype {t.dtype} (float32/float64, or bfloat16/float16 storage)") from None


def _need_cuda(*ts: torch.Tensor) -> None:
    for t in ts:
        if not t.is_cuda:
            # same behaviour as the reference ops: there is no CPU implementation
            raise NotImplementedError("GFLA warp ops are CUDA-only (sm_100a); got a CPU tensor")
    dev = ts[0].device
    for t in ts:
        if t.device != dev:
            raise ValueError("all tensors must live on the same CUDA device")


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


# --------------------------------------------------------------------------- block_extractor
def block_extract_fwd(source: torch.Tensor, flow: torch.Tensor, k: int) -> torch.Tensor:
    assert source.is_contiguous() and flow.is_contiguous()
    bs, ds, hs, ws = source.size()
    bf, df, hf, wf = flow.size()
    assert df == 2
    _need_cuda(source, flow)
    out = source.new_empty((bs, ds, k * hf, k * wf))   # fully written by the kernel: no zero fill needed
    with torch.cuda.device_of(source):
        _lib.check(_lib.lib().gfla_block_extract_fwd(_p(source), _p(flow), _p(out), bs, ds, hs, ws, hf, wf, k,
                                                     _dt(source), _dt(flow), _stream(source)), "block_extract_fwd")
    return out


def convert(t: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """fp32 <-> bf16/f16 copy with the library's kernel (contiguous tensors)."""
    assert t.is_contiguous()
    out = torch.empty_like(t, dtype=dtype)
    with torch.cuda.device_of(t):
        _lib.check(_lib.lib().gfla_convert(_p(t), _dt(t), _p(out), _DT[dtype], t.numel(), _stream(t)), "convert")
    return out


def block_extract_bwd(source, flow, grad_out, k, grad_source=None, grad_flow=None):
    """Returns (grad_source, grad_flow).  If buffers are passed, gradients are ADDED
    into them (reference contract, block_extractor.py:35-40)."""
    assert source.is_contiguous() and flow.is_contiguous()
    grad_out = grad_out.contiguous()
    _need_cuda(source, flow, grad_out)
    bs, ds, hs, ws = source.size()
    _, _, hf, wf = flow.size()
    accumulate, narrow = 1, False
    if grad_source is None:
        accumulate = 0
        # 16-bit storage: scatter into an fp32 buffer (native red.global.f32; a 16-bit scalar atomicAdd is a
        # compare-and-swap loop, ~50x slower) and narrow afterwards
        narrow = source.dtype in (torch.bfloat16, torch.float16)
        grad_source = torch.empty(source.shape, dtype=torch.float32 if narrow else source.dtype, device=source.device)
        grad_flow = torch.empty_like(flow)
    with torch.cuda.device_of(source):
        _lib.check(_lib.lib().gfla_block_extract_bwd(_p(source), _p(flow), _p(grad_out), _p(grad_source), _p(grad_flow),
                                                     bs, ds, hs, ws, hf, wf, k, _dt(source), _dt(flow), _dt(grad_source),
                                                     accumulate, _stream(source)), "block_extract_bwd")
    if narrow:
        grad_source = convert(grad_source, source.dtype)
    return grad_source, grad_flow


# --------------------------------------------------------------------------- local_attn_reshape
def attn_reshape_fwd(inputs: torch.Tensor, k: int) -> torch.Tensor:
    assert inputs.is_contiguous()
    bs, ds, hs, ws = inputs.size()
    assert ds == k * k
    _need_cuda(inputs)
    out = inputs.new_empty((bs, 1, k * hs, k * ws))
    with torch.cuda.device_of(inputs):
        _lib.check(_lib.lib().gfla_attn_reshape_fwd(_p(inputs), _p(out), bs, hs, ws, k, _dt(inputs), _stream(inputs)),
                   "attn_reshape_fwd")
    return out


def attn_reshape_bwd(grad_out: torch.Tensor, k: int, grad_in=None) -> torch.Tensor:
    grad_out = grad_out.contiguous()
    _need_cuda(grad_out)
    bs, _, ho, wo = grad_out.size()
    hs, ws = ho // k, wo // k
    accumulate = 1
    if grad_in is None:
        grad_in, accumulate = grad_out.new_empty((bs, k * k, hs, ws)), 0
    with torch.cuda.device_of(grad_out):
        _lib.check(_lib.lib().gfla_attn_reshape_bwd(_p(grad_out), _p(grad_in), bs, hs, ws, k, _dt(grad_out), accumulate,
                                                    _stream(grad_out)), "attn_reshape_bwd")
    return grad_in


# --------------------------------------------------------------------------- resample2d
def resample2d_fwd(input1: torch.Tensor, input2: torch.Tensor, kernel_size: int, dilation: int) -> torch.Tensor:
    """fp32 / fp64: planar kernels, input2 in input1's dtype.  bf16 / fp16: channels-last kernels, input2 fp32; input1 may be
    channels_last (used as it is) or contiguous NCHW (re-laid), and the output comes back in input1's memory format."""
    if input1.dtype in _HALF:
        return _resample2d_fwd_16(input1, input2, kernel_size, dilation)
    assert input1.is_contiguous() and input2.is_contiguous()
    _need_cuda(input1, input2)
    _, d, hi, wi = input1.size()
    b, three, h, w = input2.size()
    assert three == 3, "input2 must be [B,3,H,W] = (dx, dy, sigma) (resample2d.py:51-52)"
    if input2.dtype != input1.dtype:
        raise TypeError("resample2d: input1 and input2 must share a dtype (float32 or float64)")
    out = input1.new_empty((b, d, h, w))
    with torch.cuda.device_of(input1):
        _lib.check(_lib.lib().gfla_resample2d_fwd(_p(input1), _p(input2), _p(out), b, d, hi, wi, h, w, kernel_size,
                                                  dilation, _dt(input1), _stream(input1)), "resample2d_fwd")
    return out


def resample2d_bwd(input1, input2, grad_out, kernel_size, dilation, grad_input1=None, grad_input2=None):
    if input1.dtype in _HALF:
        return _resample2d_bwd_16(input1, input2, grad_out, kernel_size, dilation, grad_input1, grad_input2)
    assert input1.is_contiguous() and input2.is_contiguous()
    grad_out = grad_out.contiguous()
    _need_cuda(input1, input2, grad_out)
    _, d, hi, wi = input1.size()
    b, _, h, w = input2.size()
    accumulate = 1
    if grad_input1 is None:
        grad_input1, grad_input2, accumulate = torch.empty_like(input1), torch.empty_like(input2), 0
    with torch.cuda.device_of(input1):
        _lib.check(_lib.lib().gfla_resample2d_bwd(_p(input1), _p(input2), _p(grad_out), _p(grad_input1), _p(grad_input2),
                                                  b, d, hi, wi, h, w, kernel_size, dilation, _dt(input1), accumulate,
                                                  _stream(input1)), "resample2d_bwd")
    return grad_input1, grad_input2


def resample2d_cosine_fwd(input1, input2, target, kernel_size: int, dilation: int, eps: float = 1e-8):
    """cos[b,y,x] = cosine_similarity(resample2d(input1, input2)[b,:,y,x], target[b,:,y,x]) without the warped tensor
    (external_function.py:275-279).  -> (cos [B,H,W], stats [B,3,H,W] for the backward)
    bf16 / fp16 features (input1, target; channels_last or NCHW) take the channels-last kernels with an fp32 input2, and
    cos / stats are fp32."""
    if input1.dtype in _HALF:
        return _resample2d_cosine_fwd_16(input1, input2, target, kernel_size, dilation, eps)
    assert input1.is_contiguous() and input2.is_contiguous() and target.is_contiguous()
    _need_cuda(input1, input2, target)
    _, d, hi, wi = input1.size()
    b, three, h, w = input2.size()
    assert three == 3, "input2 must be [B,3,H,W] = (dx, dy, sigma) (resample2d.py:51-52)"
    assert tuple(target.shape) == (b, d, h, w), "target must be [B,C,H,W] on the flow's grid"
    if input2.dtype != input1.dtype or target.dtype != input1.dtype:
        raise TypeError("resample2d_cosine: input1, input2 and target must share a dtype (float32 or float64)")
    cos = input1.new_empty((b, h, w))
    stats = input1.new_empty((b, 3, h, w))
    with torch.cuda.device_of(input1):
        _lib.check(_lib.lib().gfla_resample2d_cosine_fwd(_p(input1), _p(input2), _p(target), _p(cos), _p(stats), b, d, hi, wi, h, w,
                                                         kernel_size, dilation, float(eps), _dt(input1), _stream(input1)),
                   "resample2d_cosine_fwd")
    return cos, stats


def resample2d_cosine_bwd(input1, input2, target, stats, grad_cos, kernel_size, dilation, eps=1e-8, need_input1=False,
                          need_target=False):
    """-> (grad_input1 | None, grad_input2, grad_target | None)"""
    if input1.dtype in _HALF:
        return _resample2d_cosine_bwd_16(input1, input2, target, stats, grad_cos, kernel_size, dilation, eps, need_input1,
                                         need_target)
    grad_cos = grad_cos.contiguous()
    _need_cuda(input1, input2, target, stats, grad_cos)
    _, d, hi, wi = input1.size()
    b, _, h, w = input2.size()
    grad_in2 = torch.empty_like(input2)
    grad_in1 = torch.empty_like(input1) if need_input1 else None
    grad_val = torch.empty_like(target) if need_input1 else None
    grad_target = torch.empty_like(target) if need_target else None
    with torch.cuda.device_of(input1):
        _lib.check(_lib.lib().gfla_resample2d_cosine_bwd(
            _p(input1), _p(input2), _p(target), _p(stats), _p(grad_cos), _p(grad_in1) if need_input1 else None, _p(grad_in2),
            _p(grad_val) if need_input1 else None, _p(grad_target) if need_target else None, b, d, hi, wi, h, w, kernel_size, dilation,
            float(eps), _dt(input1), 0, _stream(input1)), "resample2d_cosine_bwd")
    return grad_in1, grad_in2, grad_target


# --------------------------------------------------------------------------- resample2d, 16-bit channels-last
_HALF = (torch.bfloat16, torch.float16)


def flow_f32(features: torch.Tensor, flow: torch.Tensor) -> torch.Tensor:
    """16-bit feature tensors pair with an fp32 flow: the tap indices and weights are then bit-identical to the fp32
    path (block_extractor_kernel.cu:62-76, resample2d_kernel.cu:43-60), and the tcgen05 tile kernels -- which take fp32
    flow only -- serve the call.  A bf16/f16 flow (e.g. from a network cast wholesale with .bfloat16()) is widened here;
    autograd casts its gradient back to the flow's dtype."""
    if features.dtype in _HALF and flow.dtype != torch.float32:
        return flow.float()
    return flow


def _to_nhwc(t: torch.Tensor) -> torch.Tensor:
    """a [B,C,H,W] tensor in channels-last storage: as it is when it already is, re-laid by the library when it is NCHW"""
    if t.is_contiguous(memory_format=torch.channels_last):
        return t
    return relayout(t.contiguous(), True)


def _like_caller(t: torch.Tensor, planar: bool) -> torch.Tensor:
    """a channels-last result back in the caller's memory format (planar = the caller's tensor was contiguous NCHW)"""
    return relayout(t, False) if planar and not t.is_contiguous() else t


def _narrow(t: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """fp32 -> 16-bit copy of a dense (NCHW or channels-last) tensor with the library's kernel, keeping its strides"""
    out = torch.empty_like(t, dtype=dtype)
    with torch.cuda.device_of(t):
        _lib.check(_lib.lib().gfla_convert(_p(t), _dt(t), _p(out), _DT[dtype], t.numel(), _stream(t)), "convert")
    return out


def _in2_f32(input2: torch.Tensor) -> None:
    assert input2.is_contiguous()
    b, three, h, w = input2.size()
    assert three == 3, "input2 must be [B,3,H,W] = (dx, dy, sigma) (resample2d.py:51-52)"
    if input2.dtype != torch.float32:
        raise TypeError("resample2d: bfloat16/float16 input1 takes a float32 input2 (dx, dy, sigma)")


def _resample2d_fwd_16(input1, input2, kernel_size, dilation):
    _in2_f32(input2)
    _need_cuda(input1, input2)
    planar = input1.is_contiguous()
    x = _to_nhwc(input1)
    _, d, hi, wi = x.size()
    b, _, h, w = input2.size()
    out = torch.empty((b, d, h, w), dtype=x.dtype, device=x.device, memory_format=torch.channels_last)
    with torch.cuda.device_of(x):
        _lib.check(_lib.lib().gfla_resample2d_fwd_nhwc(_p(x), _p(input2), _p(out), b, d, hi, wi, h, w, kernel_size, dilation, _dt(x),
                                                       _stream(x)), "resample2d_fwd_nhwc")
    return _like_caller(out, planar)


def _resample2d_bwd_16(input1, input2, grad_out, kernel_size, dilation, grad_input1=None, grad_input2=None):
    """grad_input1 comes back in input1's dtype and memory format, grad_input2 in fp32.  Buffers passed in (reference
    contract: gradients are ADDED) must be channels_last for grad_input1 (its dtype or fp32) and fp32 for grad_input2."""
    _in2_f32(input2)
    _need_cuda(input1, input2, grad_out)
    planar = input1.is_contiguous()
    x, go = _to_nhwc(input1), _to_nhwc(grad_out)
    _, d, hi, wi = x.size()
    b, _, h, w = input2.size()
    accumulate, narrow = 1, False
    if grad_input1 is None:
        # scatter into an fp32 buffer (fp32 reductions in L2) and narrow afterwards, as block_extract_bwd does
        accumulate, narrow = 0, True
        grad_input1 = torch.empty(x.shape, dtype=torch.float32, device=x.device, memory_format=torch.channels_last)
        grad_input2 = torch.empty_like(input2)
    assert grad_input1.is_contiguous(memory_format=torch.channels_last), "grad_input1 buffer must be channels_last"
    assert grad_input2.is_contiguous() and grad_input2.dtype == torch.float32
    with torch.cuda.device_of(x):
        _lib.check(_lib.lib().gfla_resample2d_bwd_nhwc(_p(x), _p(input2), _p(go), _p(grad_input1), _p(grad_input2), b, d, hi, wi, h, w,
                                                       kernel_size, dilation, _dt(x), _dt(grad_input1), accumulate, _stream(x)),
                   "resample2d_bwd_nhwc")
    if narrow:
        grad_input1 = _like_caller(_narrow(grad_input1, x.dtype), planar)
    return grad_input1, grad_input2


def _resample2d_cosine_fwd_16(input1, input2, target, kernel_size, dilation, eps):
    _in2_f32(input2)
    _need_cuda(input1, input2, target)
    if target.dtype != input1.dtype:
        raise TypeError("resample2d_cosine: input1 and target must share a dtype")
    x, tg = _to_nhwc(input1), _to_nhwc(target)
    _, d, hi, wi = x.size()
    b, _, h, w = input2.size()
    assert tuple(tg.shape) == (b, d, h, w), "target must be [B,C,H,W] on the flow's grid"
    cos = torch.empty((b, h, w), dtype=torch.float32, device=x.device)
    stats = torch.empty((b, 3, h, w), dtype=torch.float32, device=x.device)
    with torch.cuda.device_of(x):
        _lib.check(_lib.lib().gfla_resample2d_cosine_fwd_nhwc(_p(x), _p(input2), _p(tg), _p(cos), _p(stats), b, d, hi, wi, h, w,
                                                              kernel_size, dilation, float(eps), _dt(x), _stream(x)),
                   "resample2d_cosine_fwd_nhwc")
    return cos, stats


def _resample2d_cosine_bwd_16(input1, input2, target, stats, grad_cos, kernel_size, dilation, eps, need_input1, need_target):
    _in2_f32(input2)
    grad_cos = grad_cos.float().contiguous()
    _need_cuda(input1, input2, target, stats, grad_cos)
    x, tg = _to_nhwc(input1), _to_nhwc(target)
    _, d, hi, wi = x.size()
    b, _, h, w = input2.size()
    cl = torch.channels_last
    grad_in2 = torch.empty_like(input2)
    grad_in1 = torch.empty(x.shape, dtype=torch.float32, device=x.device, memory_format=cl) if need_input1 else None
    grad_val = torch.empty(tg.shape, dtype=x.dtype, device=x.device, memory_format=cl) if need_input1 else None
    grad_target = torch.empty(tg.shape, dtype=x.dtype, device=x.device, memory_format=cl) if need_target else None
    with torch.cuda.device_of(x):
        _lib.check(_lib.lib().gfla_resample2d_cosine_bwd_nhwc(
            _p(x), _p(input2), _p(tg), _p(stats), _p(grad_cos), _p(grad_in1), _p(grad_in2), _p(grad_val), _p(grad_target), b, d, hi,
            wi, h, w, kernel_size, dilation, float(eps), _dt(x), _lib.GFLA_F32, 0, _stream(x)), "resample2d_cosine_bwd_nhwc")
    if need_input1:
        grad_in1 = _like_caller(_narrow(grad_in1, x.dtype), input1.is_contiguous())
    if need_target:
        grad_target = _like_caller(grad_target, target.is_contiguous())
    return grad_in1, grad_in2, grad_target


# --------------------------------------------------------------------------- fused local attention
ALGO = {"auto": 0, "gather": 1, "tile": 2}


def _feature_layout(t: torch.Tensor) -> int:
    """GFLA_NCHW for contiguous tensors, GFLA_NHWC for torch.channels_last ones (no copy either way)."""
    if t.is_contiguous():
        return _lib.GFLA_NCHW
    if t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last):
        return _lib.GFLA_NHWC
    raise AssertionError("feature tensors must be contiguous (NCHW) or channels_last")


def _like_layout(t: torch.Tensor, shape, layout: int) -> torch.Tensor:
    fmt = torch.channels_last if layout == _lib.GFLA_NHWC else torch.contiguous_format
    return torch.empty(shape, dtype=t.dtype, device=t.device, memory_format=fmt)


def local_attn_fwd(source, flow, logits, k, return_probs=False, algo="auto"):
    """source may be contiguous (NCHW) or channels_last; `out` comes back in the same memory format."""
    layout = _feature_layout(source)
    assert flow.is_contiguous() and logits.is_contiguous()
    _need_cuda(source, flow, logits)
    bs, ds, hs, ws = source.size()
    bf, df, h, w = flow.size()
    assert df == 2 and bf == bs
    assert logits.shape == (bs, k * k, h, w) and logits.dtype == source.dtype
    out = _like_layout(source, (bs, ds, h, w), layout)
    probs = torch.empty_like(logits) if return_probs else None
    with torch.cuda.device_of(source):
        _lib.check(_lib.lib().gfla_local_attn_fwd(_p(source), _p(flow), _p(logits), _p(out), _p(probs), bs, ds, hs, ws,
                                                  h, w, k, _dt(source), _dt(flow), layout, ALGO[algo], _stream(source)),
                   "local_attn_fwd")
    return (out, probs) if return_probs else out


def local_attn_blend_fwd(source, flow, logits, prev, mask, k, algo="auto"):
    """out = prev * (1 - mask) + local_attention(source, flow, logits) * mask, in one kernel (forward only).
    prev: [B,C,H,W] in the same memory format as source; mask: [B,1,H,W]."""
    layout = _feature_layout(source)
    assert _feature_layout(prev) == layout or prev.shape[1] == 1, "prev must use the same memory format as source"
    assert flow.is_contiguous() and logits.is_contiguous()
    mask = mask.contiguous()
    _need_cuda(source, flow, logits, prev, mask)
    bs, ds, hs, ws = source.size()
    _, _, h, w = flow.size()
    assert prev.shape == (bs, ds, h, w) and mask.shape == (bs, 1, h, w)
    assert prev.dtype == source.dtype and mask.dtype == source.dtype and logits.dtype == source.dtype
    out = _like_layout(source, (bs, ds, h, w), layout)
    with torch.cuda.device_of(source):
        _lib.check(_lib.lib().gfla_local_attn_blend_fwd(_p(source), _p(flow), _p(logits), _p(prev), _p(mask), _p(out), bs, ds,
                                                        hs, ws, h, w, k, _dt(source), _dt(flow), layout, ALGO[algo],
                                                        _stream(source)), "local_attn_blend_fwd")
    return out


def relayout(t: torch.Tensor, to_channels_last: bool) -> torch.Tensor:
    """Out-of-place NCHW <-> channels_last copy of a [B,C,H,W] tensor with the library's own transpose kernel."""
    _need_cuda(t)
    b, c, h, w = t.shape
    if to_channels_last:
        assert t.is_contiguous()
        out = torch.empty((b, c, h, w), dtype=t.dtype, device=t.device, memory_format=torch.channels_last)
    else:
        assert t.is_contiguous(memory_format=torch.channels_last)
        out = torch.empty((b, c, h, w), dtype=t.dtype, device=t.device)
    with torch.cuda.device_of(t):
        _lib.check(_lib.lib().gfla_relayout(_p(t), _p(out), b, c, h, w, _dt(t), 1 if to_channels_last else 0, _stream(t)),
                   "relayout")
    return out


def _tile_bwd_eligible(source, flow, k) -> bool:
    """what the backward tile kernels serve (mirrors local_attn_bwd_tc_supported in csrc/local_attn_bwd_tc.cu)"""
    c = source.shape[1]
    return (source.dtype == torch.bfloat16 and flow.dtype == torch.float32 and k in (3, 5)
            and (c % 256 == 0 or c in (64, 128)))


def local_attn_bwd(source, flow, logits, grad_out, k, algo="auto"):
    layout = _feature_layout(source)
    assert flow.is_contiguous() and logits.is_contiguous()
    _need_cuda(source, flow, logits, grad_out)
    if (layout == _lib.GFLA_NCHW and algo == "auto" and _tile_bwd_eligible(source, flow, k)
            and not source.is_contiguous(memory_format=torch.channels_last)):   # H=W=1 / C=1: both formats at once
        # The backward tile kernels are channels-last only (every operand must be channel-contiguous for TMA).
        # For planar callers, re-lay the two feature tensors (two extra passes over them) instead of falling
        # back to the scalar-atomics kernel: ~100x faster at cfg2.
        go = grad_out if grad_out.is_contiguous() else grad_out.contiguous()
        gs, gf, gl = local_attn_bwd(relayout(source, True), flow, logits, relayout(go, True), k, algo="auto")
        return relayout(gs, False), gf, gl
    fmt = torch.channels_last if layout == _lib.GFLA_NHWC else torch.contiguous_format
    grad_out = grad_out.contiguous(memory_format=fmt)
    bs, ds, hs, ws = source.size()
    _, _, h, w = flow.size()
    gs, gf, gl = _like_layout(source, source.shape, layout), torch.empty_like(flow), torch.empty_like(logits)
    with torch.cuda.device_of(source):
        # scratch for the fused kernel's in-kernel zero-fill of grad_source (per-sample counters; the library never allocates)
        nws = int(_lib.lib().gfla_local_attn_bwd_workspace_bytes(bs))
        wsb = torch.empty(max(nws, 4), dtype=torch.uint8, device=source.device)
        _lib.check(_lib.lib().gfla_local_attn_bwd_ws(_p(source), _p(flow), _p(logits), _p(grad_out), _p(gs), _p(gf), _p(gl),
                                                     bs, ds, hs, ws, h, w, k, _dt(source), _dt(flow), layout, 0, ALGO[algo],
                                                     _p(wsb), nws, _stream(source)), "local_attn_bwd")
    return gs, gf, gl
