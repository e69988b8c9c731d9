"""torch.autograd glue over the C ABI: tensors in, raw device pointers + current stream out.

PyTorch is plumbing here (device memory, streams, autograd graph); every arithmetic step of the hot
path runs in libkdcc.so.  Activations are kept NHWC-physical (torch.channels_last) so no transposes
are inserted around the kernels.

Reference call sites replaced (reference file:line):
  depthwise_conv      models/students/transform_blocks/depthwise_separable_conv.py:12
  pointwise_conv      models/students/transform_blocks/depthwise_separable_conv.py:13
  kd_loss             losses/KLDiv.py:19-23, losses/EnsembleKLDiv.py:18-22
  hint_loss           losses/WeightedHintMSELoss.py:12-16, losses/MSELoss.py:14-16
  cross_entropy       losses/CrossEntropy.py:10-15
  logits_stats        trainer/layerwise_trainer.py:225-227,244-250 (logged losses + confusion matrices, one pass)
"""
import os

import torch

from . import _abi

_DTYPES = {torch.float32: _abi.F32, torch.bfloat16: _abi.BF16}


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise _abi.KdccError("kdcc kernels need CUDA tensors (sm_100a); got a %s tensor -- there is no CPU fallback"
                                 % t.device.type)


def _dtype_code(t):
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise _abi.KdccError("kdcc supports float32 and bfloat16 activations, got %s" % t.dtype)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _device_guard(fn):
    """Run `fn` with the device of its first CUDA tensor argument current: kernels, TMA descriptors, function attributes
    and `_stream()` belong to the device the tensors live on, which need not be the current one (a process driving
    several devices, a model moved by hand).  Costs one `current_device()` query when the devices already agree."""
    import functools

    @functools.wraps(fn)
    def wrapped(*args, **kwargs):
        for a in args:
            if torch.is_tensor(a) and a.is_cuda:
                if a.device.index != torch.cuda.current_device():
                    with torch.cuda.device(a.device):
                        return fn(*args, **kwargs)
                break
        return fn(*args, **kwargs)
    return wrapped


def _ptr(t):
    return t.data_ptr() if t is not None else None


_WS = {}


def _workspace(nbytes, device):
    """Scratch for one kernel call.  One buffer per (device, stream), grown on demand and reused: launches on a stream
    are serialised, so the next call may overwrite what the previous one has finished with -- and the caching allocator
    is not asked twice per block and step."""
    nbytes = max(int(nbytes), 16)
    key = (device.index if device.index is not None else torch.cuda.current_device(), torch.cuda.current_stream(device).cuda_stream)
    buf = _WS.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = _WS[key] = torch.empty(nbytes, dtype=torch.uint8, device=device)
    return buf


_DISPATCH = {}


def _supported(op, N, H, W, C, Cout, k, dil, pad, layout, code):
    """kdcc_dispatch_name(...) != "unsupported", memoised (it is asked for every forward of every block)."""
    key = (op, N, H, W, C, Cout, k, dil, pad, layout, code)
    r = _DISPATCH.get(key)
    if r is None:
        r = _DISPATCH[key] = _abi.dispatch_name(*key) != "unsupported"
    return r


def _nhwc(t):
    """NCHW-logical tensor in NHWC-physical memory (no copy when it already is)."""
    return t.contiguous(memory_format=torch.channels_last)


def _empty_nhwc(n, c, h, w, like):
    return torch.empty((n, c, h, w), dtype=like.dtype, device=like.device, memory_format=torch.channels_last)


def _is_plain_nchw(t):
    """True for a dense NCHW tensor that is not also a valid channels_last view."""
    return t.dim() == 4 and t.is_contiguous() and not t.is_contiguous(memory_format=torch.channels_last)


def _is_channels_last(t):
    """True for a dense channels_last tensor that is not also plain NCHW."""
    return t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last) and not t.is_contiguous()


def _convertible(t):
    """kdcc_layout_convert takes bf16 with 16-byte rows in both layouts."""
    return t.dtype == torch.bfloat16 and t.dim() == 4 and t.shape[1] % 8 == 0 and (t.shape[2] * t.shape[3]) % 8 == 0


def _convert(t, to_nchw):
    """NHWC-physical -> NCHW-physical (or back) through kdcc_layout_convert; `t` must be dense in the source layout."""
    N, C, H, W = t.shape
    out = torch.empty((N, C, H, W), dtype=t.dtype, device=t.device,
                      memory_format=torch.contiguous_format if to_nchw else torch.channels_last)
    _abi.check(_abi.lib().kdcc_layout_convert(_ptr(t), _ptr(out), N, C, H * W, int(to_nchw), _dtype_code(t), _stream()),
               "kdcc_layout_convert")
    return out


def _format(t, layout):
    """`t` dense in `layout`; the bf16 re-layout runs in libkdcc (a tiled transpose at HBM speed), anything else in torch."""
    if layout == _abi.NCHW:
        if t.is_contiguous():
            return t
        return _convert(t, True) if (_is_channels_last(t) and _convertible(t)) else t.contiguous()
    if t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last):
        return t
    return _convert(t, False) if (_is_plain_nchw(t) and _convertible(t)) else _nhwc(t)


def _empty_like_layout(n, c, h, w, like, layout):
    if layout == _abi.NCHW:
        return torch.empty((n, c, h, w), dtype=like.dtype, device=like.device)
    return _empty_nhwc(n, c, h, w, like)


@_device_guard
def cast_weight(w_f32, dtype):
    """fp32 master parameter -> activation dtype through kdcc_cast_f32_to_bf16 (no torch arithmetic)."""
    if w_f32.dtype == dtype:
        return w_f32.contiguous()
    if w_f32.dtype != torch.float32 or dtype != torch.bfloat16:
        raise _abi.KdccError("kdcc keeps fp32 master weights and casts them to bf16 activations; got %s -> %s" % (w_f32.dtype, dtype))
    out = torch.empty(w_f32.shape, dtype=torch.bfloat16, device=w_f32.device)
    src = w_f32.contiguous()
    _abi.check(_abi.lib().kdcc_cast_f32_to_bf16(_ptr(src), _ptr(out), src.numel(), _stream()), "kdcc_cast_f32_to_bf16")
    return out


# bf16 copies of fp32 master weights, keyed by the parameter object: (parameter version, copy).  A forward reuses the copy
# while the parameter's version counter has not moved; kdcc.optim.RAdam rewrites the copy inside its fused step and
# re-stamps it (lp_refreshed), so a training loop never launches a cast after the first step.
import weakref

_LP = {}   # id(param) -> (weakref to param, version, copy); the weakref's callback drops the entry with the parameter


def _lp_entry(param):
    hit = _LP.get(id(param))
    return hit if hit is not None and hit[0]() is param else None


def _lp_store(param, lp):
    key = id(param)
    _LP[key] = (weakref.ref(param, lambda _r, key=key: _LP.pop(key, None)), param._version, lp)


def lp_weight(param, dtype):
    """The activation-dtype copy of `param` (an fp32 master weight), cached across calls."""
    if param.dtype == dtype:
        return param.detach()
    hit = _lp_entry(param)
    if hit is not None and hit[1] == param._version and hit[2].dtype == dtype and hit[2].device == param.device:
        return hit[2]
    lp = cast_weight(param.detach(), dtype)
    _lp_store(param, lp)
    return lp


def lp_copy_of(param):
    """The cached low-precision copy of `param`, or None (used by the fused optimizer step to refresh it in place)."""
    hit = _lp_entry(param)
    return hit[2] if hit is not None and hit[2].device == param.device else None


def lp_refreshed(param):
    """The optimizer has just rewritten param and its cached copy together: the copy is current for the new version."""
    hit = _lp_entry(param)
    if hit is not None:
        _lp_store(param, hit[2])


# ---------------------------------------------------------------------------------------------------
# depthwise
# ---------------------------------------------------------------------------------------------------
class _DepthwiseConv(torch.autograd.Function):
    @staticmethod
    @_device_guard
    def forward(ctx, x, weight, bias, k, dil, pad):
        _require_cuda(x, weight, bias)
        N, C, H, W = x.shape
        Ho, Wo = H + 2 * pad - dil * (k - 1), W + 2 * pad - dil * (k - 1)
        code = _dtype_code(x)
        # the reference's own NCHW layout runs on the tensor-core kernels (bf16); channels_last and fp32 run NHWC
        layout = _abi.NHWC
        in_cl = False
        if bias is None and _supported(0, N, H, W, C, C, k, dil, pad, _abi.NCHW, code):
            if _is_plain_nchw(x):
                layout = _abi.NCHW
            elif k > 3 and _is_channels_last(x) and _convertible(x) and not os.environ.get("KDCC_DW_KEEP_NHWC"):
                # a channels_last trunk: the large dilated kernels only reach tensor-core speed on channel planes, so the
                # input is re-laid at the block boundary (layout_convert.cu); 3x3 stays on the streaming NHWC kernels
                layout, in_cl = _abi.NCHW, True
        x = _format(x, layout)
        w = weight.detach().reshape(C, k * k).float().contiguous()
        b = bias.detach().float().contiguous() if bias is not None else None
        y = _empty_like_layout(N, C, Ho, Wo, x, layout)
        _abi.check(_abi.lib().kdcc_dw_fwd(_ptr(x), _ptr(w), _ptr(b), _ptr(y), N, H, W, C, k, dil, pad, layout,
                                          code, _stream()), "kdcc_dw_fwd")
        ctx.save_for_backward(x, w)
        ctx.geom = (k, dil, pad, bias is not None, weight.shape, layout)
        ctx.in_cl = in_cl
        ctx.wdtype = weight.dtype   # fp32 master weights normally; a model cast wholesale to bf16 gets its gradients in bf16
        return y

    @staticmethod
    @_device_guard
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        k, dil, pad, has_bias, wshape, layout = ctx.geom
        N, C, H, W = x.shape
        dy = _format(dy, layout)
        need_dx, need_dw, need_db = ctx.needs_input_grad[0], ctx.needs_input_grad[1], has_bias and ctx.needs_input_grad[2]
        dx = _empty_like_layout(N, C, H, W, x, layout) if need_dx else None
        dw = torch.empty((C, k * k), dtype=torch.float32, device=x.device) if need_dw else None
        db = torch.empty((C,), dtype=torch.float32, device=x.device) if need_db else None
        L = _abi.lib()
        code = _dtype_code(x)
        ws = _workspace(L.kdcc_dw_bwd_workspace_bytes(N, H, W, C, k, dil, pad, layout, code), x.device)
        _abi.check(L.kdcc_dw_bwd(_ptr(x), _ptr(w), _ptr(dy), _ptr(dx), _ptr(dw), _ptr(db), _ptr(ws), ws.numel(),
                                 N, H, W, C, k, dil, pad, layout, code, _stream()), "kdcc_dw_bwd")
        if need_dx and ctx.in_cl:
            dx = _convert(dx, False)   # the gradient goes back in the layout the input came in
        return dx, (dw.reshape(wshape).to(ctx.wdtype) if need_dw else None), db, None, None, None


def depthwise_conv(x, weight, bias, kernel_size, dilation, padding):
    """F.conv2d(x, weight (C,1,k,k), bias, stride=1, padding, dilation, groups=C) on libkdcc."""
    return _DepthwiseConv.apply(x, weight, bias, int(kernel_size), int(dilation), int(padding))


# ---------------------------------------------------------------------------------------------------
# pointwise
# ---------------------------------------------------------------------------------------------------
class _PointwiseConv(torch.autograd.Function):
    @staticmethod
    @_device_guard
    def forward(ctx, x, weight, bias, scale, shift, relu, residual=None, out_channels_last=False):
        _require_cuda(x, weight, bias)
        N, K, H, W = x.shape
        Co = weight.shape[0]
        M = N * H * W
        code = _dtype_code(x)
        layout = _abi.NHWC
        if _is_plain_nchw(x) and _supported(2, N, H, W, K, Co, 1, 1, 0, _abi.NCHW, code):
            layout = _abi.NCHW
            # planes in, channels_last out: the GEMM writes the caller's layout itself (no re-layout pass for y and dy)
            if out_channels_last and Co % 8 == 0 and _supported(2, N, H, W, K, Co, 1, 1, 0, _abi.PLANES_TO_NHWC, code):
                layout = _abi.PLANES_TO_NHWC
        x = _format(x, _abi.NCHW if layout == _abi.PLANES_TO_NHWC else layout)
        w = lp_weight(weight, x.dtype).reshape(Co, K)
        y = _empty_like_layout(N, Co, H, W, x, _abi.NHWC if layout == _abi.PLANES_TO_NHWC else layout)
        fused = scale is not None or shift is not None or relu
        eff_shift = shift
        if bias is not None and not fused:
            eff_shift = bias.detach().float().contiguous()
        elif bias is not None:
            raise _abi.KdccError("conv bias together with a fused BN epilogue is not supported; fold the bias into shift")
        use_act = fused or bias is not None or residual is not None
        if residual is not None:
            if residual.shape != y.shape:
                raise _abi.KdccError("residual %s does not match the output %s" % (tuple(residual.shape), tuple(y.shape)))
            res = _format(residual.detach().to(x.dtype), _abi.NHWC if layout == _abi.PLANES_TO_NHWC else layout)
            _abi.check(_abi.lib().kdcc_pw_fwd_residual(_ptr(x), _ptr(w), _ptr(scale), _ptr(eff_shift), _ptr(res), int(bool(relu)),
                                                       None, _ptr(y), M, K, Co, N, layout, code, _stream()), "kdcc_pw_fwd_residual")
        else:
            _abi.check(_abi.lib().kdcc_pw_fwd(_ptr(x), _ptr(w), _ptr(scale), _ptr(eff_shift), int(bool(relu)),
                                              None if use_act else _ptr(y), _ptr(y) if use_act else None,
                                              M, K, Co, N, layout, code, _stream()), "kdcc_pw_fwd")
        if out_channels_last and layout == _abi.NCHW and _convertible(y):
            y = _convert(y, False)          # hand the result back in the caller's (channels_last) layout
        if fused:
            ctx.mark_non_differentiable(y)  # inference-only epilogue (eval-mode BN fold)
        ctx.save_for_backward(x, w)
        ctx.meta = (bias is not None, weight.shape, layout)
        ctx.wdtype = weight.dtype
        ctx.has_residual = residual is not None
        return y

    @staticmethod
    @_device_guard
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        has_bias, wshape, layout = ctx.meta
        N, K, H, W = x.shape
        Co = w.shape[0]
        M = N * H * W
        mixed = layout == _abi.PLANES_TO_NHWC
        dy = _format(dy, _abi.NHWC if mixed else layout)
        L = _abi.lib()
        code = _dtype_code(x)
        st = _stream()
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = _empty_like_layout(N, K, H, W, x, _abi.NCHW if mixed else layout)
            _abi.check(L.kdcc_pw_bwd_dx(_ptr(dy), _ptr(w), _ptr(dx), None, 0, M, K, Co, N, layout, code, st), "kdcc_pw_bwd_dx")
        if ctx.needs_input_grad[1]:
            dw = torch.empty((Co, K), dtype=torch.float32, device=x.device)
            ws = _workspace(L.kdcc_pw_bwd_workspace_bytes(1, M, K, Co, code), x.device)
            _abi.check(L.kdcc_pw_bwd_dw(_ptr(dy), _ptr(x), _ptr(dw), _ptr(ws), ws.numel(), M, K, Co, N, layout, code, st),
                       "kdcc_pw_bwd_dw")
            dw = dw.reshape(wshape).to(ctx.wdtype)
        if has_bias and ctx.needs_input_grad[2]:
            db = torch.empty((Co,), dtype=torch.float32, device=x.device)
            dyr = _nhwc(dy)  # column sums are taken over the pixel-major view
            ws = _workspace(L.kdcc_colsum_workspace_bytes(M, Co), x.device)
            _abi.check(L.kdcc_colsum(_ptr(dyr), _ptr(db), _ptr(ws), ws.numel(), M, Co, code, st), "kdcc_colsum")
        # y = conv + residual: the shortcut receives the output gradient as it is
        dres = dy if (ctx.has_residual and ctx.needs_input_grad[6]) else None
        return dx, dw, db, None, None, None, dres, None


def pointwise_conv(x, weight, bias=None, scale=None, shift=None, relu=False, residual=None, out_channels_last=False):
    """F.conv2d(x, weight (Co,C,1,1), bias) on libkdcc; optional fused eval-mode BN (scale, shift) + ReLU, optional
    shortcut added in the epilogue (`out = convs(x); out.add_(shortcut)` of a residual block in one kernel;
    differentiable when no BN / ReLU is fused)."""
    return _PointwiseConv.apply(x, weight, bias, scale, shift, bool(relu), residual, bool(out_channels_last))


# ---------------------------------------------------------------------------------------------------
# losses
# ---------------------------------------------------------------------------------------------------
def _take_grad(ctx):
    """The loss kernels emit d loss / d input in the forward pass; backward scales that buffer in place and hands it
    out, so it can be consumed once.  A second backward through the same node (retain_graph=True, or one loss tensor
    used in two graphs) raises instead of silently returning no gradient."""
    if getattr(ctx, "consumed", False):
        raise _abi.KdccError("this kdcc loss was already back-propagated; its fused gradient buffer is consumed by the first "
                             "backward -- call the criterion again instead of backward(retain_graph=True)")
    ds = ctx.ds
    ctx.ds = None
    ctx.consumed = ds is not None
    return ds


def _logit_strides(t):
    """(N, C, HW, batch_stride, class_stride, pixel_stride) of a (N,C,*spatial) tensor, or None."""
    N, C = t.shape[0], t.shape[1]
    HW = 1
    for d in t.shape[2:]:
        HW *= d
    if t.is_contiguous():
        return N, C, HW, C * HW, HW, 1
    if t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last):
        return N, C, HW, HW * C, 1, C
    return None


class _KdLoss(torch.autograd.Function):
    @staticmethod
    @_device_guard
    def forward(ctx, s, t, temperature, target_is_prob, expected=1.0):
        _require_cuda(s, t)
        if s.shape != t.shape or s.dim() < 2:
            raise _abi.KdccError("kd loss expects matching (N, C, ...) tensors, got %s and %s" % (tuple(s.shape), tuple(t.shape)))
        s = s.detach()
        if s.dim() == 4 and s.is_contiguous(memory_format=torch.channels_last) and not s.is_contiguous():
            fmt = torch.channels_last
        else:
            fmt = torch.contiguous_format
            s = s.contiguous()
        t = t.detach().to(s.dtype).contiguous(memory_format=fmt)
        geo = _logit_strides(s)
        N, C, HW, bs, cs, ps = geo
        need_grad = ctx.needs_input_grad[0]
        ds = torch.empty_like(s) if need_grad else None
        loss = torch.empty((), dtype=torch.float32, device=s.device)
        L = _abi.lib()
        ws = _workspace(L.kdcc_loss_workspace_bytes(), s.device)
        _abi.check(L.kdcc_kd_loss(_ptr(s), _ptr(t), _ptr(ds), _ptr(loss), _ptr(ws), ws.numel(), N, C, HW, bs, cs, ps,
                                  float(temperature), int(bool(target_is_prob)), _dtype_code(s), float(expected), _stream()),
                   "kdcc_kd_loss")
        ctx.ds = ds
        ctx.expected = float(expected)
        return loss

    @staticmethod
    @_device_guard
    def backward(ctx, g):
        ds = _take_grad(ctx)
        if ds is None:
            return None, None, None, None, None
        g = g.detach().float().contiguous()
        _abi.check(_abi.lib().kdcc_scale_inplace_expect(_ptr(ds), _ptr(g), ctx.expected, ds.numel(), _dtype_code(ds), _stream()),
                   "kdcc_scale_inplace_expect")
        return ds, None, None, None, None


def kd_loss(inputs, targets, temperature=1.0, target_is_prob=False, expected_upstream=1.0):
    """T^2/(N*HW) * sum_pix KL(p_t || softmax(inputs/T)); fp32 0-dim tensor with grad_fn.
    `expected_upstream`: the value autograd is expected to hand to this node's backward (1 for `loss.backward()`,
    1/accumulation_steps for `(sum of losses / accumulation_steps).backward()`).  It is folded into the gradient the
    forward kernel emits; backward verifies it on the device and rescales only if it differs, so it is a performance
    hint, never a correctness assumption."""
    return _KdLoss.apply(inputs, targets, float(temperature), bool(target_is_prob), float(expected_upstream))


class _KdLossMulti(torch.autograd.Function):
    @staticmethod
    @_device_guard
    def forward(ctx, s, temperature, weights, expected, *teachers):
        import ctypes
        _require_cuda(s, *teachers)
        K = len(teachers)
        if K == 0 or K != len(weights):
            raise _abi.KdccError("kd_loss_multi needs one weight per teacher (got %d teachers, %d weights)" % (K, len(weights)))
        for t in teachers:
            if t.shape != s.shape:
                raise _abi.KdccError("kd_loss_multi expects matching (N, C, ...) tensors, got %s and %s" % (tuple(s.shape), tuple(t.shape)))
        s = s.detach()
        if s.dim() == 4 and s.is_contiguous(memory_format=torch.channels_last) and not s.is_contiguous():
            fmt = torch.channels_last
        else:
            fmt = torch.contiguous_format
            s = s.contiguous()
        ts = [t.detach().to(s.dtype).contiguous(memory_format=fmt) for t in teachers]
        N, C, HW, bs, cs, ps = _logit_strides(s)
        need_grad = ctx.needs_input_grad[0]
        ds = torch.empty_like(s) if need_grad else None
        loss = torch.empty((), dtype=torch.float32, device=s.device)
        L = _abi.lib()
        ws = _workspace(L.kdcc_loss_workspace_bytes(), s.device)
        ptrs = (ctypes.c_void_p * K)(*[t.data_ptr() for t in ts])
        wts = (ctypes.c_float * K)(*[float(w) for w in weights])
        _abi.check(L.kdcc_kd_loss_multi(_ptr(s), ptrs, wts, K, _ptr(ds), _ptr(loss), _ptr(ws), ws.numel(), N, C, HW, bs, cs, ps,
                                        float(temperature), _dtype_code(s), float(expected), _stream()), "kdcc_kd_loss_multi")
        ctx.ds = ds
        ctx.K = K
        ctx.expected = float(expected)
        return loss

    @staticmethod
    @_device_guard
    def backward(ctx, g):
        ds = _take_grad(ctx)
        if ds is None:
            return (None,) * (4 + ctx.K)
        g = g.detach().float().contiguous()
        _abi.check(_abi.lib().kdcc_scale_inplace_expect(_ptr(ds), _ptr(g), ctx.expected, ds.numel(), _dtype_code(ds), _stream()),
                   "kdcc_scale_inplace_expect")
        return (ds,) + (None,) * (3 + ctx.K)


def kd_loss_multi(inputs, teachers, weights, temperature=1.0, expected_upstream=1.0):
    """sum_k weights[k] * T^2/(N*HW) * sum_pix KL(softmax(teachers[k]/T) || softmax(inputs/T)) in one pass over the
    student logits (trainer/ensemble_trainer.py:76-83); fp32 0-dim tensor with grad_fn."""
    teachers = list(teachers)
    return _KdLossMulti.apply(inputs, float(temperature), tuple(float(w) for w in weights), float(expected_upstream), *teachers)


class _HintLoss(torch.autograd.Function):
    @staticmethod
    @_device_guard
    def forward(ctx, s, t, weight, scale, expected=1.0):
        _require_cuda(s, t, weight)
        if s.shape != t.shape or s.dim() < 2:
            raise _abi.KdccError("hint loss expects matching (N, C, ...) tensors, got %s and %s" % (tuple(s.shape), tuple(t.shape)))
        s = s.detach()
        N, C = s.shape[0], s.shape[1]
        HW = s.numel() // max(N * C, 1)
        if s.dim() == 4 and s.is_contiguous(memory_format=torch.channels_last) and not s.is_contiguous():
            layout = _abi.NHWC
            t = t.detach().to(s.dtype).contiguous(memory_format=torch.channels_last)
        else:
            layout = _abi.NCHW
            s = s.contiguous()
            t = t.detach().to(s.dtype).contiguous()
        w = None
        per_sample = 0
        if weight is not None:
            w = weight.detach().float().contiguous()
            if w.dim() == 2 and w.shape == (N, C):
                per_sample = 1
            elif w.numel() != C:
                raise _abi.KdccError("filter_weight must have shape (C,) or (N, C)")
        need_grad = ctx.needs_input_grad[0]
        ds = torch.empty_like(s) if need_grad else None
        loss = torch.empty((), dtype=torch.float32, device=s.device)
        L = _abi.lib()
        ws = _workspace(L.kdcc_loss_workspace_bytes() + 4 * N * C, s.device)
        _abi.check(L.kdcc_hint_loss(_ptr(s), _ptr(t), _ptr(w), per_sample, _ptr(ds), _ptr(loss), _ptr(ws), ws.numel(),
                                    N, C, HW, layout, float(scale), _dtype_code(s), float(expected), _stream()), "kdcc_hint_loss")
        ctx.ds = ds
        ctx.expected = float(expected)
        return loss

    @staticmethod
    @_device_guard
    def backward(ctx, g):
        ds = _take_grad(ctx)
        if ds is None:
            return None, None, None, None, None
        g = g.detach().float().contiguous()
        _abi.check(_abi.lib().kdcc_scale_inplace_expect(_ptr(ds), _ptr(g), ctx.expected, ds.numel(), _dtype_code(ds), _stream()),
                   "kdcc_scale_inplace_expect")
        return ds, None, None, None, None


def hint_loss(inputs, targets, filter_weight=None, scale=1.0, expected_upstream=1.0):
    """scale/N * sum_n [sum_c w mean_hw (s-t)^2 / sum_c w]; filter_weight None = uniform (MSELoss).
    `expected_upstream`: see kd_loss."""
    return _HintLoss.apply(inputs, targets, filter_weight, float(scale), float(expected_upstream))


def _ce_operands(s, target, weight, bad_labels):
    """(s dense NCHW or channels_last, int64 labels (N*HW), fp32 weight or None, geometry) for the CE entry points."""
    if s.dim() < 2:
        raise _abi.KdccError("cross entropy expects (N, C, ...) logits, got %s" % (tuple(s.shape),))
    s = s.detach()
    if not (s.dim() == 4 and s.is_contiguous(memory_format=torch.channels_last) and not s.is_contiguous()):
        s = s.contiguous()
    geo = _logit_strides(s)
    N, C, HW = geo[0], geo[1], geo[2]
    target = target.detach()
    if target.dtype != torch.int64:
        target = target.long()
    target = target.contiguous()
    if target.numel() != N * HW:
        raise _abi.KdccError("labels have %d elements, logits describe %d pixels" % (target.numel(), N * HW))
    w = None
    if weight is not None:
        w = weight.detach().float().contiguous()
        if w.numel() != C:
            raise _abi.KdccError("class weight has %d entries, logits have %d classes" % (w.numel(), C))
    if bad_labels is not None and (bad_labels.dtype != torch.int64 or bad_labels.numel() != 1):
        raise _abi.KdccError("bad_labels must be a one-element int64 device tensor")
    return s, target, w, geo


class _CeLoss(torch.autograd.Function):
    @staticmethod
    @_device_guard
    def forward(ctx, s, target, weight, ignore_index, mean, expected, bad_labels):
        _require_cuda(s, target, weight, bad_labels)
        s, target, w, (N, C, HW, bs, cs, ps) = _ce_operands(s, target, weight, bad_labels)
        ds = torch.empty_like(s) if ctx.needs_input_grad[0] else None
        loss = torch.empty((), dtype=torch.float32, device=s.device)
        L = _abi.lib()
        ws = _workspace(L.kdcc_ce_workspace_bytes(N, HW), s.device)
        _abi.check(L.kdcc_ce_loss(_ptr(s), _ptr(target), _ptr(w), int(ignore_index), int(bool(mean)), _ptr(ds), _ptr(loss),
                                  _ptr(bad_labels), _ptr(ws), ws.numel(), N, C, HW, bs, cs, ps, _dtype_code(s), float(expected),
                                  _stream()), "kdcc_ce_loss")
        ctx.ds = ds
        ctx.expected = float(expected)
        return loss

    @staticmethod
    @_device_guard
    def backward(ctx, g):
        ds = _take_grad(ctx)
        if ds is None:
            return None, None, None, None, None, None, None
        g = g.detach().float().contiguous()
        _abi.check(_abi.lib().kdcc_scale_inplace_expect(_ptr(ds), _ptr(g), ctx.expected, ds.numel(), _dtype_code(ds), _stream()),
                   "kdcc_scale_inplace_expect")
        return ds, None, None, None, None, None, None


def cross_entropy(logits, target, weight=None, ignore_index=255, mean=True, expected_upstream=1.0, bad_labels=None):
    """losses/CrossEntropy.py:10-15: NLL of log_softmax(logits, 1) at the labels, weighted by weight[label], over the
    pixels whose label is a class index other than ignore_index; mean=True divides by the summed weight (NaN when no
    pixel counts, as torch), mean=False returns the sum.  fp32 0-dim tensor with grad_fn; one kernel pass (plus a
    pre-pass over the labels when a mean-mode gradient is needed).  Labels outside [0, C) other than ignore_index are
    dropped, never used as an index, and added to `bad_labels` (one-element int64 device tensor) when given.
    `expected_upstream`: see kd_loss."""
    return _CeLoss.apply(logits, target, weight, int(ignore_index), bool(mean), float(expected_upstream), bad_labels)


def _conf_arg(conf, C):
    if conf is None:
        return None
    _require_cuda(conf)
    if conf.dtype != torch.int64 or not conf.is_contiguous() or conf.numel() != C * C:
        raise _abi.KdccError("confusion accumulator must be a contiguous int64 tensor of %d cells" % (C * C))
    return conf


@torch.no_grad()
@_device_guard
def logits_stats(s, t, target, weight=None, ignore_index=255, mean=True, kd_mode=0, temperature=1.0, kd_scale=1.0,
                 conf_s=None, conf_t=None, bad_labels=None):
    """The logged-only quantities of one layerwise step (trainer/layerwise_trainer.py:225-227,244-250) in one pass over
    the student logits `s`, the teacher logits `t` and the labels: returns (kd, ce_s, ce_t), 0-dim fp32 device tensors
    (views of one buffer; nothing is read back to the host).
      kd   = kd_mode 1: KLDivergenceLoss(temperature)(s, t); 2: MSELoss(num_classes=kd_scale)(s, t); 0: None
      ce_s = cross_entropy(s, target, weight, ignore_index, mean), ce_t the same for t
    conf_s / conf_t (int64 C*C, device) += the confusion matrices of argmax(s) / argmax(t), as confusion_update.
    t=None (validation): only ce_s and conf_s; kd and ce_t are None."""
    _require_cuda(s, t, target, weight, conf_s, conf_t, bad_labels)
    s, target, w, (N, C, HW, bs, cs, ps) = _ce_operands(s, target, weight, bad_labels)
    if t is not None:
        if t.shape != s.shape:
            raise _abi.KdccError("logits_stats expects matching (N, C, ...) tensors, got %s and %s" % (tuple(s.shape), tuple(t.shape)))
        t = t.detach().to(s.dtype).contiguous(memory_format=torch.channels_last if ps != 1 else torch.contiguous_format)
    else:
        kd_mode, conf_t = 0, None
    conf_s, conf_t = _conf_arg(conf_s, C), _conf_arg(conf_t, C)
    out3 = torch.empty(3, dtype=torch.float32, device=s.device)
    L = _abi.lib()
    ws = _workspace(L.kdcc_ce_workspace_bytes(N, HW), s.device)
    _abi.check(L.kdcc_logits_stats(_ptr(s), _ptr(t), _ptr(target), _ptr(w), int(ignore_index), int(bool(mean)), int(kd_mode),
                                   float(temperature), float(kd_scale), _ptr(out3), _ptr(conf_s), _ptr(conf_t), _ptr(bad_labels),
                                   _ptr(ws), ws.numel(), N, C, HW, bs, cs, ps, _dtype_code(s), _stream()), "kdcc_logits_stats")
    return (out3[0] if kd_mode else None), out3[1], (out3[2] if t is not None else None)


# ---------------------------------------------------------------------------------------------------
# segmentation metric (SURVEY.md 8f n1)
# ---------------------------------------------------------------------------------------------------
@torch.no_grad()
@_device_guard
def confusion_update(conf, logits, target, ignore_index=255):
    """conf (C*C int64, device) += confusion matrix of argmax(logits, 1) against target -- utils/util.py:108-128.
    One kernel pass over the logits and labels; nothing is copied to the host."""
    _require_cuda(conf, logits, target)
    if conf.dtype != torch.int64 or not conf.is_contiguous():
        raise _abi.KdccError("confusion_update needs a contiguous int64 accumulator")
    N, C = logits.shape[0], logits.shape[1]
    if conf.numel() != C * C:
        raise _abi.KdccError("accumulator has %d cells, logits have %d classes" % (conf.numel(), C))
    logits = logits.detach().contiguous()
    target = target.detach()
    if target.dtype != torch.int64:
        target = target.long()
    target = target.contiguous()
    HW = logits.numel() // max(1, N * C)
    if target.numel() != N * HW:
        raise _abi.KdccError("labels have %d elements, logits describe %d pixels" % (target.numel(), N * HW))
    _abi.check(_abi.lib().kdcc_confusion_update(_ptr(logits), _ptr(target), _ptr(conf), N, C, HW, C * HW, HW, int(ignore_index),
                                                _dtype_code(logits), _stream()), "kdcc_confusion_update")
    return conf


# ---------------------------------------------------------------------------------------------------
# sliding-window test-time inference (SURVEY.md 8f n4)
# ---------------------------------------------------------------------------------------------------
_COUNT_MODES = {"reference": 0, "coverage": 1}


@torch.no_grad()
@_device_guard
def tta_stitch(windows, coords, h, w, out, flip=False, count_mode="reference", alpha=1.0, accumulate=False):
    """out (C, h, w) fp32 (+)= alpha * overlap-add of `windows` (n, C, th, tw) placed at `coords` (n, 4) int32 device
    tensor of (x1, y1, x2, y2), divided by the window counter -- utils/tta_process.py:39-52; flip=True un-mirrors the
    stitched map (the np.fliplr of :19-20).  count_mode "reference" keeps the reference's counter as written."""
    _require_cuda(windows, coords, out)
    if windows.dtype != torch.float32 or out.dtype != torch.float32 or coords.dtype != torch.int32:
        raise _abi.KdccError("tta_stitch needs fp32 windows / output and int32 coordinates")
    if not (windows.is_contiguous() and out.is_contiguous() and coords.is_contiguous()):
        raise _abi.KdccError("tta_stitch needs contiguous tensors")
    n, C, th, tw = windows.shape
    if coords.numel() != 4 * n or out.numel() != C * h * w:
        raise _abi.KdccError("tta_stitch: %d windows of %d classes do not match coords %s / output %s"
                             % (n, C, tuple(coords.shape), tuple(out.shape)))
    _abi.check(_abi.lib().kdcc_tta_stitch(_ptr(windows), _ptr(coords), n, C, th, tw, int(h), int(w), int(bool(flip)),
                                          _COUNT_MODES[count_mode], float(alpha), _ptr(out), int(bool(accumulate)), _stream()),
               "kdcc_tta_stitch")
    return out


@torch.no_grad()
@_device_guard
def resize_bilinear(src, out, alpha=1.0, accumulate=False):
    """out (C, H, W) (+)= alpha * cv2.INTER_LINEAR resize of every plane of src (C, h, w) -- utils/tta_process.py:29-36."""
    _require_cuda(src, out)
    if src.dtype != torch.float32 or out.dtype != torch.float32 or not (src.is_contiguous() and out.is_contiguous()):
        raise _abi.KdccError("resize_bilinear needs contiguous fp32 tensors")
    C, h, w = src.shape
    if out.shape[0] != C:
        raise _abi.KdccError("resize_bilinear: %d source planes, %d destination planes" % (C, out.shape[0]))
    _abi.check(_abi.lib().kdcc_resize_bilinear(_ptr(src), C, h, w, _ptr(out), out.shape[1], out.shape[2], float(alpha),
                                               int(bool(accumulate)), _stream()), "kdcc_resize_bilinear")
    return out
