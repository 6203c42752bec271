"""Head post-processing that feeds Detect / MultiBoxLoss (SURVEY 8f rank 1).

The reference does this inline in every model's forward (pyramid.py:291-309 and :331-332, same code in
pyramid_mobile_try1.py:297-327 and pyramid_mb2_try3/4/5.py): per pyramid level the 4-channel confidence map is
reduced to (neg, pos) by max-in-out, both maps are permuted NCHW -> NHWC, flattened and concatenated over the
levels into loc[B,N,4] / conf[B,N,2], and the test phase applies a 2-way softmax before Detect.

`heads_to_loc_conf` materialises exactly those tensors with one kernel and is differentiable; `Detect.detect_heads`
(detection.py here) and `MultiBoxLoss.forward_heads` (multibox_loss.py) skip the materialisation altogether.  No CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import torch

from ... import _lib


class HeadMap(C.Structure):
    """fdt_head_map / fdt_head_grad_map (include/fdt_b200.h): element (b, ch, y, x) at data[b*bs + ch*cs + (y*W + x)*ps]"""
    _fields_ = [("data", C.c_void_p), ("batch_stride", C.c_int64), ("channel_stride", C.c_int64), ("pixel_stride", C.c_int64)]


DTYPES = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}       # FDT_DTYPE_*


def map_layout(m):
    """'nchw' or 'channels_last' if the kernels can read the [B,4,H,W] map `m` in place (dense in either memory format, any storage
    offset; size-1 dimensions have no meaningful stride), else None"""
    if m.dim() != 4:
        return None
    if m.is_contiguous():
        return "nchw"
    if m.is_contiguous(memory_format=torch.channels_last):
        return "channels_last"
    return None


def native_dtype(loc_maps, conf_maps):
    """the FDT_DTYPE_* code when every map can be passed as it is (one dtype in fp32 / bf16 / fp16, one device, each map dense NCHW
    or dense channels_last), else None: the maps are then converted to fp32 NCHW first"""
    maps = [*conf_maps, *(loc_maps if loc_maps is not None else ())]
    dt, dev = maps[0].dtype, maps[0].device
    if dt not in DTYPES or any(m.dtype != dt or m.device != dev or map_layout(m) is None for m in maps):
        return None
    return DTYPES[dt]


def map_descs(maps):
    """HeadMap array of `maps` (dense NCHW or channels_last, see map_layout) with the strides their layout implies"""
    d = (HeadMap * len(maps))()
    for l, m in enumerate(maps):
        hw = int(m.size(2)) * int(m.size(3))
        cs, ps = (hw, 1) if map_layout(m) == "nchw" else (1, 4)
        d[l] = HeadMap(m.data_ptr(), 4 * hw, cs, ps)
    return d


def _head_args(loc_maps, conf_maps, neg_max, native=True):
    """-> (device, B, N, (conf maps, loc maps) as the kernels read them, ctypes arguments of the C ABI's `_ex` entries:
    (loc descriptors, conf descriptors, dtype, f_h, f_w, neg_max, L)).  Maps the kernels can read in place (native_dtype) are
    passed as they are; anything else -- and everything with native=False -- is converted to fp32 NCHW."""
    _lib.require_cuda()
    L = len(conf_maps)
    if L == 0 or (loc_maps is not None and len(loc_maps) != L):
        raise ValueError("heads: need one loc map and one conf map per pyramid level")
    dev = conf_maps[0].device
    if not conf_maps[0].is_cuda:
        raise ValueError("heads: the maps must be CUDA tensors (there is no CPU path)")
    B = conf_maps[0].size(0)
    dt = native_dtype(loc_maps, conf_maps) if native else None
    if dt is not None:
        conf = list(conf_maps)
        loc = list(loc_maps) if loc_maps is not None else None
    else:
        dt = DTYPES[torch.float32]
        conf = [_lib.dev_f32(m, dev) for m in conf_maps]
        loc = [_lib.dev_f32(m, dev) for m in loc_maps] if loc_maps is not None else None
    for l, m in enumerate(conf):
        if m.dim() != 4 or m.size(1) != 4 or m.size(0) != B:
            raise ValueError(f"heads: conf map {l} must be [B,4,H,W], got {tuple(m.shape)}")
        if loc is not None and tuple(loc[l].shape) != tuple(m.shape):
            raise ValueError(f"heads: loc map {l} must match the conf map {tuple(m.shape)}, got {tuple(loc[l].shape)}")
    if neg_max is None:
        neg_max = [1] + [0] * (L - 1)                    # level 0: three negatives, the others three positives
    fh = (C.c_int * L)(*[int(m.size(2)) for m in conf])
    fw = (C.c_int * L)(*[int(m.size(3)) for m in conf])
    nm = (C.c_int * L)(*[int(bool(v)) for v in neg_max])
    cd = map_descs(conf)
    ld = map_descs(loc) if loc is not None else None
    N = sum(int(m.size(2)) * int(m.size(3)) for m in conf)
    return dev, B, N, (conf, loc), (ld, cd, dt, fh, fw, nm, L)


def _level_args(loc_maps, conf_maps, neg_max):
    """_head_args for the entries without `_ex`: the maps converted to fp32 NCHW, passed as host arrays of device pointers
    -> (device, B, N, (conf, loc), (loc pointers, conf pointers, f_h, f_w, neg_max, L))"""
    dev, B, N, (conf, loc), (_, _, _, fh, fw, nm, L) = _head_args(loc_maps, conf_maps, neg_max, native=False)
    cp = (C.c_void_p * L)(*[m.data_ptr() for m in conf])
    lp = (C.c_void_p * L)(*[m.data_ptr() for m in loc]) if loc is not None else None
    return dev, B, N, (conf, loc), (lp, cp, fh, fw, nm, L)


def _map_grads(maps, needed):
    """gradient buffers like `maps` (their dtype, shape and memory format; None where not needed) and their descriptors"""
    if not needed:
        return None, None
    g = [torch.empty_like(m) for m in maps]
    return g, map_descs(g)


class _HeadsToLocConfFn(torch.autograd.Function):
    """heads_to_loc_conf with a backward: loc rows copied into the loc maps, conf rows (through the softmax's backward when it
    was applied) routed into the conf maps the way torch's chunk / max / cat backward routes them."""

    @staticmethod
    def forward(ctx, neg_max, softmax, L, *maps):
        loc_maps, conf_maps = maps[:L], maps[L:]
        dev, B, N, (conf, loc), (ld, cd, dt, fh, fw, nm, _) = _head_args(loc_maps, conf_maps, neg_max)
        with torch.cuda.device(dev):
            loc_out = torch.empty((B, N, 4), dtype=torch.float32, device=dev)
            conf_out = torch.empty((B, N, 2), dtype=torch.float32, device=dev)
            _lib.check(_lib.lib().fdt_heads_to_loc_conf_ex(ld, cd, dt, fh, fw, nm, L, B, 1 if softmax else 0,
                                                           _lib.ptr(loc_out), _lib.ptr(conf_out), _lib.stream_ptr()))
        ctx.save_for_backward(*conf)
        ctx.level = (fh, fw, nm, L, B, softmax, dev, dt)
        return loc_out, conf_out

    @staticmethod
    def backward(ctx, g_loc, g_conf):
        conf = ctx.saved_tensors
        fh, fw, nm, L, B, softmax, dev, dt = ctx.level
        need_loc, need_conf = any(ctx.needs_input_grad[3:3 + L]), any(ctx.needs_input_grad[3 + L:])
        gl_maps, gld = _map_grads(conf, need_loc)                # (loc maps have the conf maps' shape, dtype and layout)
        gc_maps, gcd = _map_grads(conf, need_conf)
        gl = _lib.dev_f32(g_loc, dev) if need_loc else None
        gc = _lib.dev_f32(g_conf, dev) if need_conf else None
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().fdt_heads_to_loc_conf_backward_ex(map_descs(conf), dt, fh, fw, nm, L, B, 1 if softmax else 0,
                                                                    _lib.ptr(gl), _lib.ptr(gc), gld, gcd, _lib.stream_ptr()))
        return (None, None, None, *(gl_maps or [None] * L), *(gc_maps or [None] * L))


def heads_to_loc_conf(loc_maps, conf_maps, neg_max=None, softmax=True):
    """Per-level NCHW maps -> (loc[B,N,4], conf[B,N,2]) as pyramid.py:291-309 builds them; softmax=True also
    applies nn.Softmax(dim=-1) (:332, test phase), softmax=False keeps the raw logits MultiBoxLoss consumes.
    Differentiable: when a map requires grad, backward writes the gradients of the maps (those of the max-in-out
    reduction go where torch's max(dim) backward sends them)."""
    if torch.is_grad_enabled() and any(m.requires_grad for m in (*loc_maps, *conf_maps)):
        L = len(conf_maps)
        if len(loc_maps) != L:
            raise ValueError("heads: need one loc map and one conf map per pyramid level")
        nmx = None if neg_max is None else tuple(int(bool(v)) for v in neg_max)
        return _HeadsToLocConfFn.apply(nmx, bool(softmax), L, *loc_maps, *conf_maps)
    dev, B, N, keep, (ld, cd, dt, fh, fw, nm, L) = _head_args(loc_maps, conf_maps, neg_max)
    with torch.cuda.device(dev):
        loc = torch.empty((B, N, 4), dtype=torch.float32, device=dev)
        conf = torch.empty((B, N, 2), dtype=torch.float32, device=dev)
        _lib.check(_lib.lib().fdt_heads_to_loc_conf_ex(ld, cd, dt, fh, fw, nm, L, B, 1 if softmax else 0,
                                                       _lib.ptr(loc), _lib.ptr(conf), _lib.stream_ptr()))
    del keep
    return loc, conf
