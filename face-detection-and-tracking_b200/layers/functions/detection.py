"""Detect -- drop-in for layers/functions/detection.py:9-84 on hand-written sm_100a kernels."""
from __future__ import annotations

import ctypes as C
import threading
import weakref

import torch

from ... import _lib
from ...data import face as cfg

_host_ctx = threading.local()


def _ctx(device_index: int):
    """One fdt_ctx (stream + device staging buffers) per host thread and device."""
    d = getattr(_host_ctx, "ctx", None)
    if d is None:
        d = _host_ctx.ctx = {}
    if device_index not in d:
        h = C.c_void_p()
        _lib.check(_lib.lib().fdt_ctx_create(device_index, C.byref(h)))
        d[device_index] = h
        f = weakref.finalize(threading.current_thread(), _lib.lib().fdt_ctx_destroy, h)  # freed when the owning thread goes away
        f.atexit = False                                                                 # (not at interpreter exit: CUDA may be gone)
    return d[device_index]


class Detect:
    """At test time, Detect is the final layer of SSD: decode, threshold, top-k, NMS (detection.py:9-14).

    Same constructor, attributes and call signature as the reference.  CUDA inputs are processed in
    place on the current stream (asynchronous, CUDA-graph capturable) and the result is a CUDA tensor;
    consecutive calls on one stream overlap on the device (the instance owns a ring of scratch slots per
    stream and shape; completion stays in stream order, see fdt_detect in include/fdt_b200.h);
    CPU inputs go through fdt_detect_host (H2D copy, kernels, D2H copy) and the result is a CPU tensor,
    like the reference's torch.zeros(...) output on a CPU default device (detection.py:48).
    """

    def __init__(self, num_classes, bkg_label, top_k, conf_thresh, nms_thresh):
        self.num_classes = num_classes
        self.background_label = bkg_label
        self.top_k = top_k
        self.nms_thresh = nms_thresh
        if nms_thresh <= 0:
            raise ValueError('nms_threshold must be non negative.')      # detection.py:28-29
        self.conf_thresh = conf_thresh
        self.variance = cfg['variance']
        self.nms_top_k = 5000                                            # detection.py:32
        self._workspaces = _lib.DetectWorkspaces()                       # stateful scratch, one per (device, stream, shape)

    def __call__(self, loc_data, conf_data, prior_data, return_aux=False):
        """loc_data [B,N,4] (or [B,N*4]), conf_data [B,N,C] (or [B*N,C]) post-softmax, prior_data [N,4]
        -> output [B, num_classes, top_k, 5] rows [score, x1, y1, x2, y2].
        return_aux=True additionally returns (counts[B,C] int32, kept_prior[B,C,top_k] int64)."""
        _lib.require_cuda()
        num = loc_data.size(0)
        num_priors = prior_data.size(0)
        C_ = self.num_classes
        args = (num, num_priors, C_, int(self.top_k), int(self.nms_top_k), float(self.conf_thresh),
                float(self.nms_thresh), float(self.variance[0]), float(self.variance[1]))
        if not loc_data.is_cuda:
            return self._call_host(loc_data, conf_data, prior_data, args, return_aux)
        dev = loc_data.device
        with torch.cuda.device(dev):
            loc = _lib.dev_f32(loc_data, dev).view(num, num_priors, 4)
            conf = _lib.dev_f32(conf_data, dev).view(num, num_priors, C_)
            pri = _lib.dev_f32(prior_data, dev).view(num_priors, 4)
            out = torch.empty((num, C_, self.top_k, 5), dtype=torch.float32, device=dev)
            counts = torch.empty((num, C_), dtype=torch.int32, device=dev) if return_aux else None
            kept = torch.empty((num, C_, self.top_k), dtype=torch.int64, device=dev) if return_aux else None
            L = _lib.lib()
            ws = self._workspaces.get(num, num_priors, C_, dev)
            _lib.check(L.fdt_detect(_lib.ptr(loc), _lib.ptr(conf), _lib.ptr(pri), *args, _lib.ptr(out),
                                    _lib.ptr(counts), _lib.ptr(kept), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
        return (out, counts, kept) if return_aux else out

    def detect_heads(self, loc_maps, conf_maps, prior_data, neg_max=None, return_aux=False):
        """Detect straight from the models' per-level NCHW prediction maps (loc_l[B,4,H,W], 4-channel max-in-out
        conf_l[B,4,H,W]): the max-in-out reduction, NHWC permute/concat and the 2-way softmax of
        pyramid.py:291-309, 331-332 are fused into the threshold kernel, and NMS gathers the loc rows it decodes
        from the maps -- loc[B,N,4] / conf[B,N,2] are never materialised.  Same output as
        self(*heads_to_loc_conf(loc_maps, conf_maps), prior_data)."""
        from .heads import _head_args
        dev, num, num_priors, keep, (ld, cd, dt, fh, fw, nm, L) = _head_args(loc_maps, conf_maps, neg_max)
        if self.num_classes != 2:
            raise NotImplementedError("detect_heads: the max-in-out heads are two-class (background / face)")
        if prior_data.size(0) != num_priors:
            raise ValueError(f"detect_heads: {prior_data.size(0)} priors for {num_priors} map positions")
        with torch.cuda.device(dev):
            pri = _lib.dev_f32(prior_data, dev).view(num_priors, 4)
            out = torch.empty((num, 2, self.top_k, 5), dtype=torch.float32, device=dev)
            counts = torch.empty((num, 2), dtype=torch.int32, device=dev) if return_aux else None
            kept = torch.empty((num, 2, self.top_k), dtype=torch.int64, device=dev) if return_aux else None
            Lb = _lib.lib()
            ws = self._workspaces.get(num, num_priors, 2, dev)
            _lib.check(Lb.fdt_detect_heads_ex(ld, cd, dt, fh, fw, nm, L, _lib.ptr(pri), num, int(self.top_k), int(self.nms_top_k),
                                              float(self.conf_thresh), float(self.nms_thresh), float(self.variance[0]),
                                              float(self.variance[1]), _lib.ptr(out), _lib.ptr(counts), _lib.ptr(kept),
                                              _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
        del keep
        return (out, counts, kept) if return_aux else out

    def _call_host(self, loc_data, conf_data, prior_data, args, return_aux):
        return self.submit(loc_data, conf_data, prior_data, return_aux).result()

    def submit(self, loc_data, conf_data, prior_data, return_aux=False):
        """Asynchronous form of __call__ for HOST tensors (a stream of video batches): enqueues the copies and kernels
        (fdt_detect_host_submit) and returns a PendingDetections whose .result() blocks until the output landed.  Keeping two
        batches in flight hides everything but the host-to-device copy of `conf`.  Pinned inputs make the submit non-blocking;
        the tensors must stay untouched until .result().  A prior tensor that was already uploaded by this thread (same storage,
        same version counter) is not copied again."""
        _lib.require_cuda()
        if loc_data.is_cuda:
            raise ValueError("Detect.submit is the host-tensor path; CUDA tensors are already asynchronous through __call__")
        num, num_priors, C_ = loc_data.size(0), prior_data.size(0), self.num_classes
        args = (num, num_priors, C_, int(self.top_k), int(self.nms_top_k), float(self.conf_thresh),
                float(self.nms_thresh), float(self.variance[0]), float(self.variance[1]))
        loc = loc_data.detach().to(torch.float32).contiguous()
        conf = conf_data.detach().to(torch.float32).contiguous()
        pri = prior_data.detach().to(torch.float32).contiguous().cpu()
        out = torch.empty((num, C_, self.top_k, 5), dtype=torch.float32, pin_memory=True)
        counts = torch.empty((num, C_), dtype=torch.int32, pin_memory=True) if return_aux else None
        kept = torch.empty((num, C_, self.top_k), dtype=torch.int64, pin_memory=True) if return_aux else None
        dev_index = torch.cuda.current_device()
        ctx = _ctx(dev_index)
        # the prior set is a constant of the model: uploaded once per (thread, device) and tensor.  The cache holds the tensor, so
        # its storage cannot be recycled under the key; in-place torch writes bump _version (writes through a numpy alias do not).
        resident = _host_ctx.__dict__.setdefault("priors", {})
        key = (pri.data_ptr(), pri._version, num_priors)
        hit = dev_index in resident and resident[dev_index][0] == key
        ticket = C.c_uint64(0)
        _lib.check(_lib.lib().fdt_detect_host_submit(ctx, _lib.ptr(loc), _lib.ptr(conf), None if hit else _lib.ptr(pri),
                                                     *args, _lib.ptr(out), _lib.ptr(counts), _lib.ptr(kept), C.byref(ticket)))
        resident[dev_index] = (key, pri)
        return PendingDetections(ctx, ticket.value, (out, counts, kept) if return_aux else out, (loc, conf, pri))


class PendingDetections:
    """Result handle of Detect.submit: .result() waits for the call (fdt_detect_host_wait) and returns what __call__ would."""

    def __init__(self, ctx, ticket, value, keep_alive):
        self._ctx, self._ticket, self._value, self._keep = ctx, ticket, value, keep_alive

    def result(self):
        if self._keep is not None:
            _lib.check(_lib.lib().fdt_detect_host_wait(self._ctx, self._ticket))
            self._keep = None
        return self._value
