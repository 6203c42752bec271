"""MultiBoxLoss -- drop-in for layers/modules/multibox_loss.py:9-136 on hand-written sm_100a kernels."""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn

from ... import _lib
from ...data import face as cfg
from ..functions.heads import _head_args, _map_grads, map_descs


def pack_targets(targets, device):
    """list[B] of [G_i,5] tensors -> (gt[total,5] fp32, gt_off[B+1] int64, total) on `device`.
    One concatenation + one small H2D copy of the offsets; images without GT get an empty range."""
    counts = [int(t.shape[0]) if t is not None and t.numel() else 0 for t in targets]
    off = [0]
    for c in counts:
        off.append(off[-1] + c)
    total = off[-1]
    rows = [t for t, c in zip(targets, counts) if c]
    if not rows:
        gt = torch.zeros((1, 5), dtype=torch.float32, device=device)
    elif all(t.device == device and t.dtype == torch.float32 and t.dim() == 2 for t in rows):
        gt = torch.cat(rows, 0).detach()                  # the training loop's case: one launch for the whole batch
    else:
        gt = torch.cat([t.detach().reshape(-1, 5).to(device=device, dtype=torch.float32) for t in rows], 0).contiguous()
    return gt, torch.tensor(off, dtype=torch.int64).to(device, non_blocking=True), total


class _MultiBoxLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, loc_data, conf_data, priors, gt, gt_off, total_gt, threshold, negpos_ratio, bipartite, variance):
        dev = loc_data.device
        B, N, _ = loc_data.shape
        C_ = conf_data.shape[-1]
        loc = _lib.dev_f32(loc_data, dev)
        conf = _lib.dev_f32(conf_data, dev)
        pri = _lib.dev_f32(priors, dev)
        losses = torch.empty(2, dtype=torch.float32, device=dev)
        norm = torch.empty(1, dtype=torch.float32, device=dev)
        loc_t = torch.empty((B, N, 4), dtype=torch.float32, device=dev)
        conf_t = torch.empty((B, N), dtype=torch.int64, device=dev)
        sel = torch.empty((B, N), dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            L = _lib.lib()
            ws = _lib.workspace(L.fdt_multibox_workspace_bytes(B, N, C_, total_gt), dev, "multibox")
            _lib.check(L.fdt_multibox_loss_forward(
                _lib.ptr(loc), _lib.ptr(conf), _lib.ptr(pri), _lib.ptr(gt), _lib.ptr(gt_off), total_gt, B, N, C_,
                float(threshold), int(negpos_ratio), int(bool(bipartite)), float(variance[0]), float(variance[1]),
                _lib.ptr(losses), _lib.ptr(norm), _lib.ptr(loc_t), _lib.ptr(conf_t), _lib.ptr(sel), None,
                _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
        ctx.save_for_backward(loc, conf, loc_t, conf_t, sel, norm)
        ctx.mark_non_differentiable(loc_t, conf_t, sel)
        # two independent 0-dim tensors, as the reference returns (views of one buffer would forbid in-place ops on them)
        return losses[0].clone(), losses[1].clone(), loc_t, conf_t, sel

    @staticmethod
    def backward(ctx, g_l, g_c, *_):
        loc, conf, loc_t, conf_t, sel, norm = ctx.saved_tensors
        B, N, _ = loc.shape
        C_ = conf.shape[-1]
        grad_loc = torch.empty_like(loc)
        grad_conf = torch.empty_like(conf)
        # the upstream gradients stay on the device: no float() synchronisation, the loss can be captured in a CUDA graph
        dev = loc.device
        zero = None
        def scalar(g):
            nonlocal zero
            if g is None:
                if zero is None:
                    zero = torch.zeros((), dtype=torch.float32, device=dev)
                return zero
            return g.detach().to(device=dev, dtype=torch.float32).contiguous()
        gl, gc = scalar(g_l), scalar(g_c)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().fdt_multibox_loss_backward_dev(
                _lib.ptr(loc), _lib.ptr(conf), _lib.ptr(loc_t), _lib.ptr(conf_t), _lib.ptr(sel), _lib.ptr(norm),
                _lib.ptr(gl), _lib.ptr(gc), B, N, C_, _lib.ptr(grad_loc), _lib.ptr(grad_conf), _lib.stream_ptr()))
        return grad_loc, grad_conf, None, None, None, None, None, None, None, None


class _MultiBoxLossHeadsFn(torch.autograd.Function):
    """MultiBoxLoss straight from the per-level NCHW head maps (C = 2): the loss kernels read the maps, the backward writes
    the map gradients -- nothing [B,N,4] / [B,N,2] is materialised in either direction."""

    @staticmethod
    def forward(ctx, priors, gt, gt_off, total_gt, threshold, negpos_ratio, bipartite, variance, neg_max, L, *maps):
        dev, B, N, (conf, loc), (ld, cd, dt, fh, fw, nm, _) = _head_args(maps[:L], maps[L:], neg_max)
        pri = _lib.dev_f32(priors, dev)
        if pri.dim() != 2 or pri.size(1) != 4 or pri.size(0) != N:
            raise ValueError(f"MultiBoxLoss.forward_heads: priors must be [{N},4] (one per map position), got {tuple(pri.shape)}")
        losses = torch.empty(2, dtype=torch.float32, device=dev)
        norm = torch.empty(1, dtype=torch.float32, device=dev)
        loc_t = torch.empty((B, N, 4), dtype=torch.float32, device=dev)
        conf_t = torch.empty((B, N), dtype=torch.int64, device=dev)
        sel = torch.empty((B, N), dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            lib = _lib.lib()
            ws = _lib.workspace(lib.fdt_multibox_workspace_bytes(B, N, 2, total_gt), dev, "multibox")
            _lib.check(lib.fdt_multibox_loss_forward_heads_ex(
                ld, cd, dt, fh, fw, nm, L, _lib.ptr(pri), _lib.ptr(gt), _lib.ptr(gt_off), total_gt, B,
                float(threshold), int(negpos_ratio), int(bool(bipartite)), float(variance[0]), float(variance[1]),
                _lib.ptr(losses), _lib.ptr(norm), _lib.ptr(loc_t), _lib.ptr(conf_t), _lib.ptr(sel), None,
                _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
        ctx.save_for_backward(loc_t, conf_t, sel, norm, *loc, *conf)
        ctx.level = (fh, fw, nm, L, B, dev, dt)
        ctx.mark_non_differentiable(loc_t, conf_t, sel)
        return losses[0].clone(), losses[1].clone(), loc_t, conf_t, sel

    @staticmethod
    def backward(ctx, g_l, g_c, *_):
        fh, fw, nm, L, B, dev, dt = ctx.level
        loc_t, conf_t, sel, norm, *maps = ctx.saved_tensors
        loc, conf = maps[:L], maps[L:]
        need_loc, need_conf = any(ctx.needs_input_grad[10:10 + L]), any(ctx.needs_input_grad[10 + L:])
        gl_maps, gld = _map_grads(loc, need_loc)
        gc_maps, gcd = _map_grads(conf, need_conf)
        zero = torch.zeros((), dtype=torch.float32, device=dev)
        gl = zero if g_l is None else g_l.detach().to(device=dev, dtype=torch.float32).contiguous()
        gc = zero if g_c is None else g_c.detach().to(device=dev, dtype=torch.float32).contiguous()
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().fdt_multibox_loss_backward_heads_dev_ex(
                map_descs(loc), map_descs(conf), dt, fh, fw, nm, L, _lib.ptr(loc_t), _lib.ptr(conf_t), _lib.ptr(sel), _lib.ptr(norm),
                _lib.ptr(gl), _lib.ptr(gc), B, gld, gcd, _lib.stream_ptr()))
        return (None,) * 10 + (*(gl_maps or [None] * L), *(gc_maps or [None] * L))


class MultiBoxLoss(nn.Module):
    """SSD weighted loss (multibox_loss.py:9-30): match + encode, smooth-L1 on positives, hard-negative
    mining (negpos_ratio:1), cross-entropy over positives and mined negatives, both divided by the
    number of positives.  Same constructor and forward signature as the reference.

    Differences that are deliberate and documented (DESIGN.md):
      * images with zero ground-truth boxes (the reference raises IndexError) count as all-background;
      * `use_gpu` is accepted for compatibility; compute always runs on the CUDA device of loc_data
        (or the current device for CPU inputs) -- there is no CPU path."""

    def __init__(self, num_classes, overlap_thresh, prior_for_matching,
                 bkg_label, neg_mining, neg_pos, neg_overlap, encode_target, bipartite=True,
                 use_gpu=True):
        super(MultiBoxLoss, self).__init__()
        self.use_gpu = use_gpu
        self.num_classes = num_classes
        self.threshold = overlap_thresh
        self.background_label = bkg_label
        self.encode_target = encode_target
        self.use_prior_for_matching = prior_for_matching
        self.do_neg_mining = neg_mining
        self.negpos_ratio = neg_pos
        self.neg_overlap = neg_overlap
        self.bipartite = bipartite
        self.variance = cfg['variance']
        self.last_aux = None          # (loc_t, conf_t, sel) of the latest forward, for inspection / tests

    def forward(self, predictions, targets):
        """predictions = (loc [B,N,4], conf [B,N,C] raw logits, priors [N,4]);
        targets = list[B] of [G_i,5] rows [xmin, ymin, xmax, ymax, label]  ->  (loss_l, loss_c)"""
        loc_data, conf_data, priors = predictions
        dev = _lib.require_cuda()
        src = loc_data.device
        if src.type == "cuda":
            dev = src
        else:
            loc_data, conf_data = loc_data.to(dev), conf_data.to(dev)
        gt, gt_off, total = pack_targets(targets, dev)
        loss_l, loss_c, loc_t, conf_t, sel = _MultiBoxLossFn.apply(
            loc_data, conf_data, priors, gt, gt_off, total, self.threshold, self.negpos_ratio, self.bipartite,
            self.variance)
        self.last_aux = (loc_t, conf_t, sel)
        return loss_l.to(src), loss_c.to(src)

    def forward_heads(self, loc_maps, conf_maps, priors, targets, neg_max=None):
        """The loss straight from the models' per-level NCHW head maps (pyramid.py:291-309): loc_maps[l] [B,4,H_l,W_l] and the
        4-channel max-in-out conf_maps[l] [B,4,H_l,W_l]; neg_max[l] as in heads_to_loc_conf (default: level 0 reduces the
        negatives).  Equals forward((*heads_to_loc_conf(loc_maps, conf_maps, neg_max, softmax=False), priors), targets), and is
        differentiable with respect to every map that requires grad, without materialising loc / conf or their gradients."""
        if self.num_classes != 2:
            raise NotImplementedError("MultiBoxLoss.forward_heads: the head maps carry two classes (num_classes=2)")
        L = len(conf_maps)
        if len(loc_maps) != L:
            raise ValueError("MultiBoxLoss.forward_heads: need one loc map and one conf map per pyramid level")
        dev = _lib.require_cuda()
        if conf_maps[0].is_cuda:
            dev = conf_maps[0].device
        gt, gt_off, total = pack_targets(targets, dev)
        nmx = None if neg_max is None else tuple(int(bool(v)) for v in neg_max)
        loss_l, loss_c, loc_t, conf_t, sel = _MultiBoxLossHeadsFn.apply(
            priors, gt, gt_off, total, self.threshold, self.negpos_ratio, self.bipartite, self.variance, nmx, L,
            *loc_maps, *conf_maps)
        self.last_aux = (loc_t, conf_t, sel)
        return loss_l, loss_c
