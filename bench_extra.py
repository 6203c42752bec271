#!/usr/bin/env python
"""Secondary measurements for the other SURVEY section-8 rows (not the driver's headline; bench.py is):

    python bench_extra.py multibox   # BASELINE config 3: MultiBoxLoss B=32, N=34,125, G in [0,200]
    python bench_extra.py tracker    # BASELINE config 4: IoU tracker, 10k frames x 1-300 detections
    python bench_extra.py detect1024 # BASELINE config 5 shape on one GPU: Detect B=64 @1024^2 (N=87,360)
    python bench_extra.py priorbox
    python bench_extra.py siblings   # SURVEY 8f rank 3: FaceBoxes decode_np (21,824 default boxes) and MTCNN nms variants
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 bench_extra.py config5
                                     # BASELINE config 5: Detect B=512 @1024^2 sharded over N GPUs, gather fused / NCCL
    python bench_extra.py torchref   # BASELINE.md 5.4: the reference's python-loop Detect restated in torch, on CUDA tensors and on the CPU
    python bench_extra.py heads      # SURVEY 8f rank 1: Detect straight from the per-level NCHW head maps, B=64 @640^2
    python bench_extra.py heads_train # SURVEY 8f rank 1: MultiBoxLoss (+ backward) straight from the head maps, B=32 @640^2 (config 3)
    python bench_extra.py match_mine # fdt_match_encode and fdt_hard_negative_mine on their own (box_utils.match_*, DataEncoder.encode)
    python bench_extra.py flat_amp   # bf16 / fp16 flat loc / conf read in place by Detect, Detect.submit and MultiBoxLoss vs converted
    python bench_extra.py track_stream # online tracker: V in {1, 64, 148} streams x 2,000 config-4 frames, one frame per stream per
                                     # step, vs the offline tracker per video; Detect B=64 @640^2 + step_detections vs Detect alone

Each prints one JSON line with device time (CUDA events, L2 flushed between repetitions), the algorithmic bytes of
SURVEY 8(d) and the CPU oracle port timed on the host beside it."""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch

import fdt_b200  # noqa: F401
from fdt_b200 import _lib, synth
from oracle import oracle as orc

PEAK = 6500.6
try:
    PEAK = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
except Exception:
    pass


def timed(fn, reps=20, warm=3):
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush.zero_()
        torch.cuda._sleep(250_000)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.mean(ts)), float(np.min(ts))


def cpu_time(fn, budget=8.0):
    fn()
    n, t0 = 0, time.perf_counter()
    while True:
        fn(); n += 1
        dt = time.perf_counter() - t0
        if dt > budget or n >= 20:
            return dt / n, n


def multibox():
    from fdt_b200.layers import MultiBoxLoss
    from fdt_b200.layers.modules.multibox_loss import pack_targets
    B = 32
    pri = synth.priors_numpy(640, 640); N = pri.shape[0]
    loc, conf, targets = synth.multibox_inputs(B, pri, 3030, 0, 200)
    dev = torch.device("cuda")
    l, c, p = (torch.from_numpy(a).to(dev) for a in (loc, conf, pri))
    tg = [torch.from_numpy(t).to(dev) for t in targets]
    out = {}
    for bip in (False, True):
        crit = MultiBoxLoss(2, 0.35, True, 0, True, 3, 0.35, False, bipartite=bip)
        gt, off, total = pack_targets(tg, dev)
        L = _lib.lib()
        losses = torch.empty(2, device=dev); norm = torch.empty(1, device=dev)
        loc_t = torch.empty((B, N, 4), device=dev); conf_t = torch.empty((B, N), dtype=torch.int64, device=dev)
        sel = torch.empty((B, N), dtype=torch.uint8, device=dev)
        ws = _lib.workspace(L.fdt_multibox_workspace_bytes(B, N, 2, total), dev, "bx")

        def fwd():
            _lib.check(L.fdt_multibox_loss_forward(l.data_ptr(), c.data_ptr(), p.data_ptr(), gt.data_ptr(), off.data_ptr(), total,
                                                   B, N, 2, 0.35, 3, int(bip), 0.1, 0.2, losses.data_ptr(), norm.data_ptr(),
                                                   loc_t.data_ptr(), conf_t.data_ptr(), sel.data_ptr(), None, ws.data_ptr(),
                                                   ws.numel(), _lib.stream_ptr()))
        ms, ms_min = timed(fwd)
        lr = l.clone().requires_grad_(True); cr = c.clone().requires_grad_(True)

        def fwdbwd():
            ll, lc = crit((lr, cr, p), tg)
            (ll + lc).backward()
        ms_fb, _ = timed(fwdbwd, reps=10)
        out["bipartite" if bip else "default"] = {"forward_ms": ms, "forward_ms_min": ms_min, "images_per_s": B / (ms * 1e-3),
                                                  "module_fwd_bwd_ms": ms_fb}
    G = sum(t.shape[0] for t in targets)
    alg = B * 48 * N + 20 * G
    cpu_s, n = cpu_time(lambda: orc.multibox_loss(loc, conf, pri, targets, 0.35, 3, False, want_aux=False))
    d = out["default"]
    print(json.dumps({"workload": "MultiBoxLoss match/encode + mining + loss, B=32, N=34,125, G~U{0..200} (config 3)", "results": out,
                      "algorithmic_bytes": alg, "achieved_gbs": alg / (d["forward_ms"] * 1e-3) / 1e9,
                      "roofline_frac_of_measured_hbm": alg / (d["forward_ms"] * 1e-3) / 1e9 / PEAK, "gt_total": G,
                      "iou_evaluations": int(sum(t.shape[0] for t in targets) * N),
                      "cpu_baseline": {"images_per_s": B / cpu_s, "cores": orc.max_threads(), "kind": "port", "sample": f"{n} batches"}}))


def tracker():
    from fdt_b200 import tracker as T
    frames = synth.tracker_frames(F=10000, seed=4040, d_lo=1, d_hi=300, n_objects=300, empty_every=1000)
    dets, off = T.pack_frames(frames)
    d = torch.from_numpy(dets).cuda(); o = torch.from_numpy(off).cuda()
    F = len(frames); total = int(off[-1]); max_d = int(np.diff(off).max())
    L = _lib.lib()
    dev = torch.device("cuda")
    n = torch.zeros(1, dtype=torch.int64, device=dev); t_off = torch.zeros(total + 2, dtype=torch.int64, device=dev)
    t_dets = torch.zeros(total, dtype=torch.int64, device=dev); t_start = torch.zeros(total + 1, dtype=torch.int64, device=dev)
    t_max = torch.zeros(total + 1, dtype=torch.float64, device=dev)
    ws = _lib.workspace(L.fdt_iou_track_workspace_bytes(F, total, max_d), dev, "tx")

    def run():
        _lib.check(L.fdt_iou_track(d.data_ptr(), o.data_ptr(), F, total, max_d, 0.4, 0.6, 5, n.data_ptr(), t_off.data_ptr(),
                                   t_dets.data_ptr(), t_start.data_ptr(), t_max.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr()))
    ms, ms_min = timed(run, reps=5, warm=1)
    t0 = time.perf_counter(); tr = T.iou_track(frames); api_s = time.perf_counter() - t0
    t0 = time.perf_counter(); ref = orc.iou_track(frames); cpu_s = time.perf_counter() - t0
    same = len(tr) == len(ref) and all(a["bboxes"] == b["bboxes"] and a["start_frame"] == b["start_frame"] for a, b in zip(tr, ref))
    print(json.dumps({"workload": "IoU tracker association, 10,000 frames x U{1..300} detections (config 4)", "frames": F,
                      "detections": total, "tracks": len(tr), "device_ms": ms, "device_ms_min": ms_min, "frames_per_s_device": F / (ms * 1e-3),
                      "frames_per_s_api_incl_python_dict_build": F / api_s, "identical_to_oracle": bool(same),
                      "algorithmic_bytes": 28 * total, "note": "latency-bound serial chain; roofline fraction not meaningful (SURVEY 8d)",
                      "cpu_baseline": {"frames_per_s": F / cpu_s, "cores": 1, "kind": "port", "sample": "whole video, C oracle, single thread"}}))


def detect1024():
    from fdt_b200.layers import Detect
    B = 64
    pri = synth.priors_numpy(1024, 1024); N = pri.shape[0]
    loc, conf = synth.detect_inputs(B, pri, 5050, 0.05)
    det = Detect(2, 0, 750, 0.05, 0.3)
    a = [torch.from_numpy(x).cuda() for x in (loc, conf, pri)]
    ms, ms_min = timed(lambda: det(*a))
    alg = B * (24 * N + 30000) + 16 * N
    print(json.dumps({"workload": "Detect B=64 @1024x1024 (N=87,360), conf 0.05, nms 0.3 (config 5 shard shape)", "ms": ms, "ms_min": ms_min,
                      "frames_per_s": B / (ms * 1e-3), "algorithmic_bytes": alg, "roofline_frac_of_measured_hbm": alg / (ms * 1e-3) / 1e9 / PEAK,
                      "candidates_per_image": float((conf[..., 1] > 0.05).sum(1).mean())}))


def detect512():
    """BASELINE config 5 on ONE GPU: B=512 @1024x1024 (N=87,360).  Inputs are generated on the device (1.07 GB)."""
    from fdt_b200.layers import Detect
    B = 512
    pri = synth.priors_numpy(1024, 1024); N = pri.shape[0]
    g = torch.Generator(device="cuda"); g.manual_seed(5)
    loc = torch.randn((B, N, 4), device="cuda", generator=g) * 0.5
    d = torch.randn((B, N), device="cuda", generator=g) * 2.0 - 4.5
    s1 = torch.sigmoid(d)
    conf = torch.stack([1 - s1, s1], -1).contiguous()
    det = Detect(2, 0, 750, 0.05, 0.3)
    p = torch.from_numpy(pri).cuda()
    ms, ms_min = timed(lambda: det(loc, conf, p), reps=10)
    alg = B * (24 * N + 30000) + 16 * N
    print(json.dumps({"workload": "Detect B=512 @1024x1024 (N=87,360) on one GPU (config 5 unsharded; device-generated inputs, scores may tie)",
                      "ms": ms, "ms_min": ms_min, "frames_per_s": B / (ms * 1e-3), "algorithmic_bytes": alg,
                      "roofline_frac_of_measured_hbm": alg / (ms * 1e-3) / 1e9 / PEAK,
                      "candidates_per_image": float((conf[..., 1] > 0.05).sum(1).float().mean())}))


def config5():
    """BASELINE config 5: Detect batch 512 @1024x1024 (N=87,360) sharded over the ranks of a torchrun launch (strong scaling: every
    rank owns 512 / world images), detections gathered on every rank -- fused into the NMS kernel over NVLink peer memory, and with
    an NCCL all-gather for comparison.  Device-generated inputs (as detect512)."""
    import torch.distributed as dist
    from fdt_b200.layers import Detect
    from fdt_b200.sharding import PeerGatherDetect, ShardedDetect
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B_total = 512
    B = B_total // world
    pri = synth.priors_numpy(1024, 1024); N = pri.shape[0]
    g = torch.Generator(device=dev); g.manual_seed(5 + rank)
    loc = torch.randn((B, N, 4), device=dev, generator=g) * 0.5
    s1 = torch.sigmoid(torch.randn((B, N), device=dev, generator=g) * 2.0 - 4.5)
    conf = torch.stack([1 - s1, s1], -1).contiguous()
    p = torch.from_numpy(pri).to(dev)
    det = Detect(2, 0, 750, 0.05, 0.3)
    res = {}
    variants = [("single", det)] if world == 1 else [("peer_gather_to_rank0", PeerGatherDetect(det, B, dest=0, signal="kernel")), ("peer_all_gather", PeerGatherDetect(det, B, dest="all", signal="kernel")),
                                                       ("nccl_all_gather", ShardedDetect(det, gather="block"))]
    for name, fn in variants:
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        for _ in range(3):
            fn(loc, conf, p)
        torch.cuda.synchronize()
        ts = []
        for _ in range(12):
            flush.zero_()
            if world > 1:
                dist.barrier()
            torch.cuda._sleep(400_000)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); out = fn(loc, conf, p); e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        t = torch.tensor([float(np.mean(ts))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res[name] = {"ms_per_step": float(t.item()), "frames_per_s": B_total / (float(t.item()) * 1e-3), "gathered_shape": list(out.shape)}
    alg = B_total * (24 * N + 30000) + world * 16 * N
    if rank == 0:
        best = min(v["ms_per_step"] for v in res.values())
        print(json.dumps({"workload": "Detect B=512 @1024x1024 (N=87,360) sharded over %d GPU(s), strong scaling (config 5)" % world, "n_gpus": world,
                          "images_per_gpu": B, "results": res, "algorithmic_bytes": alg,
                          "aggregate_roofline_frac_of_measured_hbm": alg / (best * 1e-3) / 1e9 / (PEAK * world)}))
    if world > 1:
        dist.destroy_process_group()


def torchref():
    """BASELINE config 1 (one 640x640 image, N=34,125, conf 0.05, nms 0.3) through the reference's algorithm as the reference
    deploys it -- a python loop of small torch ops (oracle/torch_ref.py restates detection.py:34-84 / box_utils.py:275-340; the
    reference itself cannot travel to the GPU box) -- on CUDA tensors on this B200 and on the host CPU, next to fdt_detect."""
    from oracle import torch_ref
    from fdt_b200.layers import Detect
    pri = synth.priors_numpy(640, 640)
    loc, conf = synth.detect_inputs(1, pri, 20261, 0.05)
    ref_det = torch_ref.Detect(2, 0, 750, 0.05, 0.3)
    res = {}
    outs = {}
    for dev in ("cuda", "cpu"):
        a = [torch.from_numpy(x).to(dev) for x in (loc, conf, pri)]
        if dev == "cpu":
            torch.set_num_threads(os.cpu_count() or 1)
        best = 1e9
        for _ in range(3):
            if dev == "cuda":
                torch.cuda.synchronize()
            t0 = time.perf_counter()
            o = ref_det(*a)
            if dev == "cuda":
                torch.cuda.synchronize()
            best = min(best, time.perf_counter() - t0)
        outs[dev] = o.cpu().numpy()
        res[f"torch_{dev}_s_per_image"] = best
        res[f"torch_{dev}_frames_per_s"] = 1.0 / best
    a = [torch.from_numpy(x).cuda() for x in (loc, conf, pri)]
    det = Detect(2, 0, 750, 0.05, 0.3)
    ours = det(*a)
    ms, _ = timed(lambda: det(*a))
    same = bool(np.array_equal(ours.cpu().numpy()[..., 0], outs["cuda"][..., 0]) and np.array_equal(outs["cuda"][..., 0], outs["cpu"][..., 0]))
    print(json.dumps({"workload": "Detect, 1 image @640x640 (N=34,125, %d candidates), conf 0.05, nms 0.3 (config 1)" % int((conf[0, :, 1] > 0.05).sum()),
                      "reference_algorithm_in_torch": res, "host_threads": os.cpu_count(), "fdt_detect_ms": ms, "fdt_detect_frames_per_s": 1e3 / ms,
                      "same_kept_scores": same}))


def priorbox():
    from fdt_b200.layers import PriorBoxLayer
    layer = PriorBoxLayer(640, 640)
    fm = synth.feature_maps(640, 640)
    ms, _ = timed(lambda: [layer(i, fw, fh) for i, (fw, fh) in enumerate(fm)])
    ref = orc.PriorBoxLayer(640, 640)
    cpu_s, _ = cpu_time(lambda: [ref(i, fw, fh) for i, (fw, fh) in enumerate(fm)], budget=2.0)
    print(json.dumps({"workload": "PriorBoxLayer(640,640) x 6 levels (34,125 priors)", "ms_6_launches_incl_python": ms, "cpu_port_ms": cpu_s * 1e3}))


def siblings():
    """FaceBoxes DataEncoder.decode_np (threshold + decode + nms_np over the 21,824 default boxes) and MTCNN nms on 3,000 boxes:
    device time through the C ABI vs the C oracle port on one host core (the reference is single-threaded numpy)."""
    dev = torch.device("cuda")
    L = _lib.lib(); st = _lib.stream_ptr()
    db_np = orc.facebox_default_boxes(); N = db_np.shape[0]
    rng = np.random.Generator(np.random.PCG64(7070))
    loc_np = (rng.standard_normal((N, 4)) * 0.5).astype(np.float32)
    s1 = (1.0 / (1.0 + np.exp(-(rng.standard_normal(N) * 2.0 - 2.0)))).astype(np.float32)
    conf_np = np.stack([1 - s1, s1], 1).astype(np.float32)
    loc, conf, db = (torch.from_numpy(a).to(dev) for a in (loc_np, conf_np, db_np))
    boxes = torch.empty((N, 4), device=dev); keep = torch.zeros(N, dtype=torch.int64, device=dev); cnt = torch.zeros(1, dtype=torch.int64, device=dev)
    ws = _lib.workspace(L.fdt_threshold_nms_workspace_bytes(N), dev, "sx")
    res = {}
    for thr in (0.35, 0.25):
        def run():
            _lib.check(L.fdt_facebox_decode(loc.data_ptr(), db.data_ptr(), N, 0.1, 0.2, boxes.data_ptr(), st))
            _lib.check(L.fdt_threshold_nms(boxes.data_ptr(), conf.data_ptr(), N, thr, 0.5, _lib.NMS_SUMFIRST, keep.data_ptr(), cnt.data_ptr(),
                                           ws.data_ptr(), ws.numel(), st))
        ms, mn = timed(run)
        cpu_s, _ = cpu_time(lambda: orc.facebox_decode_np(loc_np, conf_np, db_np, conf_thres=thr), budget=3.0)
        rb, rs = orc.facebox_decode_np(loc_np, conf_np, db_np, conf_thres=thr)
        same = int(cnt.item()) == rb.shape[0] and np.array_equal(boxes[keep[:int(cnt.item())]].cpu().numpy(), rb)
        res[f"decode_np_thr{thr}"] = {"candidates": int((s1 > thr).sum()), "kept": int(cnt.item()), "device_ms": ms, "device_ms_min": mn,
                                      "cpu_port_ms_1_core": cpu_s * 1e3, "identical_to_oracle": bool(same)}
    rng = np.random.Generator(np.random.PCG64(7071))
    n = 3000
    c = rng.uniform(20, 460, (150, 2)); ctr = c[rng.integers(0, 150, n)] + rng.normal(0, 8, (n, 2)); wh = rng.uniform(6, 120, (n, 2))
    d_np = np.concatenate([ctr - wh / 2, ctr + wh / 2, (rng.permutation(n) / n)[:, None]], 1).astype(np.float32)
    bx = torch.from_numpy(np.ascontiguousarray(d_np[:, :4])).to(dev); sc = torch.from_numpy(np.ascontiguousarray(d_np[:, 4])).to(dev)
    keep = torch.zeros(n, dtype=torch.int64, device=dev)
    ws2 = _lib.workspace(L.fdt_nms_workspace_bytes(n), dev, "sx2")
    for name, thr, flags in (("mtcnn_nms_union_0.6", 0.6, _lib.NMS_SUMFIRST), ("mtcnn_nms_minimum_0.4", 0.4, _lib.NMS_MINIMUM),
                             ("mtcnn_torch_nms_union_0.5", 0.5, _lib.NMS_SUMFIRST | _lib.NMS_PLUS1 | _lib.NMS_LE)):
        def run():
            _lib.check(L.fdt_nms_variant(bx.data_ptr(), sc.data_ptr(), n, thr, flags, keep.data_ptr(), cnt.data_ptr(), ws2.data_ptr(), ws2.numel(), st))
        ms, mn = timed(run)
        cpu_s, _ = cpu_time(lambda: orc.nms_variant(d_np[:, :4], d_np[:, 4], thr, flags), budget=2.0)
        ref = orc.nms_variant(d_np[:, :4], d_np[:, 4], thr, flags)
        res[name] = {"boxes": n, "kept": int(cnt.item()), "device_ms": ms, "device_ms_min": mn, "cpu_port_ms_1_core": cpu_s * 1e3,
                     "identical_to_oracle": bool(np.array_equal(keep[:int(cnt.item())].cpu().numpy(), ref))}
    print(json.dumps({"workload": "sibling decode+NMS implementations (FaceBoxes DataEncoder.decode_np, MTCNN nms / torch_nms)", "results": res}))


def heads():
    """Head maps -> detections, B=64 @640x640 (N=34,125): fused (fdt_detect_heads) vs materialise + Detect vs the reference's
    torch ops (pyramid.py:291-309, 331-332 on CUDA tensors) + Detect."""
    from fdt_b200.layers import Detect, heads_to_loc_conf
    B = 64
    loc_maps, conf_maps, neg_max = synth.head_maps(B, 640, 640, 6060)
    pri = torch.from_numpy(synth.priors_numpy(640, 640)).cuda(); N = pri.shape[0]
    lm, cm = [torch.from_numpy(m).cuda() for m in loc_maps], [torch.from_numpy(m).cuda() for m in conf_maps]
    det = Detect(2, 0, 750, 0.05, 0.3)

    def torch_heads():
        loc, conf = [], []
        for idx, (lx, tmp_conf) in enumerate(zip(lm, cm)):
            if idx == 0:
                a, b, c, pos_conf = tmp_conf.chunk(4, 1)
                max_conf, _ = torch.cat([a, b, c], 1).max(1)
                conf.append(torch.cat([max_conf.view_as(pos_conf), pos_conf], 1).permute(0, 2, 3, 1).contiguous())
            else:
                neg_conf, a, b, c = tmp_conf.chunk(4, 1)
                max_conf, _ = torch.cat([a, b, c], 1).max(1)
                conf.append(torch.cat([neg_conf, max_conf.view_as(neg_conf)], 1).permute(0, 2, 3, 1).contiguous())
            loc.append(lx.permute(0, 2, 3, 1).contiguous())
        loc = torch.cat([o.view(o.size(0), -1) for o in loc], 1).view(B, -1, 4)
        conf = torch.softmax(torch.cat([o.view(o.size(0), -1) for o in conf], 1).view(B, -1, 2), -1)
        return loc, conf

    fused = det.detect_heads(lm, cm, pri)
    assert torch.equal(fused, det(*heads_to_loc_conf(lm, cm, neg_max), pri))
    # the timed calls go straight to the C ABI with prebuilt arguments (as bench.py does), so that the event pairs see device time
    from fdt_b200.layers.functions.heads import _level_args
    dev, _, _, keep, (lp, cp, fh, fw, nm, nl) = _level_args(lm, cm, neg_max)
    L = _lib.lib()
    out = torch.empty((B, 2, 750, 5), device=dev); loc_b = torch.empty((B, N, 4), device=dev); conf_b = torch.empty((B, N, 2), device=dev)
    ws = _lib.workspace(L.fdt_detect_workspace_bytes(B, N, 2), dev, "hx")
    st = _lib.stream_ptr()

    def c_fused():
        _lib.check(L.fdt_detect_heads(lp, cp, fh, fw, nm, nl, pri.data_ptr(), B, 750, 5000, 0.05, 0.3, 0.1, 0.2, out.data_ptr(), None, None,
                                      ws.data_ptr(), ws.numel(), st))

    def c_heads():
        _lib.check(L.fdt_heads_to_loc_conf(lp, cp, fh, fw, nm, nl, B, 1, loc_b.data_ptr(), conf_b.data_ptr(), st))

    def c_mat():
        c_heads()
        _lib.check(L.fdt_detect(loc_b.data_ptr(), conf_b.data_ptr(), pri.data_ptr(), B, N, 2, 750, 5000, 0.05, 0.3, 0.1, 0.2, out.data_ptr(),
                                None, None, ws.data_ptr(), ws.numel(), st))
    c_fused()
    assert torch.equal(out, fused)
    ms_f, min_f = timed(c_fused)
    ms_m, _ = timed(c_mat)
    ms_h, _ = timed(c_heads)
    ms_t, _ = timed(lambda: det(*torch_heads(), pri))
    ms_th, _ = timed(torch_heads)
    # back to back (the bench.py `value` protocol): K calls on one stream over two rotating sets of head maps (140 MB > L2) and a
    # workspace ring of 4 slots, so that consecutive calls overlap on the device
    loc2, conf2, _ = synth.head_maps(B, 640, 640, 6061)
    lm2, cm2 = [torch.from_numpy(m).cuda() for m in loc2], [torch.from_numpy(m).cuda() for m in conf2]
    _, _, _, keep2, (lp2, cp2, _, _, _, _) = _level_args(lm2, cm2, neg_max)
    ws4 = torch.empty(L.fdt_detect_workspace_bytes_depth(B, N, 2, 4), dtype=torch.uint8, device=dev)
    outs = [torch.empty((B, 2, 750, 5), device=dev) for _ in range(4)]

    def c_fused_ring(i):
        a, b_ = (lp, cp) if i % 2 == 0 else (lp2, cp2)
        _lib.check(L.fdt_detect_heads(a, b_, fh, fw, nm, nl, pri.data_ptr(), B, 750, 5000, 0.05, 0.3, 0.1, 0.2, outs[i % 4].data_ptr(), None, None,
                                      ws4.data_ptr(), ws4.numel(), st))
    K = 50
    for i in range(8):
        c_fused_ring(i)
    torch.cuda.synchronize()
    assert torch.equal(outs[0], fused)
    blocks = []
    for _ in range(7):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(2_000_000)
        e0.record()
        for i in range(K):
            c_fused_ring(i)
        e1.record()
        torch.cuda.synchronize()
        blocks.append(e0.elapsed_time(e1) / K)
    ms_b2b = float(np.median(blocks))
    alg = B * (32 * N + 30000) + 16 * N            # conf maps 16 B + loc maps 16 B per prior, output rows, priors once
    cand = float((fused[:, 1, :, 0] > 0).sum(1).float().mean())
    print(json.dumps({"workload": "Detect from per-level NCHW head maps (max-in-out + permute/cat + softmax fused), B=64 @640x640, N=34,125",
                      "fused_ms": ms_f, "fused_ms_min": min_f, "frames_per_s": B / (ms_f * 1e-3),
                      "fused_ms_back_to_back": ms_b2b, "frames_per_s_back_to_back": B / (ms_b2b * 1e-3),
                      "roofline_frac_back_to_back": alg / (ms_b2b * 1e-3) / 1e9 / PEAK,
                      "materialise_then_detect_ms": ms_m, "heads_to_loc_conf_ms": ms_h,
                      "torch_head_ops_then_detect_ms": ms_t, "torch_head_ops_ms": ms_th,
                      "algorithmic_bytes": alg, "roofline_frac_of_measured_hbm": alg / (ms_f * 1e-3) / 1e9 / PEAK,
                      "rows_kept_per_image": cand}))


def heads_train():
    """MultiBoxLoss from the per-level NCHW head maps, B=32 @640x640 (N=34,125), the ground truth of config 3, both matchers:
    forward and forward+backward (gradients down to the maps) for (1) the reference's head ops restated in torch + the library's
    MultiBoxLoss -- the only way to map gradients before fdt_multibox_loss_forward_heads --, (2) fdt_heads_to_loc_conf +
    fdt_multibox_loss_forward (two steps, [B,N,4] / [B,N,2] materialised both ways) and (3) the fused entries."""
    from fdt_b200.layers import MultiBoxLoss, heads_to_loc_conf
    from fdt_b200.layers.functions.heads import _level_args
    from fdt_b200.layers.modules.multibox_loss import pack_targets
    from tests.torch_heads_ref import heads as torch_heads
    B = 32
    pri_np = synth.priors_numpy(640, 640); N = pri_np.shape[0]
    loc_maps, conf_maps, neg_max = synth.head_maps(B, 640, 640, 3032)
    _, _, targets = synth.multibox_inputs(B, pri_np, 3030, 0, 200)
    dev = torch.device("cuda")
    p = torch.from_numpy(pri_np).to(dev)
    tg = [torch.from_numpy(t).to(dev) for t in targets]
    lm, cm = [torch.from_numpy(m).to(dev) for m in loc_maps], [torch.from_numpy(m).to(dev) for m in conf_maps]
    gt, off, G = pack_targets(tg, dev)
    _, _, _, keep, (lp, cp, fh, fw, nm, nl) = _level_args(lm, cm, neg_max)
    L = _lib.lib(); st = _lib.stream_ptr()
    losses = torch.empty(2, device=dev); norm = torch.empty(1, device=dev)
    loc_t = torch.empty((B, N, 4), device=dev); conf_t = torch.empty((B, N), dtype=torch.int64, device=dev)
    sel = torch.empty((B, N), dtype=torch.uint8, device=dev)
    loc_b = torch.empty((B, N, 4), device=dev); conf_b = torch.empty((B, N, 2), device=dev)
    ws = _lib.workspace(L.fdt_multibox_workspace_bytes(B, N, 2, G), dev, "htx")

    def leaves():
        return [m.clone().requires_grad_(True) for m in lm], [m.clone().requires_grad_(True) for m in cm]
    res = {}
    for bip in (False, True):
        crit = MultiBoxLoss(2, 0.35, True, 0, True, 3, 0.35, False, bipartite=bip)

        def c_two_step():
            _lib.check(L.fdt_heads_to_loc_conf(lp, cp, fh, fw, nm, nl, B, 0, loc_b.data_ptr(), conf_b.data_ptr(), st))
            _lib.check(L.fdt_multibox_loss_forward(loc_b.data_ptr(), conf_b.data_ptr(), p.data_ptr(), gt.data_ptr(), off.data_ptr(), G, B, N, 2,
                                                   0.35, 3, int(bip), 0.1, 0.2, losses.data_ptr(), norm.data_ptr(), loc_t.data_ptr(),
                                                   conf_t.data_ptr(), sel.data_ptr(), None, ws.data_ptr(), ws.numel(), st))

        def c_fused():
            _lib.check(L.fdt_multibox_loss_forward_heads(lp, cp, fh, fw, nm, nl, p.data_ptr(), gt.data_ptr(), off.data_ptr(), G, B, 0.35, 3,
                                                         int(bip), 0.1, 0.2, losses.data_ptr(), norm.data_ptr(), loc_t.data_ptr(),
                                                         conf_t.data_ptr(), sel.data_ptr(), None, ws.data_ptr(), ws.numel(), st))
        c_two_step(); torch.cuda.synchronize()
        l2, ct2, s2 = losses.clone(), conf_t.clone(), sel.clone()
        c_fused(); torch.cuda.synchronize()
        fwd_parity = bool(torch.equal(ct2, conf_t) and torch.equal(s2, sel) and torch.allclose(l2, losses, rtol=1e-6, atol=0))

        def torch_fwd():
            with torch.no_grad():
                crit((*torch_heads(lm, cm, neg_max, False), p), tg)

        def fb(path):
            lh, ch = leaves()

            def run():
                if path == "torch":
                    ll, lc = crit((*torch_heads(lh, ch, neg_max, False), p), tg)
                elif path == "two_step":
                    ll, lc = crit((*heads_to_loc_conf(lh, ch, neg_max, softmax=False), p), tg)
                else:
                    ll, lc = crit.forward_heads(lh, ch, p, tg, neg_max)
                (ll + lc).backward()
                return ll, lc, [m.grad for m in lh + ch]
            return run
        outs = {k: fb(k)() for k in ("torch", "two_step", "fused")}
        grads_bit_equal = all(torch.equal(a.view(torch.int32), b.view(torch.int32)) for a, b in zip(outs["two_step"][2], outs["fused"][2]))
        torch_close = all(torch.allclose(a, b, rtol=1e-4, atol=1e-7) for a, b in zip(outs["torch"][2], outs["fused"][2])) and \
            all(torch.allclose(outs["torch"][i], outs["fused"][i], rtol=1e-5) for i in (0, 1))
        r = {"fwd_ms": {"torch_heads_plus_library_loss": timed(torch_fwd)[0], "two_step": timed(c_two_step)[0], "fused": timed(c_fused)[0]},
             "fwd_bwd_ms": {k: timed(fb(k), reps=10)[0] for k in ("torch", "two_step", "fused")},
             "parity": {"fused_fwd_equals_two_step": fwd_parity, "fused_map_grads_bit_equal_two_step": bool(grads_bit_equal),
                        "torch_path_close": bool(torch_close)}}
        r["fused_fwd_beats_two_step"] = r["fwd_ms"]["fused"] < r["fwd_ms"]["two_step"]
        fwd_b = B * 56 * N + 20 * G                    # maps 32 B/prior read, loc_t + conf_t 24 B/prior written, GT rows
        r["fused_fwd_gbs"] = fwd_b / (r["fwd_ms"]["fused"] * 1e-3) / 1e9
        res["bipartite" if bip else "default"] = r
    # backward alone, fused entry, default matcher (the forward above left loc_t / conf_t / sel / norm in place)
    gmaps_l = [torch.empty_like(m) for m in lm]; gmaps_c = [torch.empty_like(m) for m in cm]
    import ctypes as C
    glp = (C.c_void_p * nl)(*[t.data_ptr() for t in gmaps_l]); gcp = (C.c_void_p * nl)(*[t.data_ptr() for t in gmaps_c])
    one = torch.ones((), device=dev)

    def c_bwd():
        _lib.check(L.fdt_multibox_loss_backward_heads_dev(lp, cp, fh, fw, nm, nl, loc_t.data_ptr(), conf_t.data_ptr(), sel.data_ptr(),
                                                          norm.data_ptr(), one.data_ptr(), one.data_ptr(), B, glp, gcp, st))
    ms_bwd, _ = timed(c_bwd)
    print(json.dumps({"workload": "MultiBoxLoss from per-level NCHW head maps, B=32 @640x640 (N=34,125), GT of config 3", "gt_total": G,
                      "device": torch.cuda.get_device_name(), "results": res,
                      "fused_fwd_algorithmic_bytes": B * 56 * N + 20 * G, "fused_bwd_algorithmic_bytes": B * 89 * N,
                      "fused_bwd_ms": ms_bwd, "fused_bwd_gbs": B * 89 * N / (ms_bwd * 1e-3) / 1e9,
                      "materialisation_removed_bytes": {"forward": B * 56 * N, "backward": B * 72 * N}}))


def match_mine():
    """The standalone entries, which share the fused forward's kernels: fdt_match_encode at config 3 (B=32, N=34,125, both matchers)
    and as FaceBoxes' DataEncoder.encode calls it (B=1, the 21,824 default boxes, 10 GT boxes, bipartite); fdt_hard_negative_mine
    (B=32, N=34,125) on the fused forward's loss_c of config 3 and on rows of ties, equal zeros and quarter steps.  outputs_sha1
    identifies the outputs, so that two builds can be compared."""
    import hashlib
    from fdt_b200.layers.modules.multibox_loss import pack_targets
    L = _lib.lib(); st = _lib.stream_ptr()
    dev = torch.device("cuda")

    def sha(*ts):
        h = hashlib.sha1()
        for t in ts:
            h.update(t.cpu().numpy().tobytes())
        return h.hexdigest()[:16]

    def match_case(pri_np, gt, off, total, B, bip):
        N = pri_np.shape[0]
        p = torch.from_numpy(pri_np).to(dev)
        lt = torch.empty((B, N, 4), device=dev); ct = torch.empty((B, N), dtype=torch.int64, device=dev)
        bti = torch.empty((B, N), dtype=torch.int32, device=dev); bto = torch.empty((B, N), device=dev)
        ws = _lib.workspace(L.fdt_match_workspace_bytes(B, N, total), dev, "mm")

        def run():
            _lib.check(L.fdt_match_encode(p.data_ptr(), gt.data_ptr(), off.data_ptr(), total, B, N, 0.35, 0.1, 0.2, bip, lt.data_ptr(),
                                          ct.data_ptr(), bti.data_ptr(), bto.data_ptr(), ws.data_ptr(), ws.numel(), st))
        run(); torch.cuda.synchronize()
        ms, ms_min = timed(run)
        return {"ms": ms, "ms_min": ms_min, "outputs_sha1": sha(lt, ct, bti, bto)}

    res = {}
    B = 32
    pri = synth.priors_numpy(640, 640); N = pri.shape[0]
    _, _, targets = synth.multibox_inputs(B, pri, 3030, 0, 200)
    gt, off, G = pack_targets([torch.from_numpy(t).to(dev) for t in targets], dev)
    for bip in (0, 1):
        res[f"match_b32_config3_{'bipartite' if bip else 'default'}"] = match_case(pri, gt, off, G, B, bip)
    fb = orc.facebox_default_boxes()
    g10 = torch.from_numpy(synth.gt_boxes(10, np.random.Generator(np.random.PCG64(7)))).to(dev)
    res["match_b1_faceboxes_bipartite"] = match_case(fb, g10, torch.tensor([0, 10], dtype=torch.int64, device=dev), 10, 1, 1)

    # mining inputs: the loss_c and positives of the fused forward (config 3, default matcher), and the tie-heavy rows
    loc, conf, _ = synth.multibox_inputs(B, pri, 3030, 0, 200)
    l, c, p = (torch.from_numpy(a).to(dev) for a in (loc, conf, pri))
    lca = torch.empty((B, N), device=dev); ct = torch.empty((B, N), dtype=torch.int64, device=dev)
    ws = _lib.workspace(L.fdt_multibox_workspace_bytes(B, N, 2, G), dev, "mmf")
    _lib.check(L.fdt_multibox_loss_forward(l.data_ptr(), c.data_ptr(), p.data_ptr(), gt.data_ptr(), off.data_ptr(), G, B, N, 2, 0.35, 3, 0,
                                           0.1, 0.2, torch.empty(2, device=dev).data_ptr(), torch.empty(1, device=dev).data_ptr(),
                                           torch.empty((B, N, 4), device=dev).data_ptr(), ct.data_ptr(),
                                           torch.empty((B, N), dtype=torch.uint8, device=dev).data_ptr(), lca.data_ptr(), ws.data_ptr(),
                                           ws.numel(), st))
    rng = np.random.Generator(np.random.PCG64(34125 + 50))
    lc_t = rng.uniform(0, 5, (B, N)).astype(np.float32)
    lc_t[1::3] = np.round(lc_t[1::3] * 4) / 4
    lc_t[2::3, ::2] = 0.0
    pos_t = np.zeros((B, N), bool)
    for b in range(B):
        pos_t[b, rng.permutation(N)[:50]] = True
    lc_t[pos_t] = 0
    for name, lc, ps in (("mine_b32_config3_loss_c", lca, (ct > 0).to(torch.uint8)),
                         ("mine_b32_ties", torch.from_numpy(lc_t).to(dev), torch.from_numpy(pos_t.astype(np.uint8)).to(dev))):
        neg = torch.empty((B, N), dtype=torch.uint8, device=dev)
        ws = _lib.workspace(L.fdt_mine_workspace_bytes(B, N), dev, "mm")

        def run():
            _lib.check(L.fdt_hard_negative_mine(lc.data_ptr(), ps.data_ptr(), B, N, 3, neg.data_ptr(), ws.data_ptr(), ws.numel(), st))
        run(); torch.cuda.synchronize()
        ms, ms_min = timed(run)
        res[name] = {"ms": ms, "ms_min": ms_min, "outputs_sha1": sha(neg)}
    print(json.dumps({"workload": "fdt_match_encode (B=32 config 3 default/bipartite; B=1 FaceBoxes 21,824 boxes, 10 GT, bipartite) and "
                      "fdt_hard_negative_mine (B=32, N=34,125: config 3 loss_c; tie-heavy rows)", "device": torch.cuda.get_device_name(),
                      "results": res}))


def heads_amp():
    """Mixed-precision / channels_last head maps read in place vs today's conversion path (each map converted to fp32 NCHW first,
    [m.float().contiguous() ...]), at the heads / heads_train shapes: Detect B=64 and MultiBoxLoss B=32 (config 3 ground truth),
    both at 640x640 (N=34,125).  Cases: fp32 NCHW, bf16 NCHW and channels_last (converted and native), fp16 NCHW native.  Every
    native result is checked equal to its conversion-path twin in the same run.  Bytes are algorithmic, from the shapes: Detect
    reads the conf maps (4 channels x sizeof(T) per prior and image); the loss reads the loc and conf maps at sizeof(T) and writes
    its targets as today (loc_t 16, conf_t 8, sel 1 bytes per prior and image)."""
    from fdt_b200.layers import Detect, MultiBoxLoss
    N = synth.priors_numpy(640, 640).shape[0]
    pri = torch.from_numpy(synth.priors_numpy(640, 640)).cuda()

    def make(B, seed, dtype, layout):
        lm, cm, nm = synth.head_maps(B, 640, 640, seed)
        out = []
        for maps in (lm, cm):
            ms = [torch.from_numpy(m).to(dtype).cuda() for m in maps]
            out.append([m.contiguous(memory_format=torch.channels_last) for m in ms] if layout == "channels_last" else ms)
        return out[0], out[1], nm

    def convert(maps):
        return [m.float().contiguous() for m in maps]
    cases = [("fp32_nchw", torch.float32, "nchw", False), ("bf16_nchw_converted", torch.bfloat16, "nchw", True),
             ("bf16_nchw_native", torch.bfloat16, "nchw", False), ("bf16_cl_converted", torch.bfloat16, "channels_last", True),
             ("bf16_cl_native", torch.bfloat16, "channels_last", False), ("fp16_nchw_native", torch.float16, "nchw", False)]
    res = {}
    # ---- Detect, B = 64
    B = 64
    det = Detect(2, 0, 750, 0.05, 0.3)
    ref = {}
    for name, dtype, layout, conv in cases:
        sets = [make(B, 6060 + i, dtype, layout) for i in range(2)]

        def call(i):
            lm, cm, nm = sets[i % 2]
            return det.detect_heads(convert(lm) if conv else lm, convert(cm) if conv else cm, pri, nm)
        key = (dtype, layout)
        out = call(0)
        if key in ref:
            assert torch.equal(out, ref[key]), name
        ref[key] = out
        ms, ms_min = timed(lambda: call(0))
        for i in range(8):
            call(i)
        torch.cuda.synchronize()
        blocks = []
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(2_000_000)
            e0.record()
            for i in range(50):
                call(i)
            e1.record()
            torch.cuda.synchronize()
            blocks.append(e0.elapsed_time(e1) / 50)
        esz = torch.tensor([], dtype=dtype).element_size()
        res["detect_b64_" + name] = {"isolated_ms": ms, "isolated_ms_min": ms_min, "back_to_back_ms": float(np.median(blocks)),
                                     "conf_map_bytes": B * 4 * N * esz}
    # ---- MultiBoxLoss, B = 32
    B = 32
    _, _, targets = synth.multibox_inputs(B, synth.priors_numpy(640, 640), 3030, 0, 200)
    tg = [torch.from_numpy(t).cuda() for t in targets]
    crit = MultiBoxLoss(2, 0.35, True, 0, True, 3, 0.35, False)
    ref = {}
    for name, dtype, layout, conv in cases:
        lm0, cm0, nm = make(B, 3032, dtype, layout)
        lm = [m.requires_grad_(True) for m in lm0]
        cm = [m.requires_grad_(True) for m in cm0]

        def fwd():
            with torch.no_grad():
                return crit.forward_heads(convert(lm) if conv else lm, convert(cm) if conv else cm, pri, tg, nm)

        def fwd_bwd():
            for m in lm + cm:
                m.grad = None
            ll, lc = crit.forward_heads(convert(lm) if conv else lm, convert(cm) if conv else cm, pri, tg, nm)
            (ll + lc).backward()
            return ll, lc
        ll, lc = fwd_bwd()
        got = (float(ll.detach()), float(lc.detach()), [m.grad.clone() for m in lm + cm])
        key = (dtype, layout)
        if key in ref:
            assert got[:2] == ref[key][:2], name
            assert all(torch.equal(a, b) for a, b in zip(got[2], ref[key][2])), name
        ref[key] = got
        ms_f, _ = timed(fwd)
        ms_fb, _ = timed(fwd_bwd)
        esz = torch.tensor([], dtype=dtype).element_size()
        res["loss_b32_" + name] = {"forward_ms": ms_f, "forward_backward_ms": ms_fb,
                                   "forward_bytes": B * N * (8 * esz + 16 + 8 + 1)}
    print(json.dumps({"workload": "head maps as the network wrote them (bf16 / fp16, NCHW / channels_last) vs converted to fp32 NCHW; "
                      "Detect B=64 and MultiBoxLoss B=32 @640x640", **card(), "results": res}))


def flat_amp():
    """Flat loc[B,N,4] / conf[B,N,C] of 16-bit dtypes read in place vs the conversion path (loc.float(), conf.float() before the call,
    which is what every non-fp32 input cost before).  Rows: Detect B=64 @640x640 isolated and back to back for fp32, (bf16 loc, fp32
    conf) = inference under autocast, bf16 / bf16 and fp16 / fp16 (plus `fp32_same_values`: the fp32 call on the 16-bit values converted
    before timing, which separates what reading 16-bit data costs from what the coarser scores cost); Detect B=512 @1024x1024 bf16 (more lists than SMs: K2 + k_sort_nms);
    Detect.submit streamed from pinned host tensors, fp16 against fp32 (two batches in flight); MultiBoxLoss B=32 @640x640 bf16 forward
    and forward + backward through the autograd module, both matchers.  `equal` = the in-place result is bit-identical to the
    conversion path's in this run.  tie_runs: per dtype, the images whose nms_top_k best candidates hold a run of more than 512 equal
    scores (a bucket too large for k_sort_nms' per-window ranking: its bitonic fallback) -- a count from the inputs, not a kernel
    counter."""
    from fdt_b200.layers import Detect, MultiBoxLoss
    res = {}

    def b2b(call, n=50):
        for i in range(8):
            call(i)
        torch.cuda.synchronize()
        blocks = []
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(2_000_000)
            e0.record()
            for i in range(n):
                call(i)
            e1.record()
            torch.cuda.synchronize()
            blocks.append(e0.elapsed_time(e1) / n)
        return float(np.median(blocks))

    def tie_runs(conf, k=5000, run=512):
        s = conf[..., 1].float()
        top = torch.topk(torch.where(s > 0.05, s, torch.full_like(s, -1.0)), k, dim=1).values
        n = 0
        for row in top:
            row = row[row > 0.05]
            if row.numel() and int(torch.unique(row, return_counts=True)[1].max()) > run:
                n += 1
        return n

    def detect_rows(B, w, prefix, cases, n_b2b=50):
        pri = torch.from_numpy(synth.priors_numpy(w, w)).cuda()
        raw = [synth.detect_inputs(B, synth.priors_numpy(w, w), 7070 + i) for i in range(2)]
        det = Detect(2, 0, 750, 0.05, 0.3)
        for name, ldt, cdt in cases:
            sets = [(torch.from_numpy(l).to(ldt).cuda(), torch.from_numpy(c).to(cdt).cuda()) for l, c in raw]
            up = [(l.float(), c.float()) for l, c in sets]
            row = {}
            for mode in ("converted", "in_place", "fp32_same_values"):
                def call(i, mode=mode):
                    l, c = sets[i % 2]
                    if mode == "fp32_same_values":          # the fp32 call on the rounded values, converted before timing
                        return det(*up[i % 2], pri)
                    return det(l.float(), c.float(), pri) if mode == "converted" else det(l, c, pri)
                row[mode + "_isolated_ms"], _ = timed(lambda: call(0))
                row[mode + "_back_to_back_ms"] = b2b(call, n_b2b)
            a = det(*sets[0], pri, return_aux=True)
            b = det(sets[0][0].float(), sets[0][1].float(), pri, return_aux=True)
            row["equal"] = all(torch.equal(x.view(torch.uint8), y.view(torch.uint8)) for x, y in zip(a, b))
            row["tie_runs_over_512"] = tie_runs(sets[0][1])
            res[prefix + name] = row
    F32, BF, HF = torch.float32, torch.bfloat16, torch.float16
    detect_rows(64, 640, "detect_b64_640_", [("fp32", F32, F32), ("bf16loc_fp32conf", BF, F32), ("bf16", BF, BF), ("fp16", HF, HF)])
    detect_rows(512, 1024, "detect_b512_1024_", [("bf16", BF, BF)], n_b2b=10)
    # ---- Detect.submit from pinned host tensors, two batches in flight (the host path is bound by the conf copy)
    B = 64
    pri_h = torch.from_numpy(synth.priors_numpy(640, 640))
    l0, c0 = synth.detect_inputs(B, synth.priors_numpy(640, 640), 7171)
    det = Detect(2, 0, 750, 0.05, 0.3)
    for name, dt in (("fp32", F32), ("fp16", HF)):
        l, c = torch.from_numpy(l0).to(dt).pin_memory(), torch.from_numpy(c0).to(dt).pin_memory()
        out = det.submit(l, c, pri_h).result()
        for _ in range(4):
            det.submit(l, c, pri_h).result()
        n, t0 = 40, time.perf_counter()
        pend = [det.submit(l, c, pri_h)]
        for _ in range(n - 1):
            pend.append(det.submit(l, c, pri_h))
            pend.pop(0).result()
        pend.pop(0).result()
        dtm = (time.perf_counter() - t0) / n * 1e3
        up = det.submit(l.float(), c.float(), pri_h).result()
        res["detect_submit_b64_640_pinned_" + name] = {"ms_per_batch": dtm, "conf_bytes": B * c.shape[1] * 2 * c.element_size(),
                                                       "equal": bool(torch.equal(out.view(torch.uint8), up.view(torch.uint8)))}
    # ---- MultiBoxLoss B = 32, bf16 (training under autocast), through the autograd module
    B = 32
    pri = torch.from_numpy(synth.priors_numpy(640, 640)).cuda()
    l0, c0, targets = synth.multibox_inputs(B, synth.priors_numpy(640, 640), 3030, 0, 200)
    tg = [torch.from_numpy(t).cuda() for t in targets]
    for bip in (False, True):
        crit = MultiBoxLoss(2, 0.35, True, 0, True, 3, 0.35, False, bipartite=bip)
        loc = torch.from_numpy(l0).to(BF).cuda().requires_grad_(True)
        conf = torch.from_numpy(c0).to(BF).cuda().requires_grad_(True)
        row, got = {}, {}
        for mode in ("converted", "in_place"):
            def args(mode=mode):
                return (loc.float(), conf.float(), pri) if mode == "converted" else (loc, conf, pri)

            def fwd():
                with torch.no_grad():
                    return crit(args(), tg)

            def fwd_bwd():
                loc.grad = conf.grad = None
                ll, lc = crit(args(), tg)
                (ll + lc).backward()
                return ll, lc
            ll, lc = fwd_bwd()
            got[mode] = (float(ll.detach()), float(lc.detach()), loc.grad.view(torch.int16).clone(), conf.grad.view(torch.int16).clone())
            row[mode + "_forward_ms"], _ = timed(fwd)
            row[mode + "_forward_backward_ms"], _ = timed(fwd_bwd)
        a, b = got["converted"], got["in_place"]
        row["equal"] = a[:2] == b[:2] and torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])
        res["loss_b32_640_bf16_" + ("bipartite" if bip else "default")] = row
    print(json.dumps({"workload": "flat loc / conf in bf16 / fp16 read in place vs converted to fp32 first: Detect B=64 @640^2 and "
                      "B=512 @1024^2, Detect.submit from pinned host tensors, MultiBoxLoss B=32 @640^2", **card(), "results": res}))


def card():
    """name and power limit of the GPU the numbers of this run come from"""
    import subprocess
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        pl = "unknown"
    return {"device": torch.cuda.get_device_name(), "power_limit": pl}


def track_stream():
    """Online multi-stream tracker (StreamTracker / fdt_track_stream_step): V in {1, 64, 148} streams x 2,000 config-4-shaped
    frames each (one seed per stream), one frame per stream per step, steps back to back (eagerly through the C ABI, and replayed
    from one CUDA graph holding all steps); against the same videos through the offline fdt_iou_track, one call per video, back to
    back; and the live pipeline Detect (B=64 @640^2) + step_detections per step against Detect alone."""
    from fdt_b200 import tracker as T
    from fdt_b200.layers import Detect
    L = _lib.lib()
    dev = torch.device("cuda")
    st_ptr = _lib.stream_ptr
    F, MAXD = 2000, 300
    res = {}
    for V in (1, 64, 148):
        videos = [synth.tracker_frames(F=F, seed=4040 + v, d_lo=1, d_hi=300, n_objects=300, empty_every=1000) for v in range(V)]
        steps = []                                               # per step: packed rows of the V current frames (device)
        for f in range(F):
            d, o = T.pack_frames([videos[v][f] for v in range(V)])
            steps.append((torch.from_numpy(d).to(dev), torch.from_numpy(o).to(dev)))
        tr = T.StreamTracker(V, MAXD)
        rt = torch.empty(max(int(s[0].shape[0]) for s in steps), dtype=torch.int64, device=dev)
        rec = tr._records()

        def step(s):
            d, o = steps[s]
            _lib.check(L.fdt_track_stream_step(tr._state.data_ptr(), V, MAXD, d.data_ptr(), o.data_ptr(), None, rt.data_ptr(),
                                               rec["fin_count"].data_ptr(), rec["fin_index"].data_ptr(), rec["fin_track"].data_ptr(),
                                               rec["fin_start"].data_ptr(), rec["fin_len"].data_ptr(), rec["fin_max"].data_ptr(),
                                               tr._ws.data_ptr(), tr._ws.numel(), st_ptr()))

        def reinit():
            _lib.check(L.fdt_track_stream_init(tr._state.data_ptr(), tr._state.numel(), V, MAXD, 0, 0.4, 0.6, 5, st_ptr()))

        def eager():
            for s in range(F):
                step(s)
        reinit(); eager(); torch.cuda.synchronize()             # warm-up
        t_eager = []
        for _ in range(3):
            reinit(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); eager(); e1.record(); torch.cuda.synchronize()
            t_eager.append(e0.elapsed_time(e1))
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            reinit()
        torch.cuda.current_stream().wait_stream(side)
        with torch.cuda.graph(g):
            eager()
        t_graph = []
        for _ in range(3):
            reinit(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
            t_graph.append(e0.elapsed_time(e1))
        del g

        # parity: every stream's steps + flush against offline fdt_iou_track on its video (row grouping, start, length, max)
        reinit()
        ids, recs = [], []
        for s in range(F):
            o = tr.step(*steps[s]); ids.append(o["row_track"]); recs.append(o)
        recs.append(tr.flush())
        ids_h = [x.cpu().numpy() for x in ids]
        recs_h = [{k: t.cpu().numpy() for k, t in r.items() if k != "row_track"} for r in recs]
        offs_h = [s[1].cpu().numpy() for s in steps]
        same = True
        for v in range(V):
            d, o = T.pack_frames(videos[v])
            t_off, t_dets, t_start, t_max = (x.cpu().numpy() for x in T.iou_track_raw(d, o))
            lab = np.full(int(o[-1]), -1, np.int64)
            lab[t_dets] = np.repeat(np.arange(len(t_start)), np.diff(t_off))
            idv = np.concatenate([ids_h[s][offs_h[s][v]:offs_h[s][v + 1]] for s in range(F)])
            fin = [(int(r["fin_index"][v, k]), int(r["fin_track"][v, k]), int(r["fin_start"][v, k]), int(r["fin_len"][v, k]),
                    float(r["fin_max"][v, k])) for r in recs_h for k in range(int(r["fin_count"][v]))]
            fin.sort()
            ok = [x[0] for x in fin] == list(range(len(t_start)))
            ok = ok and all((x[2], x[3], x[4]) == (int(t_start[i]), int(t_off[i + 1] - t_off[i]), float(t_max[i])) for i, x in enumerate(fin))
            idmap = np.full(int(idv.max(initial=0)) + 2, -1, np.int64)
            idmap[[x[1] for x in fin]] = [x[0] for x in fin]
            lab2 = idmap[idv]
            same = same and ok and np.array_equal(lab, lab2)
        status = tr.status()

        # what users do today: the offline tracker, one call per video, back to back
        packed = []
        for v in range(V):
            d, o = T.pack_frames(videos[v])
            total = int(o[-1]); md = int(np.diff(o).max())
            packed.append((torch.from_numpy(d).to(dev), torch.from_numpy(o).to(dev), total, md,
                           torch.empty(max(int(L.fdt_iou_track_workspace_bytes(F, total, md)), 256), dtype=torch.uint8, device=dev)))
        n = torch.zeros(1, dtype=torch.int64, device=dev)
        tot_max = max(p[2] for p in packed)
        t_off = torch.zeros(tot_max + 2, dtype=torch.int64, device=dev); t_dets = torch.zeros(tot_max, dtype=torch.int64, device=dev)
        t_start = torch.zeros(tot_max + 1, dtype=torch.int64, device=dev); t_max = torch.zeros(tot_max + 1, dtype=torch.float64, device=dev)

        def offline():
            for d, o, total, md, ws in packed:
                _lib.check(L.fdt_iou_track(d.data_ptr(), o.data_ptr(), F, total, md, 0.4, 0.6, 5, n.data_ptr(), t_off.data_ptr(),
                                           t_dets.data_ptr(), t_start.data_ptr(), t_max.data_ptr(), ws.data_ptr(), ws.numel(), st_ptr()))
        ms_off, ms_off_min = timed(offline, reps=3, warm=1)
        ge = min(t_graph)
        res[f"V{V}"] = {"streams": V, "frames_per_stream": F, "detections": int(sum(int(s[1][-1]) for s in steps)),
                        "step_us_eager": min(t_eager) * 1e3 / F, "step_us_graph": ge * 1e3 / F,
                        "frames_per_s_graph": V * F / (ge * 1e-3), "frames_per_s_eager": V * F / (min(t_eager) * 1e-3),
                        "offline_ms_all_videos": ms_off, "offline_frames_per_s": V * F / (ms_off * 1e-3),
                        "offline_us_per_frame": ms_off * 1e3 / (V * F), "identical_to_offline": bool(same), "status": status}
        del steps, packed, ids, recs
        torch.cuda.empty_cache()

    # live pipeline: Detect at the headline configuration + one step_detections per step
    B = 64
    pri = synth.priors_numpy(640, 640)
    loc, conf = synth.detect_inputs(B, pri, 4242, 0.05)
    det = Detect(2, 0, 750, 0.05, 0.3)
    a = [torch.from_numpy(x).cuda() for x in (loc, conf, pri)]
    live = T.StreamTracker(B)
    ms_det, _ = timed(lambda: det(*a))
    ms_live, _ = timed(lambda: live.step_detections(det(*a), 640.0, 640.0))
    out = live.step_detections(det(*a), 640.0, 640.0)
    res["live_detect_b64_640"] = {"detect_ms": ms_det, "detect_plus_step_ms": ms_live, "step_ms_added": ms_live - ms_det,
                                  "rows_per_step": int(out["frame_off"][-1]), "status": live.status()}
    print(json.dumps({"workload": "online multi-stream IoU tracker: V streams x 2,000 config-4-shaped frames, one frame per stream "
                      "per step; offline fdt_iou_track per video for comparison; Detect B=64 @640^2 + step_detections",
                      **card(), "results": res}))


if __name__ == "__main__":
    for w in sys.argv[1:] or ["multibox", "tracker", "detect1024", "priorbox", "heads", "siblings"]:
        globals()[w]()
