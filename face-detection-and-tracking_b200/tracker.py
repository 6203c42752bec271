"""IoU tracker -- drop-in for the association loop of iouTracke_cal.py (:126-155, flush :174-176; use_iou=True or False)
and its `.npy` output (:177, consumed by iouTracke_display.py:29), computed by fdt_iou_track_metric on the GPU."""
from __future__ import annotations

import numpy as np
import torch

from . import _lib

# module-level defaults of the reference script (iouTracke_cal.py:22-28)
use_iou = True
sigma_iou = 0.4
sigma_dis = 8
sigma_h = 0.6
t_min = 5


def pack_frames(frames):
    """list of per-frame [D_f, 5] arrays (what detect_face returns, iouTracke_cal.py:70-84; float32 rows or
    the float64 dummy [[0,0,0,0,0.4]]) -> (dets[total,5] float64, frame_off[F+1] int64).
    The reference widens to python floats with det0.tolist() (:127), i.e. float64, exactly like this."""
    arrs = [np.asarray(f, dtype=np.float64).reshape(-1, 5) for f in frames]
    off = np.zeros(len(arrs) + 1, np.int64)
    if arrs:
        np.cumsum([a.shape[0] for a in arrs], out=off[1:])
    dets = np.concatenate(arrs, 0) if off[-1] > 0 else np.zeros((1, 5), np.float64)
    return dets, off


def iou_track_raw(dets, frame_off, sigma_iou=sigma_iou, sigma_h=sigma_h, t_min=t_min, use_iou=use_iou, sigma_dis=sigma_dis):
    """dets[total,5] float64 + frame_off[F+1] (numpy or torch, host or device)
    -> (track_off[T+1], track_dets[rows], track_start[T], track_max[T]) as CUDA tensors; tracks are in the
    reference's finishing order, track_dets are global detection rows in append order."""
    dev = _lib.require_cuda()
    d = torch.as_tensor(dets, dtype=torch.float64).to(dev).contiguous()
    off_h = torch.as_tensor(frame_off, dtype=torch.int64).cpu()
    off = off_h.to(dev)
    F = off_h.numel() - 1
    total = int(off_h[-1])
    max_d = int((off_h[1:] - off_h[:-1]).max()) if F > 0 else 0
    n = torch.zeros(1, dtype=torch.int64, device=dev)
    t_off = torch.zeros(total + 2, dtype=torch.int64, device=dev)
    t_dets = torch.zeros(max(total, 1), dtype=torch.int64, device=dev)
    t_start = torch.zeros(total + 1, dtype=torch.int64, device=dev)
    t_max = torch.zeros(total + 1, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        L = _lib.lib()
        ws = _lib.workspace(L.fdt_iou_track_workspace_bytes(F, total, max_d), dev, "track")
        _lib.check(L.fdt_iou_track_metric(_lib.ptr(d), _lib.ptr(off), F, total, max_d, 0 if use_iou else 1,
                                          float(sigma_iou if use_iou else sigma_dis), float(sigma_h),
                                          int(t_min), _lib.ptr(n), _lib.ptr(t_off), _lib.ptr(t_dets), _lib.ptr(t_start),
                                          _lib.ptr(t_max), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
    T = int(n.item())
    rows = int(t_off[T].item()) if T else 0
    return t_off[:T + 1], t_dets[:rows], t_start[:T], t_max[:T]


def detections_to_frames(detections, width, height, thresh=0.4, shrink=1.0):
    """Detect output of a whole clip, detections [F, C, top_k, 5] on the GPU (one image per frame), -> (dets [total, 5] float64,
    frame_off [F+1] int64), both CUDA tensors, exactly the per-frame arrays detect_face builds (iouTracke_cal.py:55-84: leading rows
    with score >= thresh class by class, boxes * (w, h, w, h) and / shrink in fp32, the dummy row [0, 0, 0, 0, 0.4] for a
    frame without detections) packed back to back: the tracker's input without a round trip through host lists."""
    dev = _lib.require_cuda()
    d = _lib.dev_f32(detections, detections.device if detections.is_cuda else dev)
    F, C_, K, _ = d.shape
    n_rows = torch.empty(max(F, 1), dtype=torch.int32, device=d.device)
    off = torch.empty(F + 1, dtype=torch.int64, device=d.device)
    with torch.cuda.device(d.device):
        L = _lib.lib()
        _lib.check(L.fdt_detections_to_frames_count(_lib.ptr(d), F, C_, K, float(thresh), _lib.ptr(n_rows), _lib.ptr(off), _lib.stream_ptr()))
        total = int(off[-1].item())                      # the one host read: sizes the packed array
        dets = torch.empty((max(total, 1), 5), dtype=torch.float64, device=d.device)
        _lib.check(L.fdt_detections_to_frames_pack(_lib.ptr(d), F, C_, K, float(thresh), float(width), float(height), float(shrink),
                                                   _lib.ptr(off), _lib.ptr(dets), _lib.stream_ptr()))
    return dets[:total] if total else dets[:0], off


def track_detections(detections, width, height, thresh=0.4, shrink=1.0, **kw):
    """detections [F, C, top_k, 5] (CUDA) -> tracks_finished, everything up to the final read-out on the device:
    detections_to_frames + iou_track_raw (iouTracke_cal.py:55-84 feeding :126-155)."""
    dets, off = detections_to_frames(detections, width, height, thresh, shrink)
    t_off, t_dets, t_start, t_max = iou_track_raw(dets, off, **kw)
    t_off, t_dets = t_off.cpu().numpy(), t_dets.cpu().numpy()
    boxes = dets.cpu().numpy()[t_dets, :4] if t_dets.size else np.zeros((0, 4))
    return [{'bboxes': boxes[t_off[t]:t_off[t + 1]].tolist(), 'max_score': float(t_max[t]),
             'start_frame': int(t_start[t])} for t in range(len(t_start))]


def iou_track(frames, sigma_iou=sigma_iou, sigma_h=sigma_h, t_min=t_min, use_iou=use_iou, sigma_dis=sigma_dis):
    """Run the tracker over a whole video.  -> tracks_finished: list of
    {'bboxes': [[x1,y1,x2,y2], ...], 'max_score': float, 'start_frame': int}, the structure
    iouTracke_cal.py:150-154 builds and :177 saves ("track ID" = index in this list)."""
    dets, off = pack_frames(frames)
    t_off, t_dets, t_start, t_max = iou_track_raw(dets, off, sigma_iou, sigma_h, t_min, use_iou, sigma_dis)
    t_off, t_dets = t_off.cpu().numpy(), t_dets.cpu().numpy()
    t_start, t_max = t_start.cpu().numpy(), t_max.cpu().numpy()
    boxes = dets[t_dets, :4]
    return [{'bboxes': boxes[t_off[t]:t_off[t + 1]].tolist(), 'max_score': float(t_max[t]),
             'start_frame': int(t_start[t])} for t in range(len(t_start))]


class StreamTracker:
    """Online tracker for many videos at once: every step() advances each of `num_streams` streams by one frame
    (iouTracke_cal.py:117-155 run inside the video loop, one loop per stream), flush() ends their videos (:174-176).  The
    active tracks live on the device (fdt_track_stream_*); no call synchronises with the host except check() and
    tracks_finished(), so a Detect -> step_detections chain can be captured in a CUDA graph.

    A step returns device tensors: `row_track[rows]` int64, the stream-local id of the track each input row joined or started
    (ids count from 0 per video in creation order; -1 for the rows of a stream that was not advanced or whose frame had more than
    cap = 32 * ceil(max_dets_per_frame / 32) rows, which is then skipped and flagged -- see check(); frames of up to cap rows are
    tracked), and the tracks the step finished,
    `fin_count[V]` int32 and `[V, cap]` records `fin_index` (index in the reference's tracks_finished = its "track ID"),
    `fin_track` (id), `fin_start` (1-based frame), `fin_len`, `fin_max`.  For every stream, steps + flush give exactly
    iou_track(that stream's frames).  max_dets_per_frame is at most 864."""

    def __init__(self, num_streams, max_dets_per_frame=800, sigma_iou=sigma_iou, sigma_h=sigma_h, t_min=t_min, use_iou=use_iou,
                 sigma_dis=sigma_dis, keep_history=False, device=None):
        self.device = _lib.require_cuda() if device is None else torch.device(device)
        self.V, self.max_d = int(num_streams), int(max_dets_per_frame)
        self.cap = 32 * max(1, (self.max_d + 31) // 32)
        L = _lib.lib()
        with torch.cuda.device(self.device):
            self._state = torch.empty(max(int(L.fdt_track_stream_state_bytes(self.V, self.max_d)), 256), dtype=torch.uint8,
                                      device=self.device)
            self._ws = torch.empty(max(int(L.fdt_track_stream_workspace_bytes(self.V, self.max_d)), 256), dtype=torch.uint8,
                                   device=self.device)
            _lib.check(L.fdt_track_stream_init(_lib.ptr(self._state), self._state.numel(), self.V, self.max_d, 0 if use_iou else 1,
                                               float(sigma_iou if use_iou else sigma_dis), float(sigma_h), int(t_min), _lib.stream_ptr()))
        self.keep_history = keep_history
        self._history = []                    # ("step", dets, frame_off, advance, row_track, records) / ("flush", streams, records)

    def _records(self):
        V, cap, dev = self.V, self.cap, self.device
        i64 = dict(dtype=torch.int64, device=dev)
        return dict(fin_count=torch.empty(V, dtype=torch.int32, device=dev), fin_index=torch.empty((V, cap), **i64),
                    fin_track=torch.empty((V, cap), **i64), fin_start=torch.empty((V, cap), **i64), fin_len=torch.empty((V, cap), **i64),
                    fin_max=torch.empty((V, cap), dtype=torch.float64, device=dev))

    def _mask(self, m):
        if m is None:
            return None
        m = torch.as_tensor(m).to(device=self.device, dtype=torch.uint8).contiguous()
        if m.numel() != self.V:
            raise ValueError(f"expected {self.V} per-stream flags, got {m.numel()}")
        return m

    def step(self, dets, frame_off, advance=None):
        """dets [rows, 5] float64 and frame_off [V+1] int64 (device or host; stream v's frame = dets[frame_off[v]:frame_off[v+1]]),
        advance [V] bool (None = all).  -> dict of device tensors: row_track and the finish records (see the class)."""
        d = torch.as_tensor(dets, dtype=torch.float64).to(self.device).reshape(-1, 5).contiguous()
        off = torch.as_tensor(frame_off, dtype=torch.int64).to(self.device).contiguous()
        if off.numel() != self.V + 1:
            raise ValueError(f"frame_off needs {self.V + 1} entries, got {off.numel()}")
        if d.shape[0] == 0:
            d = torch.zeros((1, 5), dtype=torch.float64, device=self.device)
        adv = self._mask(advance)
        out = self._records()
        out["row_track"] = torch.empty(d.shape[0], dtype=torch.int64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().fdt_track_stream_step(
                _lib.ptr(self._state), self.V, self.max_d, _lib.ptr(d), _lib.ptr(off), _lib.ptr(adv), _lib.ptr(out["row_track"]),
                _lib.ptr(out["fin_count"]), _lib.ptr(out["fin_index"]), _lib.ptr(out["fin_track"]), _lib.ptr(out["fin_start"]),
                _lib.ptr(out["fin_len"]), _lib.ptr(out["fin_max"]), _lib.ptr(self._ws), self._ws.numel(), _lib.stream_ptr()))
        if self.keep_history:
            self._history.append(("step", d, off, adv, out))
        return out

    def step_detections(self, detections, width, height, thresh=0.4, shrink=1.0, advance=None):
        """Detect output [V, C, top_k, 5] (one current image per stream) -> step(): detect_face's read-out (iouTracke_cal.py:55-84,
        see detections_to_frames) packed into an upper-bound buffer of V*C*top_k rows, all on the device with no host read."""
        d = _lib.dev_f32(detections, self.device)
        V, C_, K, _ = d.shape
        if V != self.V:
            raise ValueError(f"detections hold {V} images, the tracker {self.V} streams")
        n_rows = torch.empty(max(V, 1), dtype=torch.int32, device=self.device)
        off = torch.empty(V + 1, dtype=torch.int64, device=self.device)
        dets = torch.empty((max(V * C_ * K, V, 1), 5), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            L = _lib.lib()
            _lib.check(L.fdt_detections_to_frames_count(_lib.ptr(d), V, C_, K, float(thresh), _lib.ptr(n_rows), _lib.ptr(off),
                                                        _lib.stream_ptr()))
            _lib.check(L.fdt_detections_to_frames_pack(_lib.ptr(d), V, C_, K, float(thresh), float(width), float(height), float(shrink),
                                                       _lib.ptr(off), _lib.ptr(dets), _lib.stream_ptr()))
        out = self.step(dets, off, advance)
        out["dets"], out["frame_off"] = dets, off
        return out

    def flush(self, streams=None):
        """End the videos of the selected streams (None = all): their remaining tracks with len >= t_min finish (same records as
        a step); those streams then start a new video at their next step."""
        sel = self._mask(streams)
        out = self._records()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().fdt_track_stream_flush(
                _lib.ptr(self._state), self.V, self.max_d, _lib.ptr(sel), _lib.ptr(out["fin_count"]), _lib.ptr(out["fin_index"]),
                _lib.ptr(out["fin_track"]), _lib.ptr(out["fin_start"]), _lib.ptr(out["fin_len"]), _lib.ptr(out["fin_max"]),
                _lib.stream_ptr()))
        if self.keep_history:
            self._history.append(("flush", None, None, sel, out))
        return out

    def status(self):
        """FDT_STATUS_TRACK_* bits (synchronises)."""
        import ctypes
        bits = ctypes.c_uint32(0)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().fdt_track_stream_status(_lib.ptr(self._state), _lib.stream_ptr(), ctypes.byref(bits)))
        return bits.value

    def check(self):
        """Raise if a frame was skipped for having more than cap rows, or a call did not match the state."""
        bits = self.status()
        if bits & _lib.TRACK_STATUS_OVERFLOW:
            raise RuntimeError(f"StreamTracker: a frame had more than cap={self.cap} rows (max_dets_per_frame={self.max_d}) and was skipped")
        if bits & _lib.TRACK_STATUS_MISMATCH:
            raise RuntimeError("StreamTracker: a call's stream count or max_dets_per_frame did not match the state")

    def tracks_finished(self, v):
        """keep_history=True: stream v's tracks_finished (the reference's list of dicts, iouTracke_cal.py:150-154, 177) for its most
        recent video -- the one in progress if it has had a frame since its last flush, else the last flushed one."""
        if not self.keep_history:
            raise RuntimeError("StreamTracker(keep_history=True) is needed for tracks_finished()")
        videos, cur = [], None                         # per video: (boxes per id, finish records); an advanced step opens one
        for k, h in enumerate(self._history):
            if not isinstance(h, dict):                # host copy, made once per recorded call
                h = self._history[k] = {key: (t.cpu().numpy() if isinstance(t, torch.Tensor) else t) for key, t in
                                        (dict(zip(("kind", "dets", "frame_off", "sel"), h[:-1])) | h[-1]).items()}
            sel = h["sel"]
            if sel is not None and not sel[v]:
                continue
            if h["kind"] == "step":
                a, b = int(h["frame_off"][v]), int(h["frame_off"][v + 1])
                if b - a > self.cap:                   # skipped frame (over capacity)
                    continue
                if cur is None:
                    cur = ({}, []); videos.append(cur)
                for r, i in zip(h["dets"][a:b, :4].tolist(), h["row_track"][a:b].tolist()):
                    cur[0].setdefault(i, []).append(r)
            elif cur is None:                          # nothing since the last flush: nothing to finish
                continue
            for k2 in range(int(h["fin_count"][v])):
                cur[1].append((int(h["fin_index"][v, k2]), int(h["fin_track"][v, k2]), int(h["fin_start"][v, k2]),
                               float(h["fin_max"][v, k2])))
            if h["kind"] == "flush":
                cur = None
        if not videos:
            return []
        boxes, recs = videos[-1]
        recs.sort()
        return [{'bboxes': boxes[i], 'max_score': mx, 'start_frame': st} for _, i, st, mx in recs]


def save_tracks(path, tracks_finished):
    """np.save(video_file + ".npy", np.array(tracks_finished))   [iouTracke_cal.py:177] -- a pickled 1-D object
    array of dicts; `path` gets the .npy suffix from numpy exactly as in the reference."""
    arr = np.empty(len(tracks_finished), dtype=object)
    for i, t in enumerate(tracks_finished):
        arr[i] = t
    np.save(path, arr, allow_pickle=True)


def load_tracks(path):
    """tracks = np.load(video_file + '.npy').tolist()   [iouTracke_display.py:29]; modern numpy needs allow_pickle."""
    return np.load(path, allow_pickle=True).tolist()
