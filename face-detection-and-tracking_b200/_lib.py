"""ctypes binding of csrc/libfdt_b200.so (include/fdt_b200.h).  No CPU fallback: if the library or a
CUDA device is missing the product path raises."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
SO_PATH = os.environ.get("FDT_B200_LIB") or os.path.join(CSRC, "libfdt_b200.so")      # (override: experiments with build variants)

FDT_OK, FDT_E_INVALID, FDT_E_CUDA, FDT_E_WORKSPACE, FDT_E_UNSUPPORTED, FDT_E_DEVICE = 0, -1, -2, -3, -4, -5
MAX_NMS_TOP_K = 8000
NMS_SUMFIRST, NMS_MINIMUM, NMS_PLUS1, NMS_LE = 1, 2, 4, 8

_vp, _i, _i64, _f, _d, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double, C.c_size_t

# symbol -> (restype, argtypes); one entry per declaration in include/fdt_b200.h
SIGNATURES = {
    "fdt_version": (_i, []),
    "fdt_last_error": (C.c_char_p, []),
    "fdt_device_check": (_i, [_i]),
    "fdt_priorbox": (_i, [_d, _d, _d, _d, _i, _vp, _i, _vp, _i, _i, _vp, _vp]),
    "fdt_point_form": (_i, [_vp, _i64, _vp, _vp]),
    "fdt_center_size": (_i, [_vp, _i64, _vp, _vp]),
    "fdt_intersect": (_i, [_vp, _i64, _vp, _i64, _vp, _vp]),
    "fdt_calculate_iou": (_i, [_vp, _i64, _vp, _i64, _vp, _vp]),
    "fdt_calculate_iou_f64": (_i, [_vp, _i64, _vp, _i64, _vp, _vp]),
    "fdt_intersect_f64": (_i, [_vp, _i64, _vp, _i64, _vp, _vp]),
    "fdt_calculate_distance_f64": (_i, [_vp, _i64, _vp, _i64, _vp, _vp]),
    "fdt_calc_pr": (_i, [_vp, _i64, _i, _vp, _i64, _d, _vp, _vp]),
    "fdt_detections_to_rows": (_i, [_vp, _i, _i, _i, _f, _f, _f, _vp, _vp, _vp]),
    "fdt_detections_to_frames_count": (_i, [_vp, _i64, _i, _i, _f, _vp, _vp, _vp]),
    "fdt_detections_to_frames_pack": (_i, [_vp, _i64, _i, _i, _f, _f, _f, _d, _vp, _vp, _vp]),
    "fdt_encode": (_i, [_vp, _vp, _i64, _f, _f, _vp, _vp]),
    "fdt_decode": (_i, [_vp, _vp, _i64, _f, _f, _vp, _vp]),
    "fdt_log_sum_exp": (_i, [_vp, _i64, _i, _vp, _vp, _sz, _vp]),
    "fdt_selftest_cr_math": (_i, [_i, C.c_uint32, C.c_uint64, _vp, _vp]),
    "fdt_nms_workspace_bytes": (_sz, [_i64]),
    "fdt_nms": (_i, [_vp, _vp, _i64, _f, _i64, _vp, _vp, _vp, _sz, _vp]),
    "fdt_nms_variant": (_i, [_vp, _vp, _i64, _f, _i, _vp, _vp, _vp, _sz, _vp]),
    "fdt_nms_f64_workspace_bytes": (_sz, [_i64]),
    "fdt_nms_variant_f64": (_i, [_vp, _vp, _i64, _d, _i, _vp, _vp, _vp, _sz, _vp]),
    "fdt_facebox_decode": (_i, [_vp, _vp, _i64, _f, _f, _vp, _vp]),
    "fdt_threshold_nms_workspace_bytes": (_sz, [_i64]),
    "fdt_threshold_nms": (_i, [_vp, _vp, _i64, _f, _f, _i, _vp, _vp, _vp, _sz, _vp]),
    "fdt_detect_workspace_bytes": (_sz, [_i, _i64, _i]),
    "fdt_detect_workspace_bytes_depth": (_sz, [_i, _i64, _i, _i]),
    "fdt_detect_status": (_i, [_vp, _vp, _vp]),
    "fdt_set_option": (_i, [C.c_char_p, _i]),
    "fdt_detect": (_i, [_vp, _vp, _vp, _i, _i64, _i, _i, _i, _f, _f, _f, _f, _vp, _vp, _vp, _vp, _sz, _vp]),
    "fdt_detect_threshold_compact": (_i, [_vp, _i, _i64, _i, _f, _vp, _sz, _vp]),
    "fdt_detect_sort_nms": (_i, [_vp, _vp, _i, _i64, _i, _i, _i, _f, _f, _f, _vp, _vp, _vp, _vp, _sz, _vp]),
    "fdt_detect_peers": (_i, [_vp, _vp, _vp, _i, _i64, _i, _i, _i, _f, _f, _f, _f, _vp, _i, _i64, _vp, _sz, _vp]),
    "fdt_detect_gather_signal": (_i, [_vp, _vp, _vp, _i, _i64, _i, _i, _i, _f, _f, _f, _f, _vp, _i, _vp, _i, _i, _i, C.c_uint32, _i, _i64,
                                      _vp, _sz, _vp]),
    "fdt_detect_gather_store": (_i, [_vp, _vp, _vp, _i, _i64, _i, _i, _i, _f, _f, _f, _f, _vp, _i, _vp, _i, _i, _i, C.c_uint32, _i, _i64,
                                     _vp, _sz, _vp]),
    "fdt_detect_gather_await": (_i, [_vp, _i, _i, C.c_uint32, _vp, _vp]),
    "fdt_detect_candidate_counts": (_i, [_vp, _sz, _i, _i64, _i, _vp, _vp]),
    "fdt_heads_to_loc_conf": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "fdt_detect_heads": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _f, _f, _f, _f, _vp, _vp, _vp, _vp, _sz, _vp]),
    "fdt_debug_k3_profile": (_i, [_vp]),
    "fdt_ctx_create": (_i, [_i, C.POINTER(_vp)]),
    "fdt_ctx_destroy": (_i, [_vp]),
    "fdt_ctx_set_priors": (_i, [_vp, _vp, _i64]),
    "fdt_detect_host": (_i, [_vp, _vp, _vp, _vp, _i, _i64, _i, _i, _i, _f, _f, _f, _f, _vp, _vp, _vp]),
    "fdt_detect_host_submit": (_i, [_vp, _vp, _vp, _vp, _i, _i64, _i, _i, _i, _f, _f, _f, _f, _vp, _vp, _vp, C.POINTER(C.c_uint64)]),
    "fdt_detect_host_wait": (_i, [_vp, C.c_uint64]),
    "fdt_detect_ex": (_i, [_vp, _i, _vp, _i, _vp, _i, _i64, _i, _i, _i, _f, _f, _f, _f, _vp, _vp, _vp, _vp, _sz, _vp]),
    "fdt_detect_host_ex": (_i, [_vp, _vp, _i, _vp, _i, _vp, _i, _i64, _i, _i, _i, _f, _f, _f, _f, _vp, _vp, _vp]),
    "fdt_detect_host_submit_ex": (_i, [_vp, _vp, _i, _vp, _i, _vp, _i, _i64, _i, _i, _i, _f, _f, _f, _f, _vp, _vp, _vp,
                                       C.POINTER(C.c_uint64)]),
    "fdt_match_workspace_bytes": (_sz, [_i, _i64, _i64]),
    "fdt_match_encode": (_i, [_vp, _vp, _vp, _i64, _i, _i64, _f, _f, _f, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "fdt_mine_workspace_bytes": (_sz, [_i, _i64]),
    "fdt_hard_negative_mine": (_i, [_vp, _vp, _i, _i64, _i, _vp, _vp, _sz, _vp]),
    "fdt_multibox_workspace_bytes": (_sz, [_i, _i64, _i, _i64]),
    "fdt_multibox_loss_forward": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _i, _i64, _i, _f, _i, _i, _f, _f,
                                       _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "fdt_multibox_loss_backward": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _f, _f, _i, _i64, _i, _vp, _vp, _vp]),
    "fdt_multibox_loss_backward_dev": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _i, _vp, _vp, _vp]),
    "fdt_multibox_loss_forward_ex": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _i64, _i, _i64, _i, _f, _i, _i, _f, _f,
                                          _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "fdt_multibox_loss_backward_dev_ex": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _i, _vp, _vp, _vp]),
    "fdt_heads_to_loc_conf_backward": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "fdt_multibox_loss_forward_heads": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _i64, _i, _f, _i, _i, _f, _f,
                                             _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "fdt_multibox_loss_backward_heads_dev": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "fdt_heads_to_loc_conf_ex": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "fdt_detect_heads_ex": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _f, _f, _f, _f, _vp, _vp, _vp, _vp, _sz, _vp]),
    "fdt_heads_to_loc_conf_backward_ex": (_i, [_vp, _i, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "fdt_multibox_loss_forward_heads_ex": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _i64, _i, _f, _i, _i, _f, _f,
                                                _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "fdt_multibox_loss_backward_heads_dev_ex": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "fdt_iou_track_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "fdt_iou_track": (_i, [_vp, _vp, _i64, _i64, _i64, _d, _d, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "fdt_iou_track_metric": (_i, [_vp, _vp, _i64, _i64, _i64, _i, _d, _d, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "fdt_track_stream_state_bytes": (_sz, [_i64, _i64]),
    "fdt_track_stream_workspace_bytes": (_sz, [_i64, _i64]),
    "fdt_track_stream_init": (_i, [_vp, _sz, _i64, _i64, _i, _d, _d, _i64, _vp]),
    "fdt_track_stream_step": (_i, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "fdt_track_stream_flush": (_i, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "fdt_track_stream_status": (_i, [_vp, _vp, _vp]),
}
TRACK_STATUS_OVERFLOW, TRACK_STATUS_MISMATCH = 4, 8

_lib = None
_lock = threading.Lock()


def build(verbose: bool = False) -> str:
    """Compile libfdt_b200.so for sm_100a (csrc/Makefile; nvcc cross-compiles without a GPU)."""
    env = dict(os.environ)
    r = subprocess.run(["make", "-C", CSRC, "-j8", "libfdt_b200.so"], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout)
    if r.returncode != 0:
        raise RuntimeError("building libfdt_b200.so failed")
    return SO_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(SO_PATH):
                    raise RuntimeError(
                        f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(fdt_b200 has no CPU fallback)")
                l = C.CDLL(SO_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(l, name)          # AttributeError here = stale .so; rebuild
                    fn.restype, fn.argtypes = res, args
                _lib = l
    return _lib


def last_error() -> str:
    return lib().fdt_last_error().decode("utf-8", "replace")


def check(rc: int) -> None:
    if rc == FDT_OK:
        return
    msg = last_error()
    if rc == FDT_E_INVALID:
        raise ValueError(msg)
    if rc == FDT_E_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError(f"libfdt_b200 error {rc}: {msg}")


def require_cuda() -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("fdt_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def ptr(t):
    return None if t is None else t.data_ptr()


_workspaces = {}


def workspace(nbytes: int, device: torch.device, tag: str = "") -> torch.Tensor:
    """Grow-only scratch buffer per (device, stream, tag) for the STATELESS entry points (everything but the Detect family);
    torch's caching allocator returns 512-byte aligned blocks, which satisfies the library's 256-byte requirement.
    A buffer is never replaced while its stream is capturing a CUDA graph (the graph would keep the old pointer)."""
    key = (device.index, stream_ptr(), tag)
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        if ws is not None and torch.cuda.is_current_stream_capturing():
            raise RuntimeError(f"fdt_b200: workspace '{tag}' would have to grow ({ws.numel()} -> {nbytes} bytes) during CUDA-graph "
                               "capture; run the largest shape once before capturing")
        ws = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        _workspaces.pop(key, None)
        _workspaces[key] = ws                          # (re-inserted: the dict keeps the most recently allocated entries last)
        if len(_workspaces) > 64 and not torch.cuda.is_current_stream_capturing():
            for k in list(_workspaces)[:-32]:          # streams come and go: drop the oldest entries (freed in stream order)
                del _workspaces[k]
    return ws


DETECT_DEPTH = int(os.environ.get("FDT_DETECT_DEPTH", "4"))          # workspace slots: how many calls may overlap on the device
DETECT_WS_BUDGET = 2 << 30                                             # do not spend more than this on one Detect workspace


class DetectWorkspaces:
    """Workspaces of the Detect family, owned by the object that makes the calls (a Detect instance).  They are STATEFUL -- the
    control block at their head sequences consecutive calls so that they overlap on the device -- hence one buffer per
    (device, stream, B, N, C), kept for the owner's lifetime and never replaced (a captured CUDA graph may hold its pointer)."""

    def __init__(self):
        self._ws = {}

    def get(self, B: int, N: int, C: int, device: torch.device) -> torch.Tensor:
        key = (device.index, stream_ptr(), B, N, C)
        ws = self._ws.get(key)
        if ws is None:
            L = lib()
            slot = L.fdt_detect_workspace_bytes_depth(B, N, C, 2) - L.fdt_detect_workspace_bytes(B, N, C)
            depth = max(1, min(DETECT_DEPTH, DETECT_WS_BUDGET // max(slot, 1)))
            ws = torch.empty(int(L.fdt_detect_workspace_bytes_depth(B, N, C, int(depth))), dtype=torch.uint8, device=device)
            self._ws[key] = ws
            if len(self._ws) > 64:                     # streams / shapes come and go: drop the oldest entries
                for k in list(self._ws)[:-32]:
                    del self._ws[k]
        return ws

    def status(self, device=None) -> int:
        """OR of the FDT_STATUS_* bits of every workspace (synchronises)."""
        bits = 0
        out = C.c_uint32(0)
        for (dev_index, st, *_), ws in self._ws.items():
            with torch.cuda.device(dev_index):
                check(lib().fdt_detect_status(ws.data_ptr(), st, C.byref(out)))
            bits |= out.value
        return bits


def set_option(name: str, value: int) -> None:
    check(lib().fdt_set_option(name.encode(), int(value)))


def dev_f32(t: torch.Tensor, device: torch.device) -> torch.Tensor:
    """fp32, contiguous, on `device`, 16-byte aligned."""
    t = t.detach()
    if t.dtype != torch.float32 or t.device != device or not t.is_contiguous():
        t = t.to(device=device, dtype=torch.float32).contiguous()
    if t.data_ptr() % 16:
        t = t.clone()
    return t


FDT_DTYPE_F32, FDT_DTYPE_BF16, FDT_DTYPE_F16 = 0, 1, 2
_DTYPE16 = {torch.bfloat16: FDT_DTYPE_BF16, torch.float16: FDT_DTYPE_F16}


def flat_input(t: torch.Tensor, device: torch.device):
    """A flat loc / conf tensor as the `_ex` entries take it -> (tensor, FDT_DTYPE_*).  A contiguous bf16 / fp16 tensor on `device` is
    passed in place (any storage offset: the kernels take any element-aligned address); everything else becomes what it always
    became: dev_f32 on a CUDA device, a contiguous fp32 copy on the host."""
    t = t.detach()
    code = _DTYPE16.get(t.dtype)
    if code is not None and t.device == device and t.is_contiguous():
        return t, code
    if device.type == "cpu":
        return t.to(torch.float32).contiguous(), FDT_DTYPE_F32
    return dev_f32(t, device), FDT_DTYPE_F32
