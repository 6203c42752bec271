"""CPU checks of the online multi-stream tracker's C ABI: argument validation answers with error codes before any CUDA call,
and the state / workspace size queries grow with the stream count and the per-frame capacity."""
import ctypes as C

from fdt_b200 import _lib


def test_stream_size_queries_grow():
    L = _lib.lib()
    s1, s64 = L.fdt_track_stream_state_bytes(1, 300), L.fdt_track_stream_state_bytes(64, 300)
    assert 0 < s1 < s64 and L.fdt_track_stream_state_bytes(64, 800) > s64
    assert s1 >= 256 + 320 * (6 * 8 + 4 * 4)                    # header + one slot of cap = 320 rows
    w1, w64 = L.fdt_track_stream_workspace_bytes(1, 300), L.fdt_track_stream_workspace_bytes(64, 300)
    assert 0 < w1 < w64 and L.fdt_track_stream_workspace_bytes(64, 800) > w64 and w64 % 256 == 0
    assert w64 >= 64 * 320 * (10 + 4) * 4                        # one candidate row of W + 4 words per (stream, track)
    assert L.fdt_track_stream_state_bytes(1, 2000) == 0 and L.fdt_track_stream_workspace_bytes(-1, 10) == 0


def test_stream_argument_validation_without_a_gpu():
    L = _lib.lib()
    st = C.c_void_p(256)
    big = 1 << 40
    assert L.fdt_track_stream_init(None, big, 4, 300, 0, 0.4, 0.6, 5, None) == _lib.FDT_E_INVALID
    assert L.fdt_track_stream_init(C.c_void_p(258), big, 4, 300, 0, 0.4, 0.6, 5, None) == _lib.FDT_E_INVALID   # alignment
    assert L.fdt_track_stream_init(st, big, 0, 300, 0, 0.4, 0.6, 5, None) == _lib.FDT_E_INVALID
    assert L.fdt_track_stream_init(st, big, 4, 300, 2, 0.4, 0.6, 5, None) == _lib.FDT_E_INVALID and "metric" in _lib.last_error()
    assert L.fdt_track_stream_init(st, big, 4, 1025, 0, 0.4, 0.6, 5, None) == _lib.FDT_E_UNSUPPORTED
    assert L.fdt_track_stream_init(st, big, 4, 1000, 0, 0.4, 0.6, 5, None) == _lib.FDT_E_UNSUPPORTED   # shared memory
    assert L.fdt_track_stream_init(st, 1024, 4, 300, 0, 0.4, 0.6, 5, None) == _lib.FDT_E_WORKSPACE
    p = [C.c_void_p(256)] * 8
    ws_need = L.fdt_track_stream_workspace_bytes(4, 300)
    assert L.fdt_track_stream_step(st, 4, 300, *p[:3], *p[:7], st, ws_need - 1, None) == _lib.FDT_E_WORKSPACE
    assert L.fdt_track_stream_step(st, 4, 300, None, *p[:2], *p[:7], st, ws_need, None) == _lib.FDT_E_INVALID
    assert L.fdt_track_stream_step(st, 4, 300, *p[:3], *p[:7], C.c_void_p(384), ws_need, None) == _lib.FDT_E_INVALID
    assert L.fdt_track_stream_step(st, -1, 300, *p[:3], *p[:7], st, big, None) == _lib.FDT_E_INVALID
    assert L.fdt_track_stream_flush(st, 4, 300, None, None, *p[:5], None) == _lib.FDT_E_INVALID
    assert L.fdt_track_stream_flush(st, 4, 5000, None, *p[:6], None) == _lib.FDT_E_UNSUPPORTED
    assert L.fdt_track_stream_status(None, None, None) == _lib.FDT_E_INVALID
