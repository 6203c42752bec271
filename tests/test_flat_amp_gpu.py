"""Mixed-precision flat tensors: Detect.__call__ / Detect.submit and MultiBoxLoss.forward read bf16 / fp16 loc[B,N,4] / conf[B,N,C] in
place (each tensor fp32, bf16 or fp16 on its own) and return gradients of the inputs' dtypes.

The target of every GPU comparison is the same call on loc.float(), conf.float() in the same process, which the existing suites pin
to the C oracle: Detect's out / counts / kept_prior and the loss outputs bit-identical (compared as bits, so NaN rows compare too),
gradients bit-identical to what autograd returns through the explicit upcast (the fp32 gradients rounded to nearest even).  The
inputs are rounded to their dtype first, so both sides see the same values.
CPU part: the `_ex` entries' argument checks, the declarations, and which tensors the classifier passes in place."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from fdt_b200 import _lib, synth

BF, HF, F32 = torch.bfloat16, torch.float16, torch.float32
PAIRS = [(BF, BF), (HF, HF), (BF, F32), (F32, HF)]           # (loc dtype, conf dtype)
PATHS = {"auto": (-1, -1), "fused": (1, -1), "two_kernel": (0, -1), "cluster": (0, 1)}      # detect_fused, k3_cluster
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bits(t):
    t = t.detach().contiguous()
    return t.view({4: torch.int32, 2: torch.int16, 8: torch.int64, 1: torch.uint8}[t.element_size()]).cpu()


# ------------------------------------------------------------------------------------------------------------------- CPU
def test_flat_input_classification():
    cpu = torch.device("cpu")
    for dt, code in ((BF, _lib.FDT_DTYPE_BF16), (HF, _lib.FDT_DTYPE_F16)):
        t = torch.zeros((2, 6, 4), dtype=dt)
        u, c = _lib.flat_input(t, cpu)
        assert c == code and u.data_ptr() == t.data_ptr()
        off = torch.zeros(2 * 6 * 4 + 1, dtype=dt)[1:].view(2, 6, 4)          # any storage offset stays in place
        u, c = _lib.flat_input(off, cpu)
        assert c == code and u.data_ptr() == off.data_ptr()
        u, c = _lib.flat_input(t.transpose(0, 1), cpu)                          # non-contiguous: converted, as before
        assert c == _lib.FDT_DTYPE_F32 and u.dtype == F32 and u.is_contiguous()
    for t in (torch.zeros((2, 6, 4), dtype=torch.float64), torch.zeros((2, 6, 4))):
        u, c = _lib.flat_input(t, cpu)
        assert c == _lib.FDT_DTYPE_F32 and u.dtype == F32


def test_flat_ex_entries_declared():
    header = open(os.path.join(ROOT, "include", "fdt_b200.h")).read()
    for name in ("fdt_detect_ex", "fdt_detect_host_ex", "fdt_detect_host_submit_ex", "fdt_multibox_loss_forward_ex",
                 "fdt_multibox_loss_backward_dev_ex"):
        assert re.search(r"\bint %s\(" % name, header), name
        assert name in _lib.SIGNATURES, name


def test_flat_ex_entries_refuse_bad_arguments_without_a_gpu():
    lib = _lib.lib()
    p = 1 << 20
    ticket = C.c_uint64(0)

    def calls(loc, ldt, conf, cdt):
        return [
            ("fdt_detect_ex", lambda: lib.fdt_detect_ex(loc, ldt, conf, cdt, p, 2, 100, 2, 10, 10, 0.05, 0.3, 0.1, 0.2, p, None, None, p,
                                                        1 << 30, None)),
            ("fdt_detect_host_ex", lambda: lib.fdt_detect_host_ex(C.c_void_p(p), loc, ldt, conf, cdt, p, 2, 100, 2, 10, 10, 0.05, 0.3,
                                                                  0.1, 0.2, p, None, None)),
            ("fdt_detect_host_submit_ex", lambda: lib.fdt_detect_host_submit_ex(C.c_void_p(p), loc, ldt, conf, cdt, p, 2, 100, 2, 10, 10,
                                                                                0.05, 0.3, 0.1, 0.2, p, None, None, C.byref(ticket))),
            ("fdt_multibox_loss_forward_ex", lambda: lib.fdt_multibox_loss_forward_ex(
                loc, ldt, conf, cdt, p, p, p, 1, 2, 100, 2, 0.35, 3, 0, 0.1, 0.2, p, p, p, p, p, None, p, 1 << 30, None)),
            ("fdt_multibox_loss_backward_dev_ex", lambda: lib.fdt_multibox_loss_backward_dev_ex(
                loc, ldt, conf, cdt, p, p, p, p, p, p, 2, 100, 2, p, p, None)),
        ]
    for ldt, cdt in ((3, 0), (0, -1), (1, 7)):
        for name, call in calls(p, ldt, p, cdt):
            assert call() == _lib.FDT_E_INVALID, name
            assert "dtype" in _lib.last_error(), (name, _lib.last_error())
    # device entries: an fp32 loc needs 16 bytes (float4 rows); host entries: element alignment only (such a loc_h is copied)
    for loc, ldt, conf, cdt in ((p + 1, 1, p, 1), (p, 2, p + 3, 2), (p + 8, 0, p, 1), (p + 2, 0, p, 1), (p, 1, p + 2, 0)):
        for name, call in calls(loc, ldt, conf, cdt):
            if "host" in name and loc == p + 8:
                continue                                # accepted: it would go on to use the (fake) context
            assert call() == _lib.FDT_E_INVALID, name
            assert "aligned" in _lib.last_error(), (name, _lib.last_error())
    # a null loc is refused before anything is enqueued, whatever the dtypes (16-bit loc would be read through a map at address 0)
    for ldt, cdt in ((1, 1), (0, 2), (2, 0), (0, 0)):
        assert lib.fdt_detect_ex(None, ldt, p, cdt, p, 2, 100, 2, 10, 10, 0.05, 0.3, 0.1, 0.2, p, None, None, p, 1 << 30,
                                 None) == _lib.FDT_E_INVALID, (ldt, cdt)
        assert "null" in _lib.last_error(), _lib.last_error()
    # 2-byte aligned 16-bit data passes the checks (refused later for the short workspace, before any CUDA call)
    assert lib.fdt_multibox_loss_forward_ex(p + 2, 1, p + 2, 2, p, p, p, 1, 2, 100, 2, 0.35, 3, 0, 0.1, 0.2, p, p, p, p, p, None, p, 16,
                                            None) == _lib.FDT_E_WORKSPACE


# ------------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture()
def opts():
    yield _lib
    _lib.set_option("detect_fused", int(os.environ.get("FDT_DETECT_FUSED") or -1))
    _lib.set_option("k3_cluster", int(os.environ.get("FDT_K3_CLUSTER") or -1))
    _lib.set_option("host_chunk", 16)


def inputs(B, w, h, seed, mode="random"):
    pri = synth.priors_numpy(w, h)
    loc, conf = synth.detect_inputs(B, pri, seed, 0.05, mode)
    return torch.from_numpy(loc), torch.from_numpy(conf), torch.from_numpy(pri)


def as_dtypes(loc, conf, ldt, cdt, device="cuda"):
    return loc.to(ldt).to(device), conf.to(cdt).to(device)


def detect_pair(loc, conf, pri, thresh=0.05, top_k=750, C_=2):
    """(in place, upcast) Detect results with aux outputs"""
    from fdt_b200.layers import Detect
    pri = pri.to(loc.device) if loc.is_cuda else pri
    a = Detect(C_, 0, top_k, thresh, 0.3)(loc, conf, pri, return_aux=True)
    b = Detect(C_, 0, top_k, thresh, 0.3)(loc.float(), conf.float(), pri, return_aux=True)
    return a, b


def assert_same(a, b, what):
    for x, y, name in zip(a, b, ("out", "counts", "kept_prior")):
        assert torch.equal(bits(x), bits(y)), (what, name)


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("ldt,cdt", PAIRS, ids=lambda d: str(d).split(".")[-1])
def test_gpu_detect_b64_640(opts, ldt, cdt, path):
    fused, cluster = PATHS[path]
    opts.set_option("detect_fused", fused)
    opts.set_option("k3_cluster", cluster)
    loc, conf, pri = inputs(64, 640, 640, 11)
    l, c = as_dtypes(loc, conf, ldt, cdt)
    a, b = detect_pair(l, c, pri.cuda())
    assert int(a[1].sum()) > 1000
    assert_same(a, b, (ldt, cdt, path))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["b1", "lists149", "n87360", "c3"])
@pytest.mark.parametrize("ldt,cdt", PAIRS, ids=lambda d: str(d).split(".")[-1])
def test_gpu_detect_shapes(opts, ldt, cdt, shape):
    if shape == "b1":
        loc, conf, pri = inputs(1, 640, 640, 21)
    elif shape == "lists149":                           # more lists than SMs: K2 + k_sort_nms on the automatic path
        loc, conf, pri = inputs(149, 320, 320, 22)
    elif shape == "n87360":                             # rows longer than the fused kernel's first scan, visited in place
        loc, conf, pri = inputs(4, 1024, 1024, 23)
        assert pri.shape[0] == 87360
        opts.set_option("detect_fused", 1)
    else:
        pri = torch.from_numpy(synth.priors_numpy(320, 320))
        g = torch.Generator().manual_seed(24)
        loc = torch.randn((6, pri.shape[0], 4), generator=g) * 0.5
        conf = torch.softmax(torch.randn((6, pri.shape[0], 3), generator=g) * 2.0, -1)
    l, c = as_dtypes(loc, conf, ldt, cdt)
    C_ = conf.shape[-1]
    for fused in ((-1, 0, 1) if shape == "c3" else (-1,)):
        if shape == "c3":
            opts.set_option("detect_fused", fused)
        a, b = detect_pair(l, c, pri.cuda(), C_=C_)
        assert_same(a, b, (shape, fused))


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["fused", "two_kernel"])
@pytest.mark.parametrize("dt", [BF, HF], ids=["bf16", "fp16"])
def test_gpu_detect_equal_score_buckets(opts, dt, path):
    """thousands of equal 16-bit scores per image: the radix-select and bitonic fallbacks of k_sort_nms"""
    fused, cluster = PATHS[path]
    opts.set_option("detect_fused", fused)
    loc, conf, pri = inputs(8, 640, 640, 31)
    g = torch.Generator().manual_seed(32)
    levels = torch.tensor([0.25, 0.5, 0.75, 0.875])
    pick = torch.randint(0, 4, conf.shape[:2], generator=g)
    tie = torch.rand(conf.shape[:2], generator=g) < 0.3
    s = torch.where(tie, levels[pick], conf[..., 1])
    conf = torch.stack([1 - s, s], -1)
    l, c = as_dtypes(loc, conf, dt, dt)
    for top_k in (750, 5000):
        a, b = detect_pair(l, c, pri.cuda(), top_k=top_k)
        assert_same(a, b, (dt, path, top_k))


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["fused", "two_kernel"])
@pytest.mark.parametrize("thresh", [0.05, 0.0, -0.5])
@pytest.mark.parametrize("ldt,cdt", PAIRS, ids=lambda d: str(d).split(".")[-1])
def test_gpu_detect_special_scores(opts, ldt, cdt, thresh, path):
    opts.set_option("detect_fused", PATHS[path][0])
    loc, conf, pri = inputs(4, 640, 640, 41)
    g = torch.Generator().manual_seed(42)
    special = torch.tensor([float("nan"), float("inf"), -float("inf"), -0.0, 0.0, 1.5, -2.0])
    where = torch.rand(conf.shape[:2], generator=g) < 0.02
    conf[..., 1] = torch.where(where, special[torch.randint(0, len(special), conf.shape[:2], generator=g)], conf[..., 1])
    loc[0, :50] = float("nan")
    l, c = as_dtypes(loc, conf, ldt, cdt)
    a, b = detect_pair(l, c, pri.cuda(), thresh=thresh)
    assert_same(a, b, (ldt, cdt, thresh, path))


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["fused", "two_kernel"])
def test_gpu_detect_odd_storage_offsets(opts, path):
    """loc 2-byte but not 8-byte aligned, conf 2-byte but not 4-byte aligned: the scalar loads"""
    opts.set_option("detect_fused", PATHS[path][0])
    loc, conf, pri = inputs(16, 640, 640, 51)
    for dt in (BF, HF):
        lb = torch.zeros(loc.numel() + 1, dtype=dt, device="cuda")
        cb = torch.zeros(conf.numel() + 1, dtype=dt, device="cuda")
        l = lb[1:].view(loc.shape); c = cb[1:].view(conf.shape)
        l.copy_(loc.to(dt)); c.copy_(conf.to(dt))
        assert l.data_ptr() % 8 == 2 and c.data_ptr() % 4 == 2
        a, b = detect_pair(l, c, pri.cuda())
        assert_same(a, b, (dt, path))


@pytest.mark.gpu
def test_gpu_detect_back_to_back_alternating_dtypes():
    """eight calls on one stream and one Detect (its workspace ring lets them overlap), dtypes alternating, then one synchronize"""
    from fdt_b200.layers import Detect
    pri = torch.from_numpy(synth.priors_numpy(640, 640)).cuda()
    sets = []
    for i, (ldt, cdt) in enumerate([(F32, F32)] + PAIRS + [(F32, F32), (HF, BF), (BF, HF)]):
        loc, conf, _ = inputs(64, 640, 640, 600 + i)
        sets.append(as_dtypes(loc, conf, ldt, cdt))
    iso = []
    for l, c in sets:
        iso.append(Detect(2, 0, 750, 0.05, 0.3)(l.float(), c.float(), pri, return_aux=True))
    torch.cuda.synchronize()
    det = Detect(2, 0, 750, 0.05, 0.3)
    outs = [det(l, c, pri, return_aux=True) for l, c in sets]
    torch.cuda.synchronize()
    for a, b in zip(outs, iso):
        assert_same(a, b, "back to back")


@pytest.mark.gpu
def test_gpu_detect_bf16_cuda_graph():
    from fdt_b200.layers import Detect
    loc, conf, pri = inputs(64, 640, 640, 71)
    loc2, conf2, _ = inputs(64, 640, 640, 72)
    l, c = as_dtypes(loc, conf, BF, BF)
    p = pri.cuda()
    det = Detect(2, 0, 750, 0.05, 0.3)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        det(l, c, p)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            out = det(l, c, p, return_aux=True)
    torch.cuda.current_stream().wait_stream(side)
    l2, c2 = as_dtypes(loc2, conf2, BF, BF)
    l.copy_(l2); c.copy_(c2)
    torch.cuda.synchronize()
    g.replay()
    torch.cuda.synchronize()
    ref = Detect(2, 0, 750, 0.05, 0.3)(l2.float(), c2.float(), p, return_aux=True)
    assert_same(out, ref, "graph replay")


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [True, False])
@pytest.mark.parametrize("ldt,cdt", [(HF, HF), (BF, BF), (BF, F32), (F32, HF)], ids=lambda d: str(d).split(".")[-1])
def test_gpu_detect_host_tensors(opts, ldt, cdt, pinned):
    from fdt_b200.layers import Detect
    opts.set_option("host_chunk", 5)                    # chunks with a remainder
    loc, conf, pri = inputs(23, 640, 640, 81)
    l, c = as_dtypes(loc, conf, ldt, cdt, device="cpu")
    if pinned:
        l, c = l.pin_memory(), c.pin_memory()
    ref = Detect(2, 0, 750, 0.05, 0.3)(l.cuda().float(), c.cuda().float(), pri.cuda(), return_aux=True)
    det = Detect(2, 0, 750, 0.05, 0.3)
    pend = [det.submit(l, c, pri, return_aux=True) for _ in range(2)]
    for pd in pend:
        assert_same(pd.result(), ref, ("submit", pinned))
    assert_same(det(l, c, pri, return_aux=True), ref, ("call", pinned))


def loss_inputs(B, seed, ldt, cdt, C_=2):
    pri = synth.priors_numpy(640, 640)
    loc, conf, targets = synth.multibox_inputs(B, pri, seed, 1, 60)
    loc = torch.from_numpy(loc).to(ldt).cuda()
    conf = torch.from_numpy(conf).to(cdt).cuda()
    if C_ != 2:
        conf = torch.randn((B, pri.shape[0], C_), generator=torch.Generator().manual_seed(seed)).to(cdt).cuda()
    return loc, conf, torch.from_numpy(pri).cuda(), [torch.from_numpy(t).cuda() for t in targets]


@pytest.mark.gpu
@pytest.mark.parametrize("C_", [2, 3])
@pytest.mark.parametrize("bipartite", [False, True])
@pytest.mark.parametrize("ldt,cdt", PAIRS, ids=lambda d: str(d).split(".")[-1])
def test_gpu_multibox_equals_upcast(ldt, cdt, bipartite, C_):
    from fdt_b200.layers import MultiBoxLoss
    loc, conf, pri, tg = loss_inputs(8, 91, ldt, cdt, C_)
    if C_ == 3:
        tg = [torch.cat([t[:, :4], (torch.arange(len(t), device="cuda") % 2).float()[:, None]], 1) for t in tg]
    crit = MultiBoxLoss(C_, 0.35, True, 0, True, 3, 0.35, False, bipartite=bipartite)
    res = []
    for upcast in (False, True):
        l = loc.detach().clone().requires_grad_(True)
        c = conf.detach().clone().requires_grad_(True)
        ll, lc = crit((l.float(), c.float(), pri) if upcast else (l, c, pri), tg)
        aux = [t.clone() for t in crit.last_aux]
        (ll * 0.75 + lc * 1.25).backward()
        res.append((ll.detach(), lc.detach(), aux, l.grad, c.grad))
    a, b = res
    assert torch.equal(bits(a[0]), bits(b[0])) and torch.equal(bits(a[1]), bits(b[1]))
    for x, y in zip(a[2], b[2]):
        assert torch.equal(bits(x), bits(y))
    for g, x, ref in ((a[3], loc, b[3]), (a[4], conf, b[4])):
        assert g.dtype == x.dtype and g.shape == x.shape and torch.equal(bits(g), bits(ref))


@pytest.mark.gpu
def test_gpu_autocast_training_step():
    """a conv head under bf16 autocast -> flat loc / conf -> MultiBoxLoss -> backward: in place equals the explicit upcast"""
    from fdt_b200.layers import MultiBoxLoss
    torch.manual_seed(0)
    fm = synth.feature_maps(320, 320)
    B, Cin = 4, 16
    feats = [torch.randn((B, Cin, fh, fw), device="cuda") for fw, fh in fm]
    convs = [(torch.nn.Conv2d(Cin, 4, 3, padding=1).cuda(), torch.nn.Conv2d(Cin, 2, 3, padding=1).cuda()) for _ in fm]
    pri = torch.from_numpy(synth.priors_numpy(320, 320)).cuda()
    _, _, targets = synth.multibox_inputs(B, pri.cpu().numpy(), 9, 1, 40)
    tg = [torch.from_numpy(t).cuda() for t in targets]
    crit = MultiBoxLoss(2, 0.35, True, 0, True, 3, 0.35, False)

    def run(explicit_upcast):
        for cl, cc in convs:
            cl.zero_grad(); cc.zero_grad()
        with torch.autocast(device_type="cuda", dtype=torch.bfloat16):
            loc = torch.cat([cl(x).permute(0, 2, 3, 1).contiguous().view(B, -1, 4) for x, (cl, _) in zip(feats, convs)], 1)
            conf = torch.cat([cc(x).permute(0, 2, 3, 1).contiguous().view(B, -1, 2) for x, (_, cc) in zip(feats, convs)], 1)
        assert loc.dtype == BF and conf.dtype == BF
        if explicit_upcast:
            loc, conf = loc.float(), conf.float()
        ll, lc = crit((loc, conf, pri), tg)
        (ll + lc).backward()
        return ll.detach(), lc.detach(), [p.grad.clone() for cl, cc in convs for p in (*cl.parameters(), *cc.parameters())]

    with torch.backends.cudnn.flags(enabled=True, deterministic=True, benchmark=False):
        a, b = run(False), run(True)
    assert float(a[0]) == float(b[0]) and float(a[1]) == float(b[1])
    for x, y in zip(a[2], b[2]):
        assert torch.equal(bits(x), bits(y))


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [True, False])
def test_gpu_detect_host_fp32_loc_at_a_float_offset(opts, pinned):
    """an fp32 host loc one float past a 16-byte boundary (fp32 and fp16 conf): accepted as before -- copied, not gathered in place"""
    from fdt_b200.layers import Detect
    loc, conf, pri = inputs(9, 640, 640, 91)
    buf = torch.zeros(loc.numel() + 1)
    if pinned:
        buf = buf.pin_memory()
    l = buf[1:].view(loc.shape)
    l.copy_(loc)
    assert l.data_ptr() % 16 == 4 and l.is_contiguous()
    for cdt in (F32, HF):
        c = conf.to(cdt)
        ref = Detect(2, 0, 750, 0.05, 0.3)(loc.cuda(), c.cuda(), pri.cuda(), return_aux=True)
        det = Detect(2, 0, 750, 0.05, 0.3)
        assert_same(det.submit(l, c, pri, return_aux=True).result(), ref, ("submit", cdt))
        assert_same(det(l, c, pri, return_aux=True), ref, ("call", cdt))
