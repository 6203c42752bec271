"""Mixed-precision / channels_last head maps: Detect.detect_heads, heads_to_loc_conf and MultiBoxLoss.forward_heads read bf16 / fp16,
NCHW or channels_last maps in place and write map gradients of the maps' dtype and memory format.

The target of every GPU comparison is the same call on the maps upcast to fp32 NCHW ([m.float().contiguous() ...]), which the
existing suites pin to the C oracle and the reference fixtures: outputs bit-identical, map gradients bit-identical to autograd's
gradients through the upcast.  The maps are rounded to their dtype on the CPU from synth.head_maps, so both sides see the same bits.
CPU part: argument checks of the `_ex` entries, and the classification of maps into those read in place and those converted."""
import ctypes as C

import numpy as np
import pytest
import torch

from fdt_b200 import _lib, synth
from fdt_b200.layers.functions import heads as H
from oracle import oracle as orc

DTYPES = [torch.float32, torch.bfloat16, torch.float16]
LAYOUTS = ["nchw", "channels_last"]
SHAPES = {"six_640": (640, 640, synth.STRIDES6, synth.BOXES6), "five_640": (640, 640, synth.STRIDES6[:5], synth.BOXES6[:5]),
          "six_640x480": (640, 480, synth.STRIDES6, synth.BOXES6)}
VAR = (0.1, 0.2)


def rounded_maps(B, shape, seed, dtype):
    """synth.head_maps rounded to `dtype` on the CPU -> (loc maps, conf maps, neg_max, priors) as CPU tensors / numpy priors"""
    w, h, strides, boxes = SHAPES[shape]
    lm, cm, nm = synth.head_maps(B, w, h, seed, strides)
    return ([torch.from_numpy(m).to(dtype) for m in lm], [torch.from_numpy(m).to(dtype) for m in cm], nm,
            synth.priors_numpy(w, h, strides, boxes))


def place(maps, layout):
    out = [m.cuda() for m in maps]
    return [m.contiguous(memory_format=torch.channels_last) for m in out] if layout == "channels_last" else out


def upcast(maps):
    return [m.float().contiguous() for m in maps]


def bits(t):
    """the raw bits of a tensor in logical (NCHW) order: equality that also holds for NaN"""
    t = t.detach().contiguous()
    return t.view({4: torch.int32, 2: torch.int16, 8: torch.int64, 1: torch.uint8}[t.element_size()]).cpu()


def detect_aux(det, lm, cm, pri, nm):
    return det.detect_heads(lm, cm, pri, nm, return_aux=True)


def assert_same_detect(a, b, what):
    for x, y, name in zip(a, b, ("out", "counts", "kept_prior")):
        assert torch.equal(x, y), (what, name)


# ------------------------------------------------------------------------------------------------------------------- CPU
def test_classification_without_the_library():
    bf = torch.bfloat16
    nchw = torch.empty((2, 4, 5, 6), dtype=bf, device="meta")
    cl = torch.empty((2, 4, 5, 6), dtype=bf, device="meta").contiguous(memory_format=torch.channels_last)
    assert H.map_layout(nchw) == "nchw" and H.map_layout(cl) == "channels_last"
    assert H.native_dtype([nchw], [cl]) == 1
    assert H.native_dtype([nchw.half()], [cl.half()]) == 2
    assert H.native_dtype([nchw.float()], [cl.float()]) == 0
    assert H.native_dtype([nchw.half()], [cl]) is None                        # dtypes differ within one call
    assert H.native_dtype([nchw.double()], [nchw.double()]) is None           # float64: converted
    odd = torch.empty((2, 4, 6, 5), dtype=bf, device="meta").transpose(2, 3)  # neither dense NCHW nor dense channels_last
    assert H.map_layout(odd) is None and H.native_dtype([nchw], [odd]) is None
    sliced = torch.empty((2, 8, 5, 6), dtype=bf, device="meta")[:, :4]        # channel slice of a wider conv output
    assert H.map_layout(sliced) is None
    assert H.native_dtype(None, [cl]) == 1                                    # conf maps only
    # size-1 levels: torch reports arbitrary strides for size-1 dimensions; the descriptor uses the ones the layout implies
    for shape in ((2, 4, 1, 1), (2, 4, 1, 7), (1, 4, 3, 1)):
        for t in (torch.empty(shape, dtype=bf), torch.empty(shape, dtype=bf).contiguous(memory_format=torch.channels_last),
                  torch.empty(shape[:1] + shape[2:] + (4,), dtype=bf).permute(0, 3, 1, 2)):
            assert H.map_layout(t) is not None, (shape, t.stride())
            d = H.map_descs([t])[0]
            hw = shape[2] * shape[3]
            assert d.data == t.data_ptr() and d.batch_stride == 4 * hw
            assert (d.channel_stride, d.pixel_stride) in ((hw, 1), (1, 4))
    # any storage offset
    base = torch.empty(2 * 4 * 5 * 6 + 1, dtype=bf)
    view = base.as_strided((2, 4, 5, 6), (120, 1, 24, 4), 1)
    assert H.map_layout(view) == "channels_last"
    d = H.map_descs([view])[0]
    assert (d.data, d.batch_stride, d.channel_stride, d.pixel_stride) == (view.data_ptr(), 120, 1, 4)
    # CPU maps of another device than the conf maps: converted (the device check)
    assert H.native_dtype([nchw], [torch.empty((2, 4, 5, 6), dtype=bf)]) is None


def descs(L, data=256, strides=(64, 16, 1)):
    d = (H.HeadMap * 8)()
    for l in range(8):
        d[l] = H.HeadMap(data, *strides)
    return d


def test_ex_entries_refuse_bad_arguments_without_a_gpu():
    lib = _lib.lib()
    fh = (C.c_int * 8)(*([4] * 8)); fw = (C.c_int * 8)(*([4] * 8)); nm = (C.c_int * 8)(*([0] * 8))
    p = C.c_void_p(256)
    good = descs(2)

    def calls(ld, cd, dt):
        return [
            ("fdt_heads_to_loc_conf_ex", lambda: lib.fdt_heads_to_loc_conf_ex(ld, cd, dt, fh, fw, nm, 2, 1, 0, p, p, None)),
            ("fdt_detect_heads_ex", lambda: lib.fdt_detect_heads_ex(ld, cd, dt, fh, fw, nm, 2, p, 1, 10, 10, 0.05, 0.3, 0.1, 0.2,
                                                                    p, None, None, p, 1 << 30, None)),
            ("fdt_heads_to_loc_conf_backward_ex", lambda: lib.fdt_heads_to_loc_conf_backward_ex(cd, dt, fh, fw, nm, 2, 1, 0, p, p, ld, cd,
                                                                                                None)),
            ("fdt_multibox_loss_forward_heads_ex", lambda: lib.fdt_multibox_loss_forward_heads_ex(
                ld, cd, dt, fh, fw, nm, 2, p, p, p, 1, 1, 0.35, 3, 0, 0.1, 0.2, p, p, p, p, p, None, p, 1 << 30, None)),
            ("fdt_multibox_loss_backward_heads_dev_ex", lambda: lib.fdt_multibox_loss_backward_heads_dev_ex(
                ld, cd, dt, fh, fw, nm, 2, p, p, p, p, p, p, 1, ld, cd, None)),
        ]
    for dt, word in ((3, "dtype"), (-1, "dtype")):
        for name, call in calls(good, good, dt):
            assert call() == _lib.FDT_E_INVALID, name
            assert word in _lib.last_error(), (name, _lib.last_error())
    bad_null = descs(2); bad_null[1].data = None
    for name, call in calls(bad_null, bad_null, 1):
        assert call() == _lib.FDT_E_INVALID, name
        assert "null" in _lib.last_error() and "1" in _lib.last_error(), (name, _lib.last_error())
    for strides in ((0, 16, 1), (64, -1, 1), (64, 16, 0)):
        bad = descs(2, strides=strides)
        for name, call in calls(bad, bad, 1):
            assert call() == _lib.FDT_E_INVALID, name
            assert "stride" in _lib.last_error(), (name, _lib.last_error())
    for dt, data in ((1, 257), (2, 259), (0, 258)):                    # not aligned to the element size
        bad = descs(2, data=data)
        for name, call in calls(bad, bad, dt):
            assert call() == _lib.FDT_E_INVALID, name
            assert "aligned" in _lib.last_error(), (name, _lib.last_error())
    # a 2-byte aligned bf16 map is accepted by the checks (refused later for the short workspace, before any CUDA call)
    ok = descs(2, data=258, strides=(64, 1, 4))
    assert lib.fdt_multibox_loss_forward_heads_ex(ok, ok, 1, fh, fw, nm, 2, p, p, p, 1, 1, 0.35, 3, 0, 0.1, 0.2, p, p, p, p, p, None,
                                                  p, 16, None) == _lib.FDT_E_WORKSPACE


# ------------------------------------------------------------------------------------------------------------------- GPU
def plant_specials(cm, dtype):
    """NaN / +-inf in the conf maps of a 16-bit dtype, and fp16 values near 65504"""
    if dtype == torch.float32:
        return
    cm[0][0, 3, 2, 3] = float("nan")
    cm[0][0, 1, 4, 4] = float("inf")
    cm[1][0, 0, 1, 1] = float("-inf")
    cm[1][0, 2, 3, 2] = float("nan")
    cm[-1][0, 0, 0, 0] = float("inf")
    if dtype == torch.float16:
        cm[1][0, 1, 2, 2] = 65504.0
        cm[1][0, 2, 2, 2] = 65504.0
        cm[2][0, 0, 1, 2] = -65504.0
        cm[2][0, 3, 1, 2] = 65000.0


@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("dtype", DTYPES)
def test_gpu_detect_heads_equals_upcast(dtype, layout, shape):
    from fdt_b200.layers import Detect
    for B in (1, 64):
        lm, cm, nm, pri = rounded_maps(B, shape, 400 + B, dtype)
        plant_specials(cm, dtype)
        p = torch.from_numpy(pri).cuda()
        lmg, cmg = place(lm, layout), place(cm, layout)
        lmu, cmu = upcast(lmg), upcast(cmg)
        L = len(cm)
        for neg_max in (None, nm, [l % 2 for l in range(L)]):
            det_a, det_b = Detect(2, 0, 750, 0.05, 0.3), Detect(2, 0, 750, 0.05, 0.3)
            a = detect_aux(det_a, lmg, cmg, p, neg_max)
            b = detect_aux(det_b, lmu, cmu, p, neg_max)
            assert_same_detect(a, b, (dtype, layout, shape, B, neg_max))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_gpu_detect_heads_equal_score_buckets(dtype):
    """bf16 / fp16 logits are coarse, so equal scores are common: a bucket of > 512 equal scores (bitonic fallback) and one of
    thousands (radix select) still give the upcast path's result"""
    from fdt_b200.layers import Detect
    for n_tied in (600, 4000):
        lm, cm, nm, pri = rounded_maps(2, "six_640", 77, dtype)
        flat = cm[0][0].reshape(4, -1)                         # level 0 (neg_max): neg = max(ch0..2), pos = ch3
        flat[:3, :n_tied] = 0.0
        flat[3, :n_tied] = 1.0
        cm[1][1, 0].fill_(-1.0)                                # image 1, level 1: every prior scores the same
        cm[1][1, 1:].fill_(0.5)
        p = torch.from_numpy(pri).cuda()
        for layout in LAYOUTS:
            lmg, cmg = place(lm, layout), place(cm, layout)
            a = detect_aux(Detect(2, 0, 750, 0.05, 0.3), lmg, cmg, p, nm)
            b = detect_aux(Detect(2, 0, 750, 0.05, 0.3), upcast(lmg), upcast(cmg), p, nm)
            assert_same_detect(a, b, (dtype, n_tied, layout))
            assert int(a[1][0, 1]) > 0


@pytest.mark.gpu
def test_gpu_detect_heads_oracle_on_upcast_maps():
    from fdt_b200.layers import Detect
    lm, cm, nm, pri = rounded_maps(2, "six_640x480", 5, torch.bfloat16)
    out = Detect(2, 0, 750, 0.05, 0.3).detect_heads(place(lm, "channels_last"), place(cm, "channels_last"), torch.from_numpy(pri).cuda(), nm)
    lf, cf = [m.float().numpy() for m in lm], [m.float().numpy() for m in cm]
    loc, conf = orc.heads_to_loc_conf(lf, cf, nm, softmax=True)
    ref = orc.Detect(2, 0, 750, 0.05, 0.3)(loc, conf, pri)
    assert np.array_equal(out.cpu().numpy(), ref)


def grads_via(fn, maps_cpu, layout, upcast_first, need):
    """map gradients of fn(loc maps, conf maps) -> scalar, taken on leaves of the given dtype and layout"""
    lm, cm = (place(m, layout) for m in maps_cpu)
    lm = [m.requires_grad_(need[0]) for m in lm]
    cm = [m.requires_grad_(need[1]) for m in cm]
    a, b = (upcast(lm), upcast(cm)) if upcast_first else (lm, cm)
    out = fn(a, b)
    leaves = [m for m, n in zip(lm + cm, [need[0]] * len(lm) + [need[1]] * len(cm)) if n]
    return out, torch.autograd.grad(out[0], leaves)


def check_grads(ga, gb, dtype, layout, what):
    for x, y in zip(ga, gb):
        assert x.dtype == dtype and y.dtype == dtype, what
        assert torch.equal(bits(x), bits(y)), what
        if layout == "channels_last" and x.size(2) * x.size(3) > 1:
            assert x.is_contiguous(memory_format=torch.channels_last), what


@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("dtype", DTYPES)
def test_gpu_heads_to_loc_conf_equals_upcast(dtype, layout, shape):
    from fdt_b200.layers import heads_to_loc_conf
    lm, cm, nm, _ = rounded_maps(2, shape, 11, dtype)
    B, N = 2, sum(m.size(2) * m.size(3) for m in lm)
    gen = torch.Generator().manual_seed(5)
    g_loc, g_conf = torch.randn((B, N, 4), generator=gen).cuda(), torch.randn((B, N, 2), generator=gen).cuda()
    for softmax in (True, False):
        a = heads_to_loc_conf(place(lm, layout), place(cm, layout), nm, softmax=softmax)
        b = heads_to_loc_conf(upcast(place(lm, layout)), upcast(place(cm, layout)), nm, softmax=softmax)
        assert a[0].dtype == torch.float32 and torch.equal(bits(a[0]), bits(b[0]))
        assert torch.equal(bits(a[1]), bits(b[1]))

        def fn(l_, c_):
            loc, conf = heads_to_loc_conf(l_, c_, nm, softmax=softmax)
            return ((loc * g_loc).sum() + (conf * g_conf).sum(),)
        for need in ((True, True), (True, False), (False, True)):
            _, ga = grads_via(fn, (lm, cm), layout, False, need)
            _, gb = grads_via(fn, (lm, cm), layout, True, need)
            check_grads(ga, gb, dtype, layout, (softmax, need))


def loss_setup(shape, dtype, seed):
    lm, cm, nm, pri = rounded_maps(8, shape, seed, dtype)
    _, _, targets = synth.multibox_inputs(8, pri, seed + 1, 0, 200)
    targets[3] = np.zeros((0, 5), np.float32)                 # an image without ground truth
    return lm, cm, nm, torch.from_numpy(pri).cuda(), [torch.from_numpy(t).cuda() for t in targets]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("dtype", DTYPES)
def test_gpu_forward_heads_equals_upcast(dtype, layout, shape):
    from fdt_b200.layers import MultiBoxLoss
    lm, cm, nm, p, tg = loss_setup(shape, dtype, 31)
    for bip in (False, True):
        crit = MultiBoxLoss(2, 0.35, True, 0, True, 3, 0.35, False, bipartite=bip)

        def fn(l_, c_):
            ll, lc = crit.forward_heads(l_, c_, p, tg, nm)
            return (ll + 0.5 * lc, ll, lc, *[t.clone() for t in crit.last_aux])
        for need in ((True, True), (True, False), (False, True)):
            oa, ga = grads_via(fn, (lm, cm), layout, False, need)
            ob, gb = grads_via(fn, (lm, cm), layout, True, need)
            for x, y in zip(oa, ob):
                assert torch.equal(bits(x), bits(y)), (bip, need)
            check_grads(ga, gb, dtype, layout, (bip, need))


@pytest.mark.gpu
def test_gpu_forward_heads_oracle_on_upcast_maps():
    from fdt_b200.layers import MultiBoxLoss
    lm, cm, nm, p, tg = loss_setup("five_640", torch.bfloat16, 61)
    crit = MultiBoxLoss(2, 0.35, True, 0, True, 3, 0.35, False, bipartite=False)
    ll, lc = crit.forward_heads(place(lm, "channels_last"), place(cm, "channels_last"), p, tg, nm)
    _, conf_t, _ = crit.last_aux
    lf, cf = [m.float().numpy() for m in lm], [m.float().numpy() for m in cm]
    raw = orc.heads_to_loc_conf(lf, cf, nm, softmax=False)
    r = orc.multibox_loss(raw[0], raw[1], p.cpu().numpy(), [t.cpu().numpy() for t in tg], 0.35, 3, False, VAR)
    assert np.array_equal(conf_t.cpu().numpy(), r["conf_t"])
    np.testing.assert_allclose([float(ll), float(lc)], [r["loss_l"], r["loss_c"]], rtol=1e-5, atol=1e-7)


@pytest.mark.gpu
def test_gpu_autocast_end_to_end():
    """a small conv head per level under bf16 autocast -> forward_heads -> backward: the losses and the map gradients equal those of
    the same network whose bf16 maps are upcast explicitly"""
    from fdt_b200.layers import MultiBoxLoss
    torch.manual_seed(0)
    w, h, strides, boxes = SHAPES["six_640x480"]
    fm = synth.feature_maps(w, h, strides)
    B, Cin = 4, 16
    feats = [torch.randn((B, Cin, fh, fw), device="cuda") for fw, fh in fm]
    convs = [(torch.nn.Conv2d(Cin, 4, 3, padding=1).cuda(), torch.nn.Conv2d(Cin, 4, 3, padding=1).cuda()) for _ in fm]
    pri = torch.from_numpy(synth.priors_numpy(w, h, strides, boxes)).cuda()
    _, _, targets = synth.multibox_inputs(B, pri.cpu().numpy(), 9, 1, 40)
    tg = [torch.from_numpy(t).cuda() for t in targets]
    crit = MultiBoxLoss(2, 0.35, True, 0, True, 3, 0.35, False)

    def run(explicit_upcast, channels_last):
        lm, cm = [], []
        with torch.autocast(device_type="cuda", dtype=torch.bfloat16):
            for x, (cl, cc) in zip(feats, convs):
                if channels_last:
                    x = x.contiguous(memory_format=torch.channels_last)
                lm.append(cl(x)); cm.append(cc(x))
        for m in lm + cm:
            m.retain_grad()
        a, b = (upcast(lm), upcast(cm)) if explicit_upcast else (lm, cm)
        ll, lc = crit.forward_heads(a, b, pri, tg)
        (ll + lc).backward()
        return ll.detach(), lc.detach(), lm, cm

    with torch.backends.cudnn.flags(enabled=True, deterministic=True, benchmark=False):
        for channels_last in (False, True):
            na = run(False, channels_last)
            nb = run(True, channels_last)
            assert all(m.dtype == torch.bfloat16 for m in na[2] + na[3])
            for x, y in zip(na[2] + na[3], nb[2] + nb[3]):
                assert torch.equal(bits(x), bits(y))              # the same maps on both sides
            assert float(na[0]) == float(nb[0]) and float(na[1]) == float(nb[1])
            for x, y in zip(na[2] + na[3], nb[2] + nb[3]):
                assert x.grad.dtype == torch.bfloat16 and torch.equal(bits(x.grad), bits(y.grad))


def misaligned_channels_last(m):
    """a channels_last copy of `m` whose data_ptr is 2-byte but not 8-byte aligned"""
    B, Cc, Hh, Ww = m.shape
    buf = torch.zeros(m.numel() + 4, dtype=m.dtype, device="cuda")
    v = buf.as_strided(tuple(m.shape), (Cc * Hh * Ww, 1, Ww * Cc, Cc), 1)
    v.copy_(m)
    assert v.data_ptr() % 8 == 2 and H.map_layout(v) == "channels_last"
    return v


@pytest.mark.gpu
def test_gpu_misaligned_channels_last_takes_the_scalar_path():
    from fdt_b200.layers import Detect, MultiBoxLoss, heads_to_loc_conf
    lm, cm, nm, p, tg = loss_setup("six_640", torch.bfloat16, 71)
    lg, cg = place(lm, "channels_last"), place(cm, "channels_last")
    lo = [misaligned_channels_last(m) for m in lg]
    co = [misaligned_channels_last(m) for m in cg]
    assert_same_detect(detect_aux(Detect(2, 0, 750, 0.05, 0.3), lo, co, p, nm), detect_aux(Detect(2, 0, 750, 0.05, 0.3), lg, cg, p, nm),
                       "misaligned")
    a, b = heads_to_loc_conf(lo, co, nm), heads_to_loc_conf(lg, cg, nm)
    assert torch.equal(bits(a[0]), bits(b[0])) and torch.equal(bits(a[1]), bits(b[1]))
    crit = MultiBoxLoss(2, 0.35, True, 0, True, 3, 0.35, False)
    outs = []
    for l_, c_ in ((lo, co), (lg, cg)):
        l_ = [m.detach().requires_grad_(True) for m in l_]       # (leaves: the misaligned views keep their storage offset)
        c_ = [m.detach().requires_grad_(True) for m in c_]
        ll, lc = crit.forward_heads(l_, c_, p, tg, nm)
        outs.append((ll.detach(), lc.detach(), torch.autograd.grad(ll + lc, l_ + c_)))
    assert float(outs[0][0]) == float(outs[1][0]) and float(outs[0][1]) == float(outs[1][1])
    for x, y in zip(outs[0][2], outs[1][2]):
        assert torch.equal(bits(x), bits(y))


@pytest.mark.gpu
def test_gpu_bf16_forward_heads_cuda_graph():
    """bf16 forward_heads + backward captured in a CUDA graph and replayed on new maps: the eager results of the new maps"""
    from fdt_b200.layers import MultiBoxLoss
    from fdt_b200.layers.modules.multibox_loss import _MultiBoxLossHeadsFn, pack_targets
    crit = MultiBoxLoss(2, 0.35, True, 0, True, 3, 0.35, False, bipartite=False)
    lm, cm, nm, p, tg = loss_setup("six_640x480", torch.bfloat16, 81)
    lm2, cm2, _, _, _ = loss_setup("six_640x480", torch.bfloat16, 82)
    lh = [m.requires_grad_(True) for m in place(lm, "channels_last")]
    ch = [m.requires_grad_(True) for m in place(cm, "nchw")]
    gt, off, total = pack_targets(tg, p.device)
    torch.cuda.synchronize()

    def step():
        ll, lc, *_ = _MultiBoxLossHeadsFn.apply(p, gt, off, total, crit.threshold, crit.negpos_ratio, crit.bipartite, crit.variance,
                                                tuple(nm), len(cm), *lh, *ch)
        (ll + lc).backward()
        return ll, lc
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
        torch.cuda.synchronize()
        for m in lh + ch:
            m.grad = None
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            ll_g, lc_g = step()
    torch.cuda.current_stream().wait_stream(side)
    with torch.no_grad():
        for dst, src in zip(lh + ch, place(lm2, "channels_last") + place(cm2, "nchw")):
            dst.copy_(src)
    torch.cuda.synchronize()
    g.replay()
    torch.cuda.synchronize()
    el = [m.detach().clone().requires_grad_(True) for m in lh]
    ec = [m.detach().clone().requires_grad_(True) for m in ch]
    ll_e, lc_e = crit.forward_heads(el, ec, p, tg, nm)
    (ll_e + lc_e).backward()
    assert float(ll_g.detach()) == float(ll_e.detach()) and float(lc_g.detach()) == float(lc_e.detach())
    for a, b in zip([m.grad for m in lh + ch], [m.grad for m in el + ec]):
        assert a.dtype == torch.bfloat16 and torch.equal(bits(a), bits(b))


@pytest.mark.gpu
def test_gpu_bf16_detect_heads_back_to_back():
    """four bf16 detect_heads calls back to back on one stream over a depth-4 workspace (the calls overlap on the device): every
    output equals its isolated call"""
    from fdt_b200.layers import Detect
    sets = []
    for i in range(4):
        lm, cm, nm, pri = rounded_maps(64, "six_640", 500 + i, torch.bfloat16)
        layout = LAYOUTS[i % 2]
        sets.append((place(lm, layout), place(cm, layout)))
    p = torch.from_numpy(pri).cuda()
    iso = []
    for lg, cg in sets:
        iso.append(detect_aux(Detect(2, 0, 750, 0.05, 0.3), lg, cg, p, nm))
        torch.cuda.synchronize()
    det = Detect(2, 0, 750, 0.05, 0.3)
    for _ in range(2):
        outs = [detect_aux(det, lg, cg, p, nm) for lg, cg in sets]
        torch.cuda.synchronize()
        for a, b in zip(outs, iso):
            assert_same_detect(a, b, "back to back")
