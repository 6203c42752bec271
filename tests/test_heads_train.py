"""Training from head maps: the backward of heads_to_loc_conf and MultiBoxLoss.forward_heads (fused loss from the per-level NCHW
maps, gradients written straight into the maps).

CPU part: the torch restatement of the head post-processing (tests/torch_heads_ref.py, the gradient oracle) against the
reference's own outputs in tests/golden/heads.npz, and the host-side argument checks of the new C entries.
GPU part: map gradients bit-identical to CPU torch autograd, forward_heads against MultiBoxLoss on the materialised tensors and
the C oracle, its map gradients against the two-step chain and autograd, CUDA-graph capture, argument errors."""
import ctypes as C

import numpy as np
import pytest
import torch

from fdt_b200 import _lib, synth
from oracle import oracle as orc
from tests.torch_heads_ref import heads as ref_heads

CASES = {"a": synth.STRIDES6, "b": synth.STRIDES6[:5]}
VAR = (0.1, 0.2)


def golden_maps(g, tag):
    """the heads.npz inputs of case `tag` (test_heads.py builds them the same way)"""
    B, w, h, seed, _ = (int(v) for v in g[tag + "_cfg"])
    loc_maps, conf_maps, neg_max = synth.head_maps(B, w, h, seed, CASES[tag])
    if tag == "a":
        conf_maps[1][0, 2, 3, 4] = np.nan
        conf_maps[0][1, 0, 5, 6] = np.inf
    assert synth.digest(*loc_maps, *conf_maps) == str(g[tag + "_in_sha"])
    return loc_maps, conf_maps, neg_max, (w, h)


@pytest.mark.parametrize("tag", ["a", "b"])
def test_torch_ref_heads_reproduce_reference(golden, tag):
    g = golden("heads")
    loc_maps, conf_maps, neg_max, _ = golden_maps(g, tag)
    loc, raw = ref_heads([torch.from_numpy(m) for m in loc_maps], [torch.from_numpy(m) for m in conf_maps], neg_max, softmax=False)
    assert synth.digest(loc.numpy()) == str(g[tag + "_loc_sha"])
    assert synth.digest(raw.numpy()) == str(g[tag + "_raw_sha"])


def level_arrays(L):
    fh = (C.c_int * 8)(*([4] * 8)); fw = (C.c_int * 8)(*([4] * 8)); nm = (C.c_int * 8)(*([0] * 8))
    fake = (C.c_void_p * 8)(*([256] * 8))
    return fh, fw, nm, fake


def test_new_entries_refuse_bad_arguments_without_a_gpu():
    lib = _lib.lib()
    fh, fw, nm, fake = level_arrays(8)
    p = C.c_void_p(256)
    for L in (0, 9):
        assert lib.fdt_heads_to_loc_conf_backward(fake, fh, fw, nm, L, 1, 0, p, p, fake, fake, None) == _lib.FDT_E_UNSUPPORTED
        assert lib.fdt_multibox_loss_forward_heads(fake, fake, fh, fw, nm, L, p, p, p, 1, 1, 0.35, 3, 0, 0.1, 0.2, p, p, p, p, p, None,
                                                   p, 1 << 30, None) == _lib.FDT_E_UNSUPPORTED
        assert lib.fdt_multibox_loss_backward_heads_dev(fake, fake, fh, fw, nm, L, p, p, p, p, p, p, 1, fake, fake, None) \
            == _lib.FDT_E_UNSUPPORTED
    # null maps
    assert lib.fdt_heads_to_loc_conf_backward(None, fh, fw, nm, 2, 1, 0, None, p, None, fake, None) == _lib.FDT_E_INVALID
    assert lib.fdt_heads_to_loc_conf_backward(fake, fh, fw, nm, 2, 1, 0, p, None, None, None, None) == _lib.FDT_E_INVALID
    assert lib.fdt_multibox_loss_forward_heads(None, fake, fh, fw, nm, 2, p, p, p, 1, 1, 0.35, 3, 0, 0.1, 0.2, p, p, p, p, p, None,
                                               p, 1 << 30, None) == _lib.FDT_E_INVALID
    assert lib.fdt_multibox_loss_forward_heads(fake, None, fh, fw, nm, 2, p, p, p, 1, 1, 0.35, 3, 0, 0.1, 0.2, p, p, p, p, p, None,
                                               p, 1 << 30, None) == _lib.FDT_E_INVALID
    assert lib.fdt_multibox_loss_backward_heads_dev(None, fake, fh, fw, nm, 2, p, p, p, p, p, p, 1, fake, fake, None) == _lib.FDT_E_INVALID
    assert lib.fdt_multibox_loss_backward_heads_dev(fake, fake, fh, fw, nm, 2, p, p, p, p, p, p, 1, fake, (C.c_void_p * 2)(256, None),
                                                    None) == _lib.FDT_E_INVALID
    # short workspace (N = 32 priors over two 4x4 levels; the bipartite matcher needs the most)
    need = lib.fdt_multibox_workspace_bytes(1, 32, 2, 1)
    for short in (16, need - 1):
        assert lib.fdt_multibox_loss_forward_heads(fake, fake, fh, fw, nm, 2, p, p, p, 1, 1, 0.35, 3, 1, 0.1, 0.2, p, p, p, p, p, None,
                                                   p, short, None) == _lib.FDT_E_WORKSPACE
    assert "workspace" in _lib.last_error()


# ------------------------------------------------------------------------------------------------------------------- GPU
def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def bits(t):
    return t.detach().float().cpu().contiguous().view(torch.int32)


def tied_maps():
    """Two levels, both max-in-out orientations: two- and three-way ties, +-0 pairs, NaN in the 2nd or 3rd channel of the triple."""
    rng = np.random.Generator(np.random.PCG64(11))
    conf = [rng.standard_normal((2, 4, 5, 6), dtype=np.float32) for _ in range(2)]
    loc = [rng.standard_normal((2, 4, 5, 6), dtype=np.float32) for _ in range(2)]
    for m, off in ((conf[0], 0), (conf[1], 1)):                       # the triple is ch0..2 (neg_max) or ch1..3
        t = [off, off + 1, off + 2]
        m[0, t[0], 0, 0] = m[0, t[1], 0, 0] = 1.0; m[0, t[2], 0, 0] = 0.5          # (1, 1, 0.5) -> first
        m[0, t[1], 0, 1] = m[0, t[2], 0, 1] = 2.0; m[0, t[0], 0, 1] = 0.0          # tie on the last two
        m[0, t[0], 0, 2] = m[0, t[1], 0, 2] = m[0, t[2], 0, 2] = 3.0               # three-way tie
        m[0, t[0], 0, 3] = -0.0; m[0, t[1], 0, 3] = 0.0; m[0, t[2], 0, 3] = -1.0   # (-0, +0, -1) -> first
        m[0, t[0], 0, 4] = 0.0; m[0, t[1], 0, 4] = -0.0; m[0, t[2], 0, 4] = -1.0
        m[1, t[0], 1, 0] = 1.0; m[1, t[1], 1, 0] = np.nan; m[1, t[2], 1, 0] = np.nan   # (1, NaN, NaN) -> second
        m[1, t[2], 1, 1] = np.nan                                                       # NaN in the third
        m[1, t[0], 1, 2] = np.inf; m[1, t[1], 1, 2] = np.inf                            # +inf tie
    return loc, conf


def map_cases(golden):
    g = golden("heads")
    out = []
    for tag in ("a", "b"):
        lm, cm, nm, _ = golden_maps(g, tag)
        out.append((tag, lm, cm, nm))
    loc, conf = tied_maps()
    out.append(("ties_neg_first", loc, conf, [1, 0]))
    out.append(("ties_pos_first", loc, conf, [0, 1]))
    return out


def torch_map_grads(loc_maps, conf_maps, neg_max, softmax, g_loc, g_conf, need=(True, True)):
    lm = [torch.from_numpy(m).requires_grad_(need[0]) for m in loc_maps]
    cm = [torch.from_numpy(m).requires_grad_(need[1]) for m in conf_maps]
    loc, conf = ref_heads(lm, cm, neg_max, softmax)
    outs, grads = [], []
    if need[0]:
        outs.append(loc); grads.append(g_loc)
    if need[1]:
        outs.append(conf); grads.append(g_conf)
    torch.autograd.backward(outs, grads)
    return [m.grad for m in lm] if need[0] else None, [m.grad for m in cm] if need[1] else None


def lib_map_grads(loc_maps, conf_maps, neg_max, softmax, g_loc, g_conf, need=(True, True)):
    from fdt_b200.layers import heads_to_loc_conf
    lm = [cu(m).requires_grad_(need[0]) for m in loc_maps]
    cm = [cu(m).requires_grad_(need[1]) for m in conf_maps]
    loc, conf = heads_to_loc_conf(lm, cm, neg_max, softmax=softmax)
    torch.autograd.backward([loc, conf], [g_loc.cuda(), g_conf.cuda()])
    return [m.grad for m in lm] if need[0] else None, [m.grad for m in cm] if need[1] else None


def upstream(loc_maps, seed):
    B = loc_maps[0].shape[0]
    N = sum(m.shape[2] * m.shape[3] for m in loc_maps)
    gen = torch.Generator().manual_seed(seed)
    return torch.randn((B, N, 4), generator=gen), torch.randn((B, N, 2), generator=gen)


@pytest.mark.gpu
def test_gpu_heads_backward_bit_identical_to_torch(golden):
    for i, (tag, lm, cm, nm) in enumerate(map_cases(golden)):
        g_loc, g_conf = upstream(lm, 100 + i)
        for need in ((True, True), (True, False), (False, True)):
            rl, rc = torch_map_grads(lm, cm, nm, False, g_loc, g_conf, need)
            gl, gc = lib_map_grads(lm, cm, nm, False, g_loc, g_conf, need)
            for r, o in zip(rl or [], gl or []):
                assert torch.equal(bits(r), bits(o)), (tag, need, "loc")
            for r, o in zip(rc or [], gc or []):
                assert torch.equal(bits(r), bits(o)), (tag, need, "conf")
            assert (gl is None) == (not need[0]) and (gc is None) == (not need[1])


@pytest.mark.gpu
def test_gpu_heads_backward_softmax(golden):
    for i, (tag, lm, cm, nm) in enumerate(map_cases(golden)):
        g_loc, g_conf = upstream(lm, 200 + i)
        rl, rc = torch_map_grads(lm, cm, nm, True, g_loc, g_conf)
        gl, gc = lib_map_grads(lm, cm, nm, True, g_loc, g_conf)
        for r, o in zip(rl, gl):
            assert torch.equal(bits(r), bits(o))
        atol = 1e-6 * float(g_conf.abs().max())
        for r, o in zip(rc, gc):
            torch.testing.assert_close(o.cpu(), r, rtol=1e-5, atol=atol, equal_nan=True)


@pytest.mark.gpu
def test_gpu_heads_no_grad_call_unchanged():
    from fdt_b200.layers import heads_to_loc_conf
    lm, cm, nm = synth.head_maps(2, 128, 96, 5)
    a = heads_to_loc_conf([cu(m) for m in lm], [cu(m) for m in cm], nm, softmax=False)
    b = heads_to_loc_conf([cu(m).requires_grad_(True) for m in lm], [cu(m).requires_grad_(True) for m in cm], nm, softmax=False)
    assert a[0].grad_fn is None and a[1].grad_fn is None and b[0].grad_fn is not None
    assert torch.equal(a[0], b[0]) and torch.equal(bits(a[1]), bits(b[1]))


# ---- forward_heads
def forward_heads_abi(lm, cm, nm, pri, targets, bip):
    """fdt_multibox_loss_forward_heads through the C ABI -> (losses, conf_t, loc_t, sel, loss_c_all) on the device"""
    from fdt_b200.layers.functions.heads import _level_args
    from fdt_b200.layers.modules.multibox_loss import pack_targets
    dev, B, N, keep, (lp, cp, fh, fw, nma, L) = _level_args(lm, cm, nm)
    gt, off, total = pack_targets([cu(t) for t in targets], dev)
    losses = torch.empty(2, device=dev); norm = torch.empty(1, device=dev)
    loc_t = torch.empty((B, N, 4), device=dev); conf_t = torch.empty((B, N), dtype=torch.int64, device=dev)
    sel = torch.empty((B, N), dtype=torch.uint8, device=dev); lca = torch.empty((B, N), device=dev)
    lib = _lib.lib()
    ws = _lib.workspace(lib.fdt_multibox_workspace_bytes(B, N, 2, total), dev, "t-heads")
    for _ in range(2):                     # twice on one workspace: the per-call state is re-initialised by the call
        _lib.check(lib.fdt_multibox_loss_forward_heads(lp, cp, fh, fw, nma, L, pri.data_ptr(), gt.data_ptr(), off.data_ptr(), total, B,
                                                       0.35, 3, bip, VAR[0], VAR[1], losses.data_ptr(), norm.data_ptr(), loc_t.data_ptr(),
                                                       conf_t.data_ptr(), sel.data_ptr(), lca.data_ptr(), ws.data_ptr(), ws.numel(),
                                                       _lib.stream_ptr()))
    return losses, conf_t, loc_t, sel, lca


def flat_abi(loc, conf, pri, targets, bip):
    from fdt_b200.layers.modules.multibox_loss import pack_targets
    dev = loc.device
    B, N, _ = loc.shape
    gt, off, total = pack_targets([cu(t) for t in targets], dev)
    losses = torch.empty(2, device=dev); norm = torch.empty(1, device=dev)
    loc_t = torch.empty((B, N, 4), device=dev); conf_t = torch.empty((B, N), dtype=torch.int64, device=dev)
    sel = torch.empty((B, N), dtype=torch.uint8, device=dev); lca = torch.empty((B, N), device=dev)
    lib = _lib.lib()
    ws = _lib.workspace(lib.fdt_multibox_workspace_bytes(B, N, 2, total), dev, "t-flat")
    _lib.check(lib.fdt_multibox_loss_forward(loc.data_ptr(), conf.data_ptr(), pri.data_ptr(), gt.data_ptr(), off.data_ptr(), total, B, N, 2,
                                             0.35, 3, bip, VAR[0], VAR[1], losses.data_ptr(), norm.data_ptr(), loc_t.data_ptr(),
                                             conf_t.data_ptr(), sel.data_ptr(), lca.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr()))
    return losses, conf_t, loc_t, sel, lca


def geometry_cases(golden):
    """(name, loc_maps, conf_maps, neg_max, priors, targets, check_oracle)"""
    g = golden("heads")
    out = []
    for tag, strides, boxes in (("a", synth.STRIDES6, synth.BOXES6), ("b", synth.STRIDES6[:5], synth.BOXES6[:5])):
        lm, cm, nm, (w, h) = golden_maps(g, tag)
        pri = synth.priors_numpy(w, h, strides, boxes)
        _, _, targets = synth.multibox_inputs(lm[0].shape[0], pri, 900 + ord(tag), 1, 30)
        out.append((tag, lm, cm, nm, pri, targets, tag != "a"))      # (a: NaN / inf logits, covered by the flat tests)
    pri = synth.priors_numpy(640, 640)
    lm, cm, nm = synth.head_maps(32, 640, 640, 3031)
    _, _, targets = synth.multibox_inputs(32, pri, 3030, 0, 200)
    targets[5] = np.zeros((0, 5), np.float32)
    out.append(("b32_640_config3", lm, cm, nm, pri, targets, True))
    pri = synth.priors_numpy(1024, 1024)
    lm, cm, nm = synth.head_maps(4, 1024, 1024, 1025)
    _, _, targets = synth.multibox_inputs(4, pri, 1026, 1500, 1968)
    out.append(("b4_1024_many_gt", lm, cm, nm, pri, targets, False))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("bip", [0, 1])
def test_gpu_forward_heads_equals_materialised(golden, bip):
    from fdt_b200.layers import heads_to_loc_conf
    for name, lm, cm, nm, pri, targets, with_oracle in geometry_cases(golden):
        lmc, cmc, p = [cu(m) for m in lm], [cu(m) for m in cm], cu(pri)
        loss_h, conf_t_h, loc_t_h, sel_h, lca_h = forward_heads_abi(lmc, cmc, nm, p, targets, bip)
        loc, conf = heads_to_loc_conf(lmc, cmc, nm, softmax=False)
        loss_f, conf_t_f, loc_t_f, sel_f, lca_f = flat_abi(loc, conf, p, targets, bip)
        assert torch.equal(conf_t_h, conf_t_f), name
        assert torch.equal(bits(loc_t_h), bits(loc_t_f)), name
        assert torch.equal(sel_h, sel_f), name
        assert torch.equal(bits(lca_h), bits(lca_f)), name
        np.testing.assert_allclose(loss_h.cpu().numpy(), loss_f.cpu().numpy(), rtol=1e-6)
        if with_oracle:
            raw = orc.heads_to_loc_conf(lm, cm, nm, softmax=False)
            r = orc.multibox_loss(raw[0], raw[1], pri, targets, 0.35, 3, bool(bip), VAR)
            ct = conf_t_h.cpu().numpy()
            assert np.array_equal(ct, r["conf_t"]), name
            assert np.array_equal(sel_h.cpu().numpy().astype(bool), r["neg"] | (r["conf_t"] > 0)), name
            np.testing.assert_allclose(loss_h.cpu().numpy(), [r["loss_l"], r["loss_c"]], rtol=1e-5, atol=1e-7)


def torch_reference_loss(loc, conf, loc_t, conf_t, sel):
    """plain PyTorch fp32 statement of multibox_loss.py:90-135 given targets and the selection mask"""
    pos = conf_t > 0
    loss_l = torch.nn.functional.smooth_l1_loss(loc[pos], loc_t[pos], reduction="sum")
    loss_c = torch.nn.functional.cross_entropy(conf[sel.bool()], conf_t[sel.bool()], reduction="sum")
    n = pos.sum().float().clamp(min=1)
    return loss_l / n, loss_c / n


@pytest.mark.gpu
@pytest.mark.parametrize("bip", [0, 1])
def test_gpu_forward_heads_map_gradients(golden, bip):
    from fdt_b200.layers import MultiBoxLoss, heads_to_loc_conf
    crit = MultiBoxLoss(2, 0.35, True, 0, True, 3, 0.35, False, bipartite=bool(bip))
    for name, lm, cm, nm, pri, targets, finite in geometry_cases(golden)[:3]:
        p = cu(pri)
        tg = [cu(t) for t in targets]
        lh = [cu(m).requires_grad_(True) for m in lm]; ch = [cu(m).requires_grad_(True) for m in cm]
        ll, lc = crit.forward_heads(lh, ch, p, tg, nm)
        (ll + 0.5 * lc).backward()
        loc_t, conf_t, sel = crit.last_aux
        # two-step chain: differentiable heads_to_loc_conf, then MultiBoxLoss
        l2 = [cu(m).requires_grad_(True) for m in lm]; c2 = [cu(m).requires_grad_(True) for m in cm]
        ll2, lc2 = crit((*heads_to_loc_conf(l2, c2, nm, softmax=False), p), tg)
        (ll2 + 0.5 * lc2).backward()
        for a, b in zip(lh + ch, l2 + c2):
            assert torch.equal(bits(a.grad), bits(b.grad)), name
        np.testing.assert_allclose([float(ll), float(lc)], [float(ll2), float(lc2)], rtol=1e-6)
        if not finite:
            continue
        # torch autograd through the restated heads + a plain-torch loss given the library's conf_t and sel
        l3 = [torch.from_numpy(m).cuda().requires_grad_(True) for m in lm]; c3 = [torch.from_numpy(m).cuda().requires_grad_(True) for m in cm]
        loc, conf = ref_heads(l3, c3, nm, softmax=False)
        rl, rc = torch_reference_loss(loc, conf, loc_t, conf_t, sel)
        (rl + 0.5 * rc).backward()
        for a, b in zip(lh + ch, l3 + c3):
            np.testing.assert_allclose(a.grad.cpu().numpy(), b.grad.cpu().numpy(), rtol=1e-4, atol=1e-7)


@pytest.mark.gpu
def test_gpu_forward_heads_cuda_graph():
    """forward_heads' autograd function and its backward captured in a CUDA graph (the targets packed once, outside the capture:
    pack_targets copies the offsets from the host) and replayed: the same losses and map gradients as an eager run."""
    from fdt_b200.layers import MultiBoxLoss
    from fdt_b200.layers.modules.multibox_loss import _MultiBoxLossHeadsFn, pack_targets
    crit = MultiBoxLoss(2, 0.35, True, 0, True, 3, 0.35, False, bipartite=False)
    pri = synth.priors_numpy(320, 256)
    lm, cm, nm = synth.head_maps(4, 320, 256, 21)
    _, _, targets = synth.multibox_inputs(4, pri, 22, 1, 40)
    p = cu(pri)
    ll_e, lc_e = crit.forward_heads([cu(m) for m in lm], [cu(m) for m in cm], p, [cu(t) for t in targets], nm)
    lh = [cu(m).requires_grad_(True) for m in lm]; ch = [cu(m).requires_grad_(True) for m in cm]
    gt, off, total = pack_targets([cu(t) for t in targets], p.device)
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
        eager = [m.grad.clone() for m in lh + ch]
        torch.cuda.synchronize()
        for m in lh + ch:
            m.grad = None
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            ll_g, lc_g = step()
    torch.cuda.current_stream().wait_stream(side)
    for m in lh + ch:
        m.grad.zero_()
    ll_g.zero_(); lc_g.zero_()
    torch.cuda.synchronize()
    g.replay()
    torch.cuda.synchronize()
    assert float(ll_g) == float(ll_e) and float(lc_g) == float(lc_e)
    for a, b in zip(eager, [m.grad for m in lh + ch]):
        assert torch.equal(bits(a), bits(b))


@pytest.mark.gpu
def test_gpu_forward_heads_argument_errors():
    from fdt_b200.layers import MultiBoxLoss
    lm, cm, nm = synth.head_maps(2, 64, 64, 3)
    pri = cu(synth.priors_numpy(64, 64))
    _, _, targets = synth.multibox_inputs(2, synth.priors_numpy(64, 64), 4, 1, 5)
    tg = [cu(t) for t in targets]
    lmc, cmc = [cu(m) for m in lm], [cu(m) for m in cm]
    with pytest.raises(NotImplementedError):
        MultiBoxLoss(3, 0.35, True, 0, True, 3, 0.35, False).forward_heads(lmc, cmc, pri, tg)
    crit = MultiBoxLoss(2, 0.35, True, 0, True, 3, 0.35, False)
    with pytest.raises(ValueError):
        crit.forward_heads(lmc, cmc, pri[:-1], tg)
    with pytest.raises(ValueError):
        crit.forward_heads(lmc, [cmc[0][:1]] + cmc[1:], pri, tg)
    with pytest.raises(ValueError):
        crit.forward_heads(lmc[:-1], cmc, pri, tg)
