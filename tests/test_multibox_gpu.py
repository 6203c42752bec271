"""GPU parity tests for match/encode, hard-negative mining and MultiBoxLoss (forward + backward)."""
import numpy as np
import pytest
import torch

from fdt_b200 import synth
from oracle import oracle as orc

pytestmark = pytest.mark.gpu
VAR = (0.1, 0.2)


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def npy(t):
    return t.detach().cpu().numpy()


@pytest.fixture(scope="module")
def layers():
    import fdt_b200.layers as L
    return L


def gpu_match(bip, thr, gt, pri, want_best=True):
    """fdt_match_encode for one image -> loc_t, conf_t, best_truth_idx, best_truth_overlap (numpy)."""
    return tuple(a[0] for a in gpu_match_batch(bip, thr, [gt], pri))


def gpu_match_batch(bip, thr, gts, pri):
    """fdt_match_encode for len(gts) images in one call -> loc_t, conf_t, best_truth_idx, best_truth_overlap [B,N,...] (numpy)."""
    from fdt_b200 import _lib
    dev = torch.device("cuda", torch.cuda.current_device())
    B, N = len(gts), pri.shape[0]
    gt = np.concatenate(gts).astype(np.float32)
    g = cu(gt); p = cu(pri)
    off = torch.tensor(np.cumsum([0] + [t.shape[0] for t in gts]), dtype=torch.int64, device=dev)
    lt = torch.empty((B, N, 4), dtype=torch.float32, device=dev); ct = torch.empty((B, N), dtype=torch.int64, device=dev)
    bti = torch.empty((B, N), dtype=torch.int32, device=dev); bto = torch.empty((B, N), dtype=torch.float32, device=dev)
    L = _lib.lib()
    ws = _lib.workspace(L.fdt_match_workspace_bytes(B, N, gt.shape[0]), dev, "t")
    _lib.check(L.fdt_match_encode(p.data_ptr(), g.data_ptr(), off.data_ptr(), gt.shape[0], B, N, thr, VAR[0], VAR[1], int(bip),
                                  lt.data_ptr(), ct.data_ptr(), bti.data_ptr(), bto.data_ptr(), ws.data_ptr(), ws.numel(),
                                  _lib.stream_ptr()))
    return npy(lt), npy(ct), npy(bti), npy(bto)


@pytest.mark.parametrize("tag", ["g1", "g7", "g60"])
@pytest.mark.parametrize("bip", [0, 1])
def test_match_golden(golden, tag, bip):
    g = golden("multibox")
    gt, pri = g[f"{tag}_gt"], g["small_priors"]
    lt, ct, bti, bto = gpu_match(bip, 0.35, gt, pri)
    assert np.array_equal(ct, g[f"{tag}_b{bip}_conf_t"])                      # labels bit-exact vs the reference
    if not bip:
        assert np.array_equal(bti, g[f"{tag}_b{bip}_bti"])                    # match indices bit-exact
    np.testing.assert_allclose(lt, g[f"{tag}_b{bip}_loc_t"], rtol=1e-5, atol=1e-6)
    o_lt, o_ct, o_bti, o_bto = orc.match(bip, 0.35, gt[:, :4], pri, VAR, gt[:, 4])
    assert np.array_equal(ct, o_ct) and np.array_equal(bti, o_bti) and np.array_equal(bto, o_bto)
    np.testing.assert_allclose(lt, o_lt, rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("G,bip,seed", [(1, 0, 1), (200, 0, 2), (200, 1, 3), (257, 1, 4), (700, 0, 5), (1968, 1, 6),
                                        ((300, 0, 120), 0, 7), ((300, 0, 120), 1, 7)])
def test_match_production_size_vs_oracle(G, bip, seed):
    """N = 34,125; G up to the WIDER maximum (1,968 faces) -> several shared-memory GT tiles.  A tuple of G: one call for that
    many images (gt_off beyond the first image), one of them without GT boxes (all background, zeros everywhere)."""
    pri = synth.priors_numpy(640, 640)
    rng = np.random.Generator(np.random.PCG64(seed))
    gts = [synth.gt_boxes(g, rng) for g in (G if isinstance(G, tuple) else (G,))]
    for gt, (lt, ct, bti, bto) in zip(gts, zip(*gpu_match_batch(bip, 0.35, gts, pri))):
        if gt.shape[0] == 0:
            assert not lt.any() and not ct.any() and not bti.any() and not bto.any()
            continue
        o_lt, o_ct, o_bti, o_bto = orc.match(bip, 0.35, gt[:, :4], pri, VAR, gt[:, 4])
        assert np.array_equal(ct, o_ct) and np.array_equal(bti, o_bti) and np.array_equal(bto, o_bto)
        np.testing.assert_allclose(lt, o_lt, rtol=1e-6, atol=1e-7)


def test_match_duplicate_gt_ties(golden):
    """identical GT boxes: per-prior argmax keeps the first GT; bipartite override keeps the last (box_utils.py:153-154)."""
    pri = golden("multibox")["small_priors"]
    gt = np.array([[0.2, 0.2, 0.4, 0.4, 0], [0.2, 0.2, 0.4, 0.4, 0], [0.6, 0.6, 0.7, 0.8, 0]], np.float32)
    for bip in (0, 1):
        lt, ct, bti, bto = gpu_match(bip, 0.35, gt, pri)
        o_lt, o_ct, o_bti, o_bto = orc.match(bip, 0.35, gt[:, :4], pri, VAR, gt[:, 4])
        assert np.array_equal(ct, o_ct) and np.array_equal(bti, o_bti) and np.array_equal(bto, o_bto)


def test_box_utils_match_dropin_signature(layers, golden):
    g = golden("multibox")
    gt, pri = g["g7_gt"], g["small_priors"]
    N = pri.shape[0]
    for fn, bip in ((layers.box_utils.match_default, 0), (layers.box_utils.match_ensure_max_prior, 1)):
        loc_t = torch.zeros(3, N, 4); conf_t = torch.zeros(3, N, dtype=torch.long)
        fn(0.35, torch.from_numpy(gt[:, :4]), torch.from_numpy(pri), list(VAR), torch.from_numpy(gt[:, 4]), loc_t, conf_t, 1)
        assert np.array_equal(conf_t[1].numpy(), g[f"g7_b{bip}_conf_t"])
        assert not conf_t[0].any() and not conf_t[2].any()
    with pytest.raises(IndexError):
        layers.box_utils.match_default(0.35, torch.zeros(0, 4), torch.from_numpy(pri), list(VAR), torch.zeros(0),
                                       torch.zeros(1, N, 4), torch.zeros(1, N, dtype=torch.long), 0)


# ------------------------------------------------------------------------------- mining
def gpu_mine(loss_c, pos, ratio):
    from fdt_b200 import _lib
    dev = torch.device("cuda", torch.cuda.current_device())
    B, N = loss_c.shape
    lc = cu(loss_c.astype(np.float32)); ps = cu(pos.astype(np.uint8))
    neg = torch.empty((B, N), dtype=torch.uint8, device=dev)
    L = _lib.lib()
    ws = _lib.workspace(L.fdt_mine_workspace_bytes(B, N), dev, "mine")
    _lib.check(L.fdt_hard_negative_mine(lc.data_ptr(), ps.data_ptr(), B, N, ratio, neg.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr()))
    return npy(neg).astype(bool)


@pytest.mark.parametrize("bip", [0, 1])
def test_mining_on_reference_loss_bit_exact(golden, bip):
    g = golden("multibox")
    lc = g[f"fwd_b{bip}_loss_c_all"]; pos = g[f"fwd_b{bip}_conf_t"] > 0
    neg_ref = np.unpackbits(g[f"fwd_b{bip}_neg"])[:lc.size].reshape(lc.shape).astype(bool)
    assert np.array_equal(gpu_mine(lc, pos, 3), neg_ref)


@pytest.mark.parametrize("N,npos,ratio", [(34125, 50, 3), (34125, 0, 3), (34125, 20000, 3), (87360, 300, 3), (1000, 10, 7), (33, 4, 3)])
def test_mining_vs_oracle_including_ties(N, npos, ratio):
    rng = np.random.Generator(np.random.PCG64(N + npos))
    B = 5
    lc = rng.uniform(0, 5, (B, N)).astype(np.float32)
    lc[1] = np.round(lc[1] * 4) / 4                         # heavy ties: boundary value duplicated
    lc[2, ::2] = 0.0
    # the rest of the float range, which the mining histogram clamps into its first and last bins: NaN of either sign, negatives,
    # values below 2^-8 down to subnormals, values above 2^8, infinities (no -0.0: the reference's sort ties it with +0.0)
    nan2 = np.array([0x7FC00000, 0xFFC00000], np.uint32).view(np.float32)
    kinds = np.stack([nan2[rng.integers(0, 2, N)], -rng.uniform(1e-6, 1e3, N),
                      rng.uniform(0, 2.0 ** -8, N) * 10.0 ** -rng.integers(0, 40, N), rng.uniform(2.0 ** 8, 2.0 ** 30, N),
                      np.where(rng.random(N) < 0.5, np.inf, -np.inf)]).astype(np.float32)
    lc[3] = kinds[rng.integers(0, 5, N), np.arange(N)]
    lc[4] = 1.5                                             # one value: every prior in the cutoff bin
    pos = np.zeros((B, N), bool)
    for b in range(B):
        pos[b, rng.permutation(N)[:npos]] = True
    lc[pos] = 0
    assert np.array_equal(gpu_mine(lc, pos, ratio), orc.hard_negative_mine(lc, pos, ratio))


# ------------------------------------------------------------------------------- MultiBoxLoss
def run_loss(layers, loc, conf, pri, targets, bip, host=False):
    crit = layers.MultiBoxLoss(2, 0.35, True, 0, True, 3, 0.35, False, bipartite=bool(bip))
    f = (lambda a: torch.from_numpy(a)) if host else cu
    l = f(loc).requires_grad_(True); c = f(conf).requires_grad_(True)
    ll, lc = crit((l, c, f(pri)), [f(t) for t in targets])
    return crit, l, c, ll, lc


@pytest.mark.parametrize("bip", [0, 1])
def test_multibox_forward_golden_small(layers, golden, bip):
    g = golden("multibox")
    pri = g["small_priors"]
    loc, conf, targets = synth.multibox_inputs(4, pri, int(g["fwd_seed"]), 1, 20)
    crit, l, c, ll, lc = run_loss(layers, loc, conf, pri, targets, bip)
    np.testing.assert_allclose([float(ll), float(lc)], g[f"fwd_b{bip}_loss"], rtol=1e-5)
    loc_t, conf_t, sel = (npy(t) for t in crit.last_aux)
    assert np.array_equal(conf_t, g[f"fwd_b{bip}_conf_t"])
    neg_ref = np.unpackbits(g[f"fwd_b{bip}_neg"])[:conf_t.size].reshape(conf_t.shape).astype(bool)
    assert np.array_equal(sel.astype(bool), neg_ref | (conf_t > 0))            # mined negatives bit-exact
    pos = conf_t > 0                       # the fused forward encodes the positives only (zeros elsewhere); match_* fill every row
    np.testing.assert_allclose(loc_t[pos], g[f"fwd_b{bip}_loc_t"][pos], rtol=1e-5, atol=1e-6)
    assert not loc_t[~pos].any()


def test_multibox_forward_golden_production_size(layers, golden):
    g = golden("multibox")
    pri = synth.priors_numpy(640, 640)
    loc, conf, targets = synth.multibox_inputs(2, pri, int(g["big_seed"]), 1, 200)
    crit, l, c, ll, lc = run_loss(layers, loc, conf, pri, targets, 0)
    np.testing.assert_allclose([float(ll), float(lc)], g["big_loss"], rtol=1e-5)
    _, conf_t, sel = (npy(t) for t in crit.last_aux)
    assert np.array_equal(conf_t, g["big_conf_t"])
    neg_ref = np.unpackbits(g["big_neg"])[:conf_t.size].reshape(conf_t.shape).astype(bool)
    assert np.array_equal(sel.astype(bool), neg_ref | (conf_t > 0))


@pytest.mark.parametrize("bip", [0, 1])
def test_multibox_batch32_config3_vs_oracle(layers, bip):
    """BASELINE config 3: B=32, N=34,125, G_i in [0,200] (zero-GT images are defined as all-background)."""
    pri = synth.priors_numpy(640, 640)
    loc, conf, targets = synth.multibox_inputs(32, pri, 3030, 0, 200)
    targets[5] = np.zeros((0, 5), np.float32)
    crit, l, c, ll, lc = run_loss(layers, loc, conf, pri, targets, bip)
    r = orc.multibox_loss(loc, conf, pri, targets, 0.35, 3, bool(bip), VAR)
    loc_t, conf_t, sel = (npy(t) for t in crit.last_aux)
    assert np.array_equal(conf_t, r["conf_t"])
    assert np.array_equal(sel.astype(bool), r["neg"] | (r["conf_t"] > 0))
    pos = conf_t > 0
    np.testing.assert_allclose(loc_t[pos], r["loc_t"][pos], rtol=1e-6, atol=1e-7)
    assert not loc_t[~pos].any()
    np.testing.assert_allclose([float(ll), float(lc)], [r["loss_l"], r["loss_c"]], rtol=1e-5)


def torch_reference_loss(loc, conf, loc_t, conf_t, sel):
    """plain PyTorch fp32 statement of multibox_loss.py:90-135 given targets and the selection mask."""
    pos = conf_t > 0
    loss_l = torch.nn.functional.smooth_l1_loss(loc[pos], loc_t[pos], reduction="sum")
    loss_c = torch.nn.functional.cross_entropy(conf[sel.bool()], conf_t[sel.bool()], reduction="sum")
    n = pos.sum().float().clamp(min=1)
    return loss_l / n, loss_c / n


def test_multibox_backward_matches_autograd(layers, golden):
    g = golden("multibox")
    pri = g["small_priors"]
    loc, conf, targets = synth.multibox_inputs(4, pri, 404, 1, 20)
    crit, l, c, ll, lc = run_loss(layers, loc, conf, pri, targets, 0)
    (ll + 0.5 * lc).backward()
    loc_t, conf_t, sel = crit.last_aux
    l2 = cu(loc).requires_grad_(True); c2 = cu(conf).requires_grad_(True)
    rl, rc = torch_reference_loss(l2, c2, loc_t, conf_t, sel)
    (rl + 0.5 * rc).backward()
    np.testing.assert_allclose(npy(l.grad), npy(l2.grad), rtol=1e-4, atol=1e-7)
    np.testing.assert_allclose(npy(c.grad), npy(c2.grad), rtol=1e-4, atol=1e-7)
    np.testing.assert_allclose([float(ll), float(lc)], [float(rl), float(rc)], rtol=1e-5)


@pytest.mark.parametrize("bip", [0, 1])
def test_multibox_sign_bit_nan_logit_poisons_the_global_max(layers, bip):
    """x.max() of log_sum_exp (box_utils.py:268) propagates ANY NaN, also x86's default quiet NaN with the sign bit set, which
    an order-preserving key alone would rank lowest: every row of the mining loss becomes NaN, exactly as in the oracle."""
    pri = synth.priors_numpy(160, 160)
    loc, conf, targets = synth.multibox_inputs(3, pri, 66, 1, 12)
    conf = conf.copy()
    conf.view(np.uint32)[1, 77, 0] = 0xFFC00000                                  # -NaN
    assert np.isnan(conf[1, 77, 0]) and np.signbit(conf[1, 77, 0])
    dev = torch.device("cuda", torch.cuda.current_device())
    from fdt_b200 import _lib
    from fdt_b200.layers.modules.multibox_loss import pack_targets
    l, c, p = cu(loc), cu(conf), cu(pri)
    gt, off, total = pack_targets([cu(t) for t in targets], dev)
    B, N = 3, pri.shape[0]
    losses = torch.empty(2, device=dev); norm = torch.empty(1, device=dev)
    loc_t = torch.empty((B, N, 4), device=dev); conf_t = torch.empty((B, N), dtype=torch.int64, device=dev)
    sel = torch.empty((B, N), dtype=torch.uint8, device=dev); lca = torch.empty((B, N), device=dev)
    L = _lib.lib()
    ws = _lib.workspace(L.fdt_multibox_workspace_bytes(B, N, 2, total), dev, "t-nan")
    _lib.check(L.fdt_multibox_loss_forward(l.data_ptr(), c.data_ptr(), p.data_ptr(), gt.data_ptr(), off.data_ptr(), total, B, N, 2,
                                           0.35, 3, bip, 0.1, 0.2, losses.data_ptr(), norm.data_ptr(), loc_t.data_ptr(), conf_t.data_ptr(),
                                           sel.data_ptr(), lca.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr()))
    r = orc.multibox_loss(loc, conf, pri, targets, 0.35, 3, bool(bip), VAR)
    got = npy(lca)
    pos = r["conf_t"] > 0
    assert np.isnan(got[~pos]).all() and np.isnan(r["loss_c_all"][~pos]).all()  # every non-positive row is NaN on both sides
    assert np.array_equal(npy(conf_t), r["conf_t"])
    assert np.array_equal(npy(sel).astype(bool), r["neg"] | pos)                 # all-NaN ties: lower prior index first on both sides


def test_multibox_cpu_tensor_inputs(layers, golden):
    g = golden("multibox")
    pri = g["small_priors"]
    loc, conf, targets = synth.multibox_inputs(4, pri, 404, 1, 20)
    crit, l, c, ll, lc = run_loss(layers, loc, conf, pri, targets, 0, host=True)
    assert ll.device.type == "cpu"
    np.testing.assert_allclose([float(ll), float(lc)], g["fwd_b0_loss"], rtol=1e-5)
    (ll + lc).backward()
    assert l.grad is not None and l.grad.device.type == "cpu" and float(l.grad.abs().sum()) > 0


def test_multibox_no_positive_anywhere(layers, golden):
    """num_pos == 0 -> N = batch size (multibox_loss.py:132-133), nothing mined -> both losses 0."""
    pri = golden("multibox")["small_priors"]
    loc, conf, _ = synth.multibox_inputs(2, pri, 9, 1, 2)
    targets = [np.array([[0.9, 0.9, 0.9001, 0.9001, 0]], np.float32)] * 2
    crit, l, c, ll, lc = run_loss(layers, loc, conf, pri, targets, 0)
    assert float(ll) == 0.0 and float(lc) == 0.0


# ------------------------------------------------------------------ fused forward: shapes and degenerate rows vs the oracle
def fused_forward(loc, conf, pri, targets, bip=0, thr=0.35, ratio=3):
    """fdt_multibox_loss_forward through the C ABI -> (losses[2], conf_t, loc_t, sel, loss_c_all) as numpy."""
    from fdt_b200 import _lib
    from fdt_b200.layers.modules.multibox_loss import pack_targets
    dev = torch.device("cuda", torch.cuda.current_device())
    l, c, p = cu(loc), cu(conf), cu(pri)
    gt, off, total = pack_targets([cu(t) for t in targets], dev)
    B, N, Cn = conf.shape
    losses = torch.empty(2, device=dev); norm = torch.empty(1, device=dev)
    loc_t = torch.empty((B, N, 4), device=dev); conf_t = torch.empty((B, N), dtype=torch.int64, device=dev)
    sel = torch.empty((B, N), dtype=torch.uint8, device=dev); lca = torch.empty((B, N), device=dev)
    L = _lib.lib()
    ws = _lib.workspace(L.fdt_multibox_workspace_bytes(B, N, Cn, total), dev, "t-fused")
    for _ in range(2):                     # twice on the same workspace: the per-call state is re-zeroed by the call itself
        _lib.check(L.fdt_multibox_loss_forward(l.data_ptr(), c.data_ptr(), p.data_ptr(), gt.data_ptr(), off.data_ptr(), total, B, N, Cn,
                                               thr, ratio, bip, VAR[0], VAR[1], losses.data_ptr(), norm.data_ptr(), loc_t.data_ptr(),
                                               conf_t.data_ptr(), sel.data_ptr(), lca.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr()))
    return npy(losses), npy(conf_t), npy(loc_t), npy(sel).astype(bool), npy(lca)


def check_fused(loc, conf, pri, targets, bip=0, thr=0.35, ratio=3, rtol=1e-5):
    losses, conf_t, loc_t, sel, lca = fused_forward(loc, conf, pri, targets, bip, thr, ratio)
    r = orc.multibox_loss(loc, conf, pri, targets, thr, ratio, bool(bip), VAR)
    assert np.array_equal(conf_t, r["conf_t"])
    pos = conf_t > 0
    assert np.array_equal(lca.view(np.uint32), r["loss_c_all"].view(np.uint32))      # the mining input bit for bit
    assert np.array_equal(sel, r["neg"] | pos)                                       # mined mask bit-exact
    np.testing.assert_allclose(loc_t[pos], r["loc_t"][pos], rtol=1e-6, atol=1e-7)
    assert not loc_t[~pos].any()
    np.testing.assert_allclose(losses, [r["loss_l"], r["loss_c"]], rtol=rtol, atol=1e-7)
    return sel, pos


@pytest.mark.parametrize("bip", [0, 1])
@pytest.mark.parametrize("kind", ["all_equal", "confident", "quantised"])
def test_fused_forward_degenerate_losses(kind, bip):
    """Rows whose mining cutoff cannot be settled by the histogram alone: every loss equal (34 k candidates in the cutoff bin -> the
    radix path, selection by prior index), near-zero losses (cutoff in bin 0 together with the zeros of the positives), and losses
    on a coarse grid (a few thousand ties around the cutoff)."""
    pri = synth.priors_numpy(640, 640)
    loc, conf, targets = synth.multibox_inputs(3, pri, 515, 20, 60)
    rng = np.random.Generator(np.random.PCG64(3))
    if kind == "all_equal":
        conf = np.zeros_like(conf)
    elif kind == "confident":
        conf = np.stack([np.full(conf.shape[:2], 9.0, np.float32), np.full(conf.shape[:2], -9.0, np.float32)], -1)
        conf += rng.uniform(-1e-3, 1e-3, conf.shape).astype(np.float32)
    else:
        conf = (np.round(conf * 2) / 2).astype(np.float32)
    sel, pos = check_fused(loc, conf, pri, targets, bip)
    assert (sel & ~pos).sum() > 0


@pytest.mark.parametrize("bip", [0, 1])
@pytest.mark.parametrize("thr", [0.0, 0.01, 0.35, 0.5, 0.9])
def test_fused_forward_many_gt_tiles_and_thresholds(thr, bip):
    """G = 600 boxes per image (three staged tiles) at thresholds from 'area bound off' to 'almost nothing matches': the area bound
    of the fused matcher never changes a label or an encoded row."""
    pri = synth.priors_numpy(320, 320)
    loc, conf, targets = synth.multibox_inputs(2, pri, 77, 600, 600)
    rng = np.random.Generator(np.random.PCG64(5))
    for t in targets:                                                            # all box sizes from 1 % to 60 % of the image
        c = rng.uniform(0.1, 0.9, (t.shape[0], 2)); s = rng.uniform(0.01, 0.6, (t.shape[0], 2))
        t[:, :4] = np.concatenate([c - s / 2, c + s / 2], 1).astype(np.float32)
    check_fused(loc, conf, pri, targets, bip, thr)


@pytest.mark.parametrize("bip", [0, 1])
@pytest.mark.parametrize("shape", [(1, 100), (2, 257), (1, 2049), (5, 4097)])
def test_fused_forward_odd_sizes(shape, bip):
    B, N = shape
    pri = synth.priors_numpy(320, 320)[-N:].copy()
    loc, conf, targets = synth.multibox_inputs(B, pri, 1000 + N, 1, 9)
    check_fused(loc, conf, pri, targets, bip)


def test_fused_forward_four_classes():
    pri = synth.priors_numpy(160, 160)
    loc, conf, targets = synth.multibox_inputs(3, pri, 31, 3, 30)
    rng = np.random.Generator(np.random.PCG64(9))
    conf = rng.standard_normal((3, pri.shape[0], 4)).astype(np.float32)
    for t in targets:
        t[:, 4] = rng.integers(0, 3, t.shape[0])
    check_fused(loc, conf, pri, targets, 0)


def test_fused_forward_degenerate_boxes():
    """zero-area, inverted and NaN GT boxes and a zero-size prior: labels and mask as the oracle (the area bound steps aside)."""
    pri = synth.priors_numpy(160, 160).copy()
    loc, conf, targets = synth.multibox_inputs(3, pri, 8, 6, 12)
    targets[0][1, :4] = [0.3, 0.3, 0.3, 0.5]
    targets[0][2, :4] = [0.6, 0.6, 0.4, 0.4]
    targets[1][0, :4] = [0.5, 0.5, 0.2, 0.7]
    targets[2][3, :4] = [np.nan, 0.2, 0.4, 0.4]
    pri[1234, 2:] = 0.0
    losses, conf_t, loc_t, sel, lca = fused_forward(loc, conf, pri, targets, 0)
    r = orc.multibox_loss(loc, conf, pri, targets, 0.35, 3, False, VAR)
    assert np.array_equal(conf_t, r["conf_t"])
    assert np.array_equal(sel, r["neg"] | (conf_t > 0))


def test_fused_forward_bipartite_shared_best_priors():
    """box_utils.py:150-154: many GT boxes with the SAME best prior (100 copies of one box: more forced matches in one block than
    its list holds), boxes no prior overlaps (best prior = prior 0) and tiny / elongated boxes whose best overlap is far below the
    threshold: the last GT wins a shared prior, every box still claims one."""
    pri = synth.priors_numpy(640, 640)
    loc, conf, targets = synth.multibox_inputs(3, pri, 99, 5, 30)
    rng = np.random.Generator(np.random.PCG64(11))
    one = np.array([[0.31, 0.42, 0.37, 0.55, 0]], np.float32)
    targets[0] = np.concatenate([targets[0], np.repeat(one, 100, 0), targets[0][:3]], 0)
    targets[1] = np.concatenate([targets[1], np.array([[1.5, 1.5, 1.6, 1.6, 0], [0.2, 0.2, 0.2005, 0.2005, 0], [0.1, 0.5, 0.9, 0.503, 0],
                                                        [0.5, 0.05, 0.502, 0.95, 0]], np.float32)], 0)
    sel, pos = check_fused(loc, conf, pri, targets, 1)
    r = orc.multibox_loss(loc, conf, pri, targets, 0.35, 3, True, VAR)
    assert pos.sum() > (orc.multibox_loss(loc, conf, pri, targets, 0.35, 3, False, VAR)["conf_t"] > 0).sum()    # forced matches exist


@pytest.mark.parametrize("bip", [0, 1])
def test_fused_forward_under_cuda_graph_capture(bip):
    """The forward is a chain of programmatically-dependent launches without a memset node or a host read: it can be captured into
    a CUDA graph and replayed (new logits in the same buffers between replays)."""
    from fdt_b200 import _lib
    from fdt_b200.layers.modules.multibox_loss import pack_targets
    dev = torch.device("cuda", torch.cuda.current_device())
    pri = synth.priors_numpy(320, 320)
    loc, conf, targets = synth.multibox_inputs(4, pri, 2024, 2, 40)
    loc2, conf2, _ = synth.multibox_inputs(4, pri, 2025, 2, 40)
    B, N, Cn = conf.shape
    l, c, p = cu(loc), cu(conf), cu(pri)
    gt, off, total = pack_targets([cu(t) for t in targets], dev)
    losses = torch.zeros(2, device=dev); norm = torch.zeros(1, device=dev)
    loc_t = torch.empty((B, N, 4), device=dev); conf_t = torch.empty((B, N), dtype=torch.int64, device=dev)
    sel = torch.empty((B, N), dtype=torch.uint8, device=dev)
    L = _lib.lib()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        ws = torch.empty(L.fdt_multibox_workspace_bytes(B, N, Cn, total), dtype=torch.uint8, device=dev)

        def fwd():
            _lib.check(L.fdt_multibox_loss_forward(l.data_ptr(), c.data_ptr(), p.data_ptr(), gt.data_ptr(), off.data_ptr(), total, B, N, Cn,
                                                   0.35, 3, bip, VAR[0], VAR[1], losses.data_ptr(), norm.data_ptr(), loc_t.data_ptr(),
                                                   conf_t.data_ptr(), sel.data_ptr(), None, ws.data_ptr(), ws.numel(), _lib.stream_ptr()))
        fwd()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            fwd()
    for lo_, co_ in ((loc, conf), (loc2, conf2), (loc, conf)):
        l.copy_(cu(lo_)); c.copy_(cu(co_))
        losses.zero_(); sel.zero_()
        torch.cuda.synchronize()
        g.replay()
        torch.cuda.synchronize()
        r = orc.multibox_loss(lo_, co_, pri, targets, 0.35, 3, bool(bip), VAR)
        assert np.array_equal(npy(conf_t), r["conf_t"])
        assert np.array_equal(npy(sel).astype(bool), r["neg"] | (r["conf_t"] > 0))
        np.testing.assert_allclose(npy(losses), [r["loss_l"], r["loss_c"]], rtol=1e-5)


def test_fused_forward_bipartite_large_prior_set():
    """196,000 priors (1536 x 1536, 192 super-tiles of 1,024 priors): the two-level search of k_best_prior over more than one round
    of 32 super-tiles per warp."""
    pri = synth.priors_numpy(1536, 1536)
    assert pri.shape[0] > 170_000
    loc, conf, targets = synth.multibox_inputs(1, pri, 4242, 25, 25)
    check_fused(loc, conf, pri, targets, 1)
