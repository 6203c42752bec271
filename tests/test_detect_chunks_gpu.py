"""GPU parity tests for the chunked key selection of the fused Detect kernel (k_sort_nms<MODE_DETECT, 1, true, HT>).  The fused kernel
selects and scatters the best min(candidates, nms_top_k) keys of a list in chunks of two first NMS windows (2 x min(1024, max(576,
1.2 x max_keep + 16)) keys: 1,832 at max_keep 750, 1,152 at max_keep <= 466); when the windows have consumed a chunk without reaching
max_keep, the next chunk is selected among the keys below the last one processed by re-scanning the row.  Every case runs the same
inputs through the fused kernel and through the two-kernel path (K2 + k_sort_nms, which selects all keys at once); the two results must
be equal bit for bit and equal to the CPU oracle.  nms_thresh 0.02 keeps few boxes per window, so the windows run through every
candidate up to nms_top_k and take several chunks."""
import numpy as np
import pytest
import torch

from fdt_b200 import synth
from fdt_b200.layers import Detect
from oracle import oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture()
def lib():
    from fdt_b200 import _lib
    yield _lib
    _lib.set_option("detect_fused", -1)


def run_both(lib, loc, conf, pri, top_k=750, nms_top_k=5000, conf_t=0.05, nms_t=0.3, dtype=None):
    """(fused output, two-kernel output, oracle output) of the same call."""
    C_ = conf.shape[2]
    lt, ct = torch.from_numpy(loc).cuda(), torch.from_numpy(conf).cuda()
    if dtype is not None:
        lt, ct = lt.to(dtype), ct.to(dtype)
        loc, conf = lt.float().cpu().numpy(), ct.float().cpu().numpy()
    pt = torch.from_numpy(pri).cuda()
    outs = []
    for fused in (1, 0):
        lib.set_option("detect_fused", fused)
        det = Detect(C_, 0, top_k, conf_t, nms_t)
        det.nms_top_k = nms_top_k
        res = []
        for _ in range(3):                       # back to back: the calls overlap on the device
            res.append(det(lt, ct, pt))
        torch.cuda.synchronize()
        for r in res[1:]:
            assert torch.equal(r, res[0])
        outs.append(res[0].cpu().numpy())
    det = orc.Detect(C_, 0, top_k, conf_t, nms_t)
    det.nms_top_k = nms_top_k
    det.early_exit = True                        # (the oracle stops its NMS at top_k kept boxes, as the kernels do)
    ref = det(loc, conf, pri)
    return outs[0], outs[1], ref


def check(lib, *args, **kw):
    fused, k2, ref = run_both(lib, *args, **kw)
    assert np.array_equal(fused.view(np.uint32), k2.view(np.uint32)), "chunked fused kernel differs from the two-kernel path"
    assert np.array_equal(fused, ref, equal_nan=True), "fused Detect differs from the oracle"
    return ref


def inputs(B, w, h, seed, mode="random", conf_t=0.05):
    pri = synth.priors_numpy(w, h)
    loc, conf = synth.detect_inputs(B, pri, seed=seed, conf_thresh=conf_t, mode=mode)
    return loc, conf, pri


@pytest.mark.parametrize("mode", ["random", "clustered"])
def test_chunks_headline_640(lib, mode):
    loc, conf, pri = inputs(8, 640, 640, seed=11, mode=mode)
    ref = check(lib, loc, conf, pri)
    assert (ref[:, 1, :, 0] > 0).sum() > 0


def test_chunks_every_prior_a_candidate(lib):
    # 34,125 candidates per row: every warp queue overflows, every pass visits the row in place
    loc, conf, pri = inputs(2, 640, 640, seed=12)
    conf = conf.copy()
    rng = np.random.default_rng(5)
    conf[:, :, 1] = rng.uniform(0.06, 1.0, size=conf.shape[:2]).astype(np.float32)
    conf[:, :, 0] = 1.0 - conf[:, :, 1]
    check(lib, loc, conf, pri)
    check(lib, loc, conf, pri, nms_t=0.02)


@pytest.mark.parametrize("nms_top_k", [200, 1832, 1833, 3664, 3665, 8000])
@pytest.mark.parametrize("nms_t", [0.3, 0.02])
def test_chunks_nms_top_k(lib, nms_top_k, nms_t):
    # max_keep 750: chunks of 1,832 keys -> one, two, three and five chunks
    loc, conf, pri = inputs(3, 640, 640, seed=13)
    check(lib, loc, conf, pri, nms_top_k=nms_top_k, nms_t=nms_t)


@pytest.mark.parametrize("top_k", [1, 40, 466, 467, 853, 2000, 5000])
def test_chunks_max_keep(lib, top_k):
    # chunk sizes 1,152 (max_keep <= 466), 1,178 .. 2,046 and 2,048 (max_keep >= 853)
    loc, conf, pri = inputs(2, 640, 640, seed=14)
    check(lib, loc, conf, pri, top_k=top_k)
    check(lib, loc, conf, pri, top_k=top_k, nms_t=0.02)


@pytest.mark.parametrize("B", [1, 74])
def test_chunks_list_counts(lib, B):
    loc, conf, pri = inputs(B, 320, 320, seed=15)
    check(lib, loc, conf, pri, nms_t=0.02)


def test_chunks_longest_fused_row(lib):
    # N = 40,960 (the fused path's limit): priors past the queued scan of 36 x 1,024 are visited in place in every chunk
    rng = np.random.default_rng(16)
    N = 40960
    xy = rng.uniform(0.0, 1.0, size=(N, 2)).astype(np.float32)
    wh = rng.uniform(0.01, 0.3, size=(N, 2)).astype(np.float32)
    pri = np.concatenate([xy, wh], axis=1)
    loc = (rng.standard_normal((2, N, 4)) * 0.5).astype(np.float32)
    s = rng.uniform(0.0, 0.3, size=(2, N)).astype(np.float32)
    conf = np.stack([1.0 - s, s], axis=2).astype(np.float32)
    check(lib, loc, conf, pri)
    check(lib, loc, conf, pri, nms_t=0.02, nms_top_k=8000)


@pytest.mark.parametrize("levels", [2, 40, 4000])
def test_chunks_score_ties(lib, levels):
    # scores rounded to a few levels: buckets far larger than a window (bitonic fallback) and straddling buckets larger than the key
    # array (radix select), in the first chunk and in later ones
    loc, conf, pri = inputs(2, 640, 640, seed=17)
    conf = conf.copy()
    s = np.round(conf[:, :, 1] * levels) / levels
    conf[:, :, 1] = s.astype(np.float32)
    conf[:, :, 0] = (1.0 - s).astype(np.float32)
    check(lib, loc, conf, pri)
    check(lib, loc, conf, pri, nms_t=0.02)


def test_chunks_nonfinite_boxes(lib):
    loc, conf, pri = inputs(2, 640, 640, seed=18)
    loc = loc.copy()
    rng = np.random.default_rng(19)
    for v in (np.nan, np.inf, -np.inf):
        idx = rng.integers(0, loc.shape[1], size=200)
        loc[:, idx, rng.integers(0, 4)] = v
    check(lib, loc, conf, pri)
    check(lib, loc, conf, pri, nms_t=0.02)


@pytest.mark.parametrize("conf_t", [0.0, -1.0])
def test_chunks_conf_thresh_not_positive(lib, conf_t):
    # conf_thresh < 0 takes the general key map of the row scan; every prior is a candidate
    loc, conf, pri = inputs(2, 320, 320, seed=20)
    check(lib, loc, conf, pri, conf_t=conf_t, nms_t=0.02)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_chunks_16bit_inputs(lib, dtype):
    loc, conf, pri = inputs(4, 640, 640, seed=21)
    check(lib, loc, conf, pri, nms_t=0.02)
    check(lib, loc, conf, pri, dtype=dtype, nms_t=0.02)
