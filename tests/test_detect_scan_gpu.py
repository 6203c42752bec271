"""Detect's fused first row scan (csrc/detect.cu, k_sort_nms<MODE_DETECT, 1, true>, stage 1) at the edges of its compaction.

The scan loads the first 36 x 1024 priors of a row in 4 groups of 9 x 1024 (prior i is loaded by thread i % 1024); a group that lies
wholly inside the row is loaded without a per-prior bound check.  Each warp compacts its candidates into its queue, and the key of a
candidate is built with the short form `bits | sign bit` when conf_thresh >= 0 (every candidate is then a positive float) and with the
general order-preserving map otherwise.  The cases below sit on those edges: rows that end one prior before, at and one prior after
each group boundary and past the first scan, the three threshold signs with the special floats around them, and C = 3 for the
strided loads.  Every case has a regime check that runs without a GPU; the GPU test runs it fused-forced and under the automatic
policy (which fuses all of them) and compares out, counts and kept_prior bit for bit with the CPU oracle (orc.Detect,
early_exit=True)."""
import functools

import numpy as np
import pytest

from tests.test_detect_paths_gpu import c_detect, new_ws, oracle_detect, set_variant, status
from tests.test_detect_edges_gpu import (FUSED_MAX_N, K3_THREADS, NUM_SMS, SCAN_PRIORS, WQ_CAP, cu, priors, rand_loc,
                                         synth_batch, two_class, unique_scores, warp_counts)

GROUP = 9 * K3_THREADS               # priors of one load group of the first scan (4 groups of 9 loads per thread)
GROUP_BOUNDS = [GROUP * g for g in range(1, 5)]      # the last one is the end of the first scan
assert GROUP_BOUNDS[-1] == SCAN_PRIORS

# special floats of the key transform: the two zeros, the smallest denormals, the largest denormal, NaNs of both signs, infinities
DENORM_MIN = np.array(1, np.uint32).view(np.float32)
DENORM_MAX = np.array(0x007fffff, np.uint32).view(np.float32)
NEG_NAN = np.array(0xffc00000, np.uint32).view(np.float32)
SPECIALS = np.array([-0.0, 0.0, DENORM_MIN, -DENORM_MIN, DENORM_MAX, -DENORM_MAX, np.nan, NEG_NAN, np.inf, -np.inf,
                     1.5, 1.0, -0.25, -1.0], np.float32)


class Case:
    def __init__(self, cid, B, C, make, check, conf_t=0.05, top_k=750, nms_top_k=5000, nms_t=0.3):
        self.id, self.B, self.C, self.make, self.check_fn = cid, B, C, make, check
        self.conf_t, self.top_k, self.nms_top_k, self.nms_t = conf_t, top_k, nms_top_k, nms_t

    @functools.cached_property
    def inputs(self):
        loc, conf, pri = self.make()
        assert conf.shape == (self.B, pri.shape[0], self.C) and loc.shape == (self.B, pri.shape[0], 4)
        return loc, conf, pri

    @functools.cached_property
    def ref(self):
        loc, conf, pri = self.inputs
        return oracle_detect(loc, conf, pri, (self.C, 0, self.top_k, self.conf_t, self.nms_t), nms_top_k=self.nms_top_k)

    @property
    def N(self):
        return self.inputs[2].shape[0]

    def check(self):
        lists = self.B * (self.C - 1)
        assert lists <= NUM_SMS and self.N <= FUSED_MAX_N            # the automatic policy takes the fused kernel
        self.check_fn(self)


CASES = []


def case(*args, **kw):
    CASES.append(Case(*args, **kw))


# ------------------------------------------------------------------------------- A. row length at the load-group boundaries
ROW_LENGTHS = sorted({b + d for b in GROUP_BOUNDS for d in (-1, 0, 1)} | {SCAN_PRIORS + K3_THREADS, 38000, FUSED_MAX_N})


def make_row(N, C=2):
    """800 x 600 inputs (N = 40,040; longer rows from the 704 x 704 set) cut to N priors.  The last prior of the row and the first
    prior of every group it reaches score highest, so each of them is a candidate and kept first in its list."""
    w, h = (800, 600) if N <= 40040 else (704, 704)
    loc, conf = synth_batch(w, h, 3, 5100 + N % 97)
    loc, s, pri = loc[:, :N].copy(), conf[:, :N, 1].copy(), priors(w, h)[:N]
    top = [N - 1] + [g for g in [0] + GROUP_BOUNDS if g < N - 1]
    for r, i in enumerate(top):
        s[:, i] = np.float32(0.999) - np.float32(1e-3) * np.float32(r) - np.float32(1e-4) * np.arange(3, dtype=np.float32)
    loc, conf = two_class(loc, s)
    if C == 3:         # the second foreground class: the same scores one prior further on (wrapping), other boxes per image
        conf = np.concatenate([conf, np.roll(conf[..., 1:], 1, axis=1)], -1)
        conf[..., 0] = np.float32(0.0)
    return loc, conf, pri


def check_row(c, N):
    assert c.N == N
    assert any(N - b in (-1, 0, 1) for b in GROUP_BOUNDS) or N > SCAN_PRIORS
    s = c.inputs[1][..., 1]
    assert (s[:, N - 1] > np.float32(c.conf_t)).all()
    assert (c.ref[2][:, 1, 0] == N - 1).all()                    # the row's last prior is read and ranked first
    if N > SCAN_PRIORS:
        assert (s[:, SCAN_PRIORS:] > np.float32(c.conf_t)).sum(1).min() >= 1      # candidates past the first scan (visited in place)


for _N in ROW_LENGTHS:
    case(f"rows-{_N}", 3, 2, functools.partial(make_row, _N), functools.partial(check_row, N=_N))
for _N in (GROUP + 1, 2 * GROUP - 1, 3 * GROUP, SCAN_PRIORS + 1):
    case(f"rows-c3-{_N}", 3, 3, functools.partial(make_row, _N, 3), functools.partial(check_row, N=_N))


# ------------------------------------------------------------------------------- B. the sign of conf_thresh and the key transform
THRESHOLDS = {"neg": -0.5, "zero": 0.0, "pos": 0.05}


def signed_zero_safe(v, thr):
    """With a negative threshold both zeros would be candidates of one list.  The kernels' order-preserving key puts -0.0 below
    +0.0, the reference's sort ties them (and breaks the tie by prior index), so such a list is left out: +0.0 becomes -0.0."""
    v = np.asarray(v, np.float32).copy()
    if thr < 0:
        v[(v == 0) & ~np.signbit(v)] = np.float32(-0.0)
    return v


def make_signs(thr, N, C=2):
    """Most scores are not candidates (below the threshold, -inf or NaN); a few hundred per image are, spread over every group and
    past the first scan, among them the special floats that pass this threshold.  Each warp stays inside its queue."""
    rng = np.random.Generator(np.random.PCG64(5200 + N + int(thr * 100)))
    B = 2
    w, h = (800, 600) if N <= 40040 else (704, 704)
    pri = priors(w, h)[:N]
    t = np.float32(thr)
    s = (t - np.float32(1e-3) - rng.uniform(0.0, 0.5, (B, N)).astype(np.float32)).astype(np.float32)
    junk = rng.uniform(size=(B, N))
    s[junk < 0.02] = -np.inf
    s[(junk >= 0.02) & (junk < 0.04)] = np.nan
    s[(junk >= 0.04) & (junk < 0.05)] = NEG_NAN
    special = signed_zero_safe(SPECIALS, thr)
    for b in range(B):
        idx = rng.choice(N, 600, replace=False)
        s[b, idx] = signed_zero_safe(unique_scores(rng, 600, float(t), float(t) + 1.0), thr)
        sp = rng.choice(np.setdiff1d(np.arange(N), idx), special.size * 4, replace=False)
        s[b, sp] = np.tile(special, 4)
    loc, conf = two_class(rand_loc(rng, B, N), s)
    if C == 3:
        conf = np.concatenate([conf, np.roll(conf[..., 1:], 7, axis=1)], -1)
    return loc, conf, pri


def check_signs(c, thr):
    s = c.inputs[1][..., 1]
    t = np.float32(thr)
    cand = s > t
    assert (warp_counts(s[0], thr) <= WQ_CAP).all() and (warp_counts(s[1], thr) <= WQ_CAP).all()     # queues hold every candidate
    assert cand[:, :SCAN_PRIORS].sum(1).min() >= 200
    specials = [v for v in signed_zero_safe(SPECIALS, thr) if v > t]
    assert all(np.isin(np.float32(v), s[b][cand[b]]) for v in specials for b in range(c.B))
    if thr < 0:     # the general key transform orders negative candidates, -0.0 and the denormals (no list holds both zeros)
        assert all((s[b][cand[b]] < 0).any() and (np.signbit(s[b][cand[b]]) & (s[b][cand[b]] == 0)).any() for b in range(c.B))
        assert not (cand & (s == 0) & ~np.signbit(s)).any()
    elif thr == 0:  # strict: neither zero is a candidate, the smallest denormal is
        assert not (cand & (s == 0)).any() and (s[cand] == DENORM_MIN).any()
    kept = c.ref[2][:, 1]
    assert (c.ref[1][:, 1] > 1).all()
    if thr <= 0:    # a candidate a positive threshold would never see is output
        assert any(((s[b][kept[b][kept[b] >= 0]]) <= np.float32(0.05)).any() for b in range(c.B))


for _name, _thr in THRESHOLDS.items():
    for _N in (34125, 2 * GROUP + 1, FUSED_MAX_N):
        case(f"signs-{_name}-{_N}", 2, 2, functools.partial(make_signs, _thr, _N), functools.partial(check_signs, thr=_thr), conf_t=_thr)
    case(f"signs-{_name}-c3", 2, 3, functools.partial(make_signs, _thr, 34125, 3), functools.partial(check_signs, thr=_thr), conf_t=_thr)


# ------------------------------------------------------------------------------- runner
@pytest.fixture()
def lib():
    from fdt_b200 import _lib
    yield _lib
    _lib.set_option("k3_cluster", -1)
    _lib.set_option("detect_fused", -1)


@pytest.mark.parametrize("c", CASES, ids=lambda c: c.id)
def test_case_reaches_its_edge(c):
    """CPU: each generator reaches the scan edge its case is named for."""
    c.check()


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["fused", "auto"])
@pytest.mark.parametrize("c", CASES, ids=lambda c: c.id)
def test_fused_scan_case(lib, c, variant):
    import torch
    c.check()
    if variant == "auto":
        lib.set_option("detect_fused", -1); lib.set_option("k3_cluster", -1)
    else:
        set_variant(lib, variant)
    loc, conf, pri = c.inputs
    B, N, C = conf.shape
    ws = new_ws(lib, B, N, C, 2)
    out = torch.full((B, C, c.top_k, 5), -7.0, device="cuda")
    counts = torch.full((B, C), -5, dtype=torch.int32, device="cuda")
    kept = torch.full((B, C, c.top_k), -5, dtype=torch.int64, device="cuda")
    c_detect(lib, cu(loc), cu(conf), cu(pri), ws, out, counts, kept, top_k=c.top_k, nms_top_k=c.nms_top_k, conf_t=c.conf_t, nms_t=c.nms_t)
    torch.cuda.synchronize()
    assert status(lib, ws) == 0
    for g, w, name in zip((out, counts, kept), c.ref, ("out", "counts", "kept_prior")):
        assert np.array_equal(g.cpu().numpy(), w), f"{name} differs ({c.id}, {variant})"
