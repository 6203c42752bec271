"""Detect (csrc/detect.cu, k_sort_nms) at the row lengths, list counts and per-list capacities where its kernel paths switch.

Every case is a seeded generator plus a regime check that asserts, on the inputs alone (and where needed on the oracle's output),
that the case sits on the side of a kernel edge it claims.  The regime checks run without a GPU (test_case_reaches_its_edge),
so a generator that drifted off its edge fails on any machine.  The GPU test runs each case under every launch variant that can
take it -- fused forced, K2 + one CTA per list, K2 + 2-CTA cluster, the automatic policy -- and compares out, counts and
kept_prior bit for bit with the CPU oracle (orc.Detect, early_exit=True).

The kernel constants the cases aim at are named in the first block below; a rewrite that moves an edge changes that block and the
cases follow (each case brackets its edge with values computed from these constants)."""
import functools
import os

import numpy as np
import pytest
import torch

from fdt_b200 import synth
from oracle import oracle as orc
from tests.test_detect_paths_gpu import VARIANTS, c_detect, new_ws, oracle_detect, set_variant, status

# ------------------------------------------------------------------------------- kernel constants (csrc/detect.cu)
K3_THREADS = 1024                # detect.cu:40    threads of a k_sort_nms CTA: the fused first scan reads prior tid + u * 1024
SCAN_PRIORS = 36 * 1024          # detect.cu:990   U x K3_THREADS priors of the fused kernel's first scan; later priors are re-read in place
FUSED_MAX_N = 40960              # detect.cu:2089  the automatic policy fuses rows up to this length
WQ_CAP = 288                     # detect.cu:991   keys per warp queue; a warp with more first-scan candidates visits its priors in place
REG_KEYS = 8192                  # detect.cu:977   KREG x K3_THREADS keys a list may have to keep them in registers (K2 path)
BIG_BUCKET = 512                 # detect.cu:43    a larger bucket inside the top-k range -> bitonic sort of everything placed
NUM_SMS = 148                    # fdt_common.cuh:47, detect.cu:2089 (fused: lists <= 148), :1805 (cluster: 2 x lists <= 148)
NB = 2048                        # detect.cu:42    buckets of the bucket sort
MAX_NMS_TOP_K = 8000             # fdt_common.cuh (FDT_MAX_NMS_TOP_K)
KEPT_SMEM_ROWS = {3000: 2622, 5000: 1598, 8000: 1598}    # plan_smem (detect.cu:1695, :1783): most kept rows per list that stay in
#                                                          shared memory, by nms_top_k; one more and they spill to the workspace


def key_cap(nms_top_k, N):
    """Entries of the shared-memory key array (plan_smem, detect.cu:1699-1700): power of two >= min(nms_top_k, N) + 64."""
    kcap, cap = min(nms_top_k, N), 64
    while cap < kcap + 64:
        cap *= 2
    return cap


def scan_warp(i):
    """Warp of the fused kernel whose first-scan queue prior i enters (detect.cu:1012-1034); -1 past the first scan."""
    i = np.asarray(i)
    return np.where(i < SCAN_PRIORS, (i % K3_THREADS) // 32, -1)


def warp_counts(s, thr):
    """Per-warp first-scan candidate counts of one list's scores."""
    w = scan_warp(np.nonzero(s > np.float32(thr))[0])
    return np.bincount(w[w >= 0], minlength=K3_THREADS // 32)


def warp_owned(N):
    """Priors each warp loads in the first scan of a row of N priors."""
    w = scan_warp(np.arange(N))
    return np.bincount(w[w >= 0], minlength=K3_THREADS // 32)


def float_key(s):
    """fdt_float_key (fdt_common.cuh): order-preserving float -> uint32."""
    u = np.asarray(s, np.float32).view(np.uint32)
    return np.where(u & np.uint32(0x80000000), ~u, u | np.uint32(0x80000000)).astype(np.uint32)


def bucket_profile(s, thr, nms_top_k, fused):
    """First attempt of k_sort_nms's bucket sort on one list (detect.cu:1063-1121) -> (k, placed, largest bucket inside the top-k
    range).  The fused kernel maps the a-priori range (conf_thresh, 1], K2 the list's own [min, max] key range."""
    kk = float_key(s[s > np.float32(thr)]).astype(np.int64)
    k = min(kk.size, nms_top_k)
    if k <= 1:
        return k, 0, 0
    if fused:
        kmin = int(float_key(np.float32(thr))); kmax = max(int(float_key(np.float32(1.0))), kmin)
    else:
        kmin, kmax = int(kk.min()), int(kk.max())
    binv = np.float32(NB) / (np.float32(kmax - kmin) + np.float32(1.0))
    b = np.minimum(NB - 1, ((kk - kmin).astype(np.float32) * binv).astype(np.int64))
    cnt = np.bincount(b, minlength=NB)[::-1]                    # highest bucket first
    start = np.concatenate([[0], np.cumsum(cnt)[:-1]])
    live = start < k
    j = np.nonzero(live & (start + cnt >= k))[0][0]
    return k, int(start[j] + cnt[j]), int(cnt[live].max())


# ------------------------------------------------------------------------------- input builders
def unique_scores(rng, n, lo, hi):
    """n distinct float32 scores in (lo, hi), random order."""
    v = np.unique(rng.uniform(lo, hi, 2 * n + 64).astype(np.float32))
    v = v[(v > np.float32(lo)) & (v < np.float32(hi))]
    assert v.size >= n
    return rng.permutation(v)[:n]


def two_class(loc, s):
    s = np.asarray(s, np.float32)
    return loc, np.stack([np.float32(1.0) - s, s], -1).astype(np.float32)


def rand_loc(rng, B, N):
    return (rng.standard_normal((B, N, 4), dtype=np.float32) * np.float32(0.5)).astype(np.float32)


def below(rng, shape, thr):
    """Scores that are never candidates."""
    return (rng.uniform(0.0, 0.9, shape) * thr).astype(np.float32)


def spaced_level0(w, h, step):
    """Indices of every step-th level-0 prior in both directions: boxes that barely overlap, so NMS keeps nearly all of them."""
    fw, fh = synth.feature_maps(w, h)[0]
    gy, gx = np.meshgrid(np.arange(0, fh, step), np.arange(0, fw, step), indexing="ij")
    return (gy * fw + gx).ravel()


@functools.lru_cache(maxsize=None)
def priors(w, h):
    return synth.priors_numpy(w, h)


@functools.lru_cache(maxsize=None)
def synth_batch(w, h, B, seed, mode="random"):
    return synth.detect_inputs(B, priors(w, h), seed, 0.05, mode)


def lists_of(case):
    return case.B * (case.C - 1)


class Case:
    """One input set and its Detect arguments.  make() -> (loc, conf, priors); check(case) asserts the regime."""

    def __init__(self, cid, B, C, make, check, top_k=750, nms_top_k=5000, conf_t=0.05, nms_t=0.3, variants=None, depth=2):
        self.id, self.B, self.C, self.make, self.check_fn = cid, B, C, make, check
        self.top_k, self.nms_top_k, self.conf_t, self.nms_t, self.depth = top_k, nms_top_k, conf_t, nms_t, depth
        if variants is None:
            lists = B * (C - 1)
            variants = (["fused"] if lists <= NUM_SMS else []) + ["k2+single"] + (["k2+cluster"] if 2 * lists <= NUM_SMS else []) + ["auto"]
        self.variants = variants

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

    def scores(self, cls=1):
        return self.inputs[1][..., cls]

    def check(self):
        self.check_fn(self)


CASES = []


def case(*args, **kw):
    c = Case(*args, **kw)
    CASES.append(c)
    return c


# ------------------------------------------------------------------------------- A. row length
ROW_LENGTHS = [1, 2, 33, 1023, 1025, 34125, SCAN_PRIORS - 1, SCAN_PRIORS, SCAN_PRIORS + 1, SCAN_PRIORS + K3_THREADS, 40040,
               FUSED_MAX_N, FUSED_MAX_N + 1]


def make_truncated(N, mode):
    """800x600 inputs (N = 40,040; longer rows from the 704x704 set, N = 41,297) cut to N priors.  The last prior and the first
    prior past the first scan score high in every image, so every list has candidates in the tail and the output depends on them."""
    w, h = (800, 600) if N <= 40040 else (704, 704)
    loc, conf = synth_batch(w, h, 4, 3100, mode)
    loc, s, pri = loc[:, :N].copy(), conf[:, :N, 1].copy(), priors(w, h)[:N]
    assert pri.shape[0] == N
    s[:, N - 1] = np.float32(0.97) - np.float32(1e-3) * np.arange(4, dtype=np.float32)
    if N > SCAN_PRIORS:
        s[:, SCAN_PRIORS] = np.float32(0.96) - np.float32(1e-3) * np.arange(4, dtype=np.float32)
    s[0, 0] = np.float32(0.95)
    return (*two_class(loc, s), pri)


def check_row_length(c, N):
    assert c.N == N
    s = c.scores()
    tail = (s[:, SCAN_PRIORS:] > np.float32(c.conf_t)).sum(1)
    if N <= SCAN_PRIORS:
        assert tail.sum() == 0                                  # one scan holds the whole row
    else:                                                       # every list has candidates past the first scan, and they are output
        assert (tail >= 1).all()
        assert all((c.ref[2][b, 1] >= SCAN_PRIORS).any() for b in range(c.B))
    if N == 1:                                                  # one candidate per list: the list is skipped (detection.py:66-72)
        assert ((s > np.float32(c.conf_t)).sum(1) == 1).all() and (c.ref[1][:, 1] == 0).all()


for _mode in ("random", "clustered"):
    for _N in ROW_LENGTHS:
        case(f"rows-{_mode}-{_N}", 4, 2, functools.partial(make_truncated, _N, _mode), functools.partial(check_row_length, N=_N))


# frame size -> where its row falls: inside one first scan, past it but still fused by the automatic policy, past the fused limit
REAL_SIZES = {(672, 672): "in-place", (640, 720): "in-place", (768, 576): "one-scan", (704, 704): "past-fused"}


def make_real(w, h):
    loc, conf = synth_batch(w, h, 4, 3200)
    return loc, conf, priors(w, h)


def check_real(c, region):
    N = c.N
    assert region == ("one-scan" if N <= SCAN_PRIORS else "in-place" if N <= FUSED_MAX_N else "past-fused")
    tail = (c.scores()[:, SCAN_PRIORS:] > np.float32(c.conf_t)).sum(1)
    assert (tail > 0).all() if N > SCAN_PRIORS else tail.sum() == 0


for (_w, _h), _r in REAL_SIZES.items():
    case(f"real-{_w}x{_h}", 4, 2, functools.partial(make_real, _w, _h), functools.partial(check_real, region=_r))


def check_1024(c):
    assert c.N - SCAN_PRIORS > 50000 and c.N > FUSED_MAX_N
    assert ((c.scores()[:, SCAN_PRIORS:] > np.float32(c.conf_t)).sum(1) > 10000).all()


case("real-1024x1024-fused", 3, 2, lambda: (*synth_batch(1024, 1024, 3, 3300), priors(1024, 1024)), check_1024, variants=["fused"])


def make_tail_only():
    """Candidates only past the first scan: every warp queue is empty."""
    rng = np.random.Generator(np.random.PCG64(3400))
    pri = priors(800, 600); N = pri.shape[0]; B = 3
    s = below(rng, (B, N), 0.05)
    for b in range(B):
        idx = SCAN_PRIORS + rng.permutation(N - SCAN_PRIORS)[:(N - SCAN_PRIORS) // 2]
        s[b, idx] = unique_scores(rng, idx.size, 0.05, 1.0)
    return (*two_class(rand_loc(rng, B, N), s), pri)


def check_tail_only(c):
    for b in range(c.B):
        assert warp_counts(c.scores()[b], c.conf_t).sum() == 0
        assert (c.scores()[b, SCAN_PRIORS:] > np.float32(c.conf_t)).sum() > 1
    assert (c.ref[1][:, 1] > 0).all()


case("tail-only-candidates", 3, 2, make_tail_only, check_tail_only)


def make_tail_top():
    """The highest scores of every list lie past the first scan: an output that skipped the tail differs in its first row."""
    loc, conf = synth_batch(800, 600, 4, 3500)
    rng = np.random.Generator(np.random.PCG64(3501))
    s = conf[..., 1].copy()
    s[:, :SCAN_PRIORS] = np.minimum(s[:, :SCAN_PRIORS], np.float32(0.9))
    for b in range(4):
        idx = SCAN_PRIORS + rng.permutation(s.shape[1] - SCAN_PRIORS)[:200]
        s[b, idx] = unique_scores(rng, 200, 0.95, 1.0)
    return (*two_class(loc, s), priors(800, 600))


def check_tail_top(c):
    s = c.scores()
    assert (s[:, SCAN_PRIORS:].max(1) > s[:, :SCAN_PRIORS].max(1)).all()
    assert (c.ref[2][:, 1, 0] >= SCAN_PRIORS).all()


case("tail-top-scores", 4, 2, make_tail_top, check_tail_top)


TAIL_TIES_NMS_TOP_K = 1000


def make_tail_ties():
    """3,000 equal scores past the first scan straddle rank nms_top_k: the straddling bucket overflows the key array, and the
    radix-select fallback has to find the k-th key among the tied tail priors."""
    rng = np.random.Generator(np.random.PCG64(3600))
    pri = priors(800, 600); N = pri.shape[0]; B = 3
    loc, conf = synth_batch(800, 600, B, 3601)
    s = conf[..., 1].copy()
    s = np.where(s >= np.float32(0.6), s * np.float32(0.5), s).astype(np.float32)       # below the ties, out of their bucket
    for b in range(B):
        top = rng.permutation(SCAN_PRIORS)[:TAIL_TIES_NMS_TOP_K // 2]
        s[b, top] = unique_scores(rng, top.size, 0.8, 1.0)
        ties = SCAN_PRIORS + rng.permutation(N - SCAN_PRIORS)[:3000]
        s[b, ties] = np.float32(0.7)
    return (*two_class(loc, s), pri)


def check_tail_ties(c):
    for b in range(c.B):
        s = c.scores()[b]
        cand = np.nonzero(s > np.float32(c.conf_t))[0]
        order = np.lexsort((cand, s[cand]))[::-1]               # descending key (score, then prior index)
        assert cand[order[c.nms_top_k - 1]] >= SCAN_PRIORS      # the k-th key is a tail prior
        for fused in (True, False):
            k, placed, _ = bucket_profile(s, c.conf_t, c.nms_top_k, fused)
            assert placed > key_cap(c.nms_top_k, c.N)           # -> radix select over the whole row


case("tail-ties-radix-select", 3, 2, make_tail_ties, check_tail_ties, nms_top_k=TAIL_TIES_NMS_TOP_K)


def make_three_class(B, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    pri = priors(800, 600); N = pri.shape[0]
    logits = rng.standard_normal((B, N, 3), dtype=np.float32) * np.float32(2.0) + np.array([3.0, 0.0, 0.5], np.float32)
    e = np.exp(logits.astype(np.float64))
    conf = (e / e.sum(-1, keepdims=True)).astype(np.float32)
    return rand_loc(rng, B, N), conf, pri


def check_three_class(c, lists):
    assert c.C == 3 and lists_of(c) == lists and c.N == 40040
    for cls in (1, 2):                                          # candidates past the first scan in both classes: strided reads of the tail
        assert ((c.scores(cls)[:, SCAN_PRIORS:] > np.float32(c.conf_t)).sum(1) > 0).all()


case("three-class-40040", 4, 3, functools.partial(make_three_class, 4, 3700), functools.partial(check_three_class, lists=8))


# ------------------------------------------------------------------------------- B. lists per call
def check_lists(c, lists):
    assert lists_of(c) == lists and c.N == 40040
    assert (lists <= NUM_SMS) == ("fused" in c.variants)
    assert (2 * lists <= NUM_SMS) == ("k2+cluster" in c.variants)


for _B in (NUM_SMS - 1, NUM_SMS, NUM_SMS + 1):
    case(f"lists-c2-b{_B}", _B, 2,
         (lambda B: lambda: (*(a[:B] for a in synth_batch(800, 600, NUM_SMS + 1, 3800)), priors(800, 600)))(_B),
         functools.partial(check_lists, lists=_B))
for _B in (NUM_SMS // 2, NUM_SMS // 2 + 1):
    case(f"lists-c3-b{_B}", _B, 3,
         (lambda B: lambda: tuple(a[:B] if a.ndim == 3 else a for a in make_three_class(NUM_SMS // 2 + 1, 3900)))(_B),
         functools.partial(check_lists, lists=2 * _B))


def check_cluster_policy(c, cluster):
    assert c.depth == 1 and c.variants == ["k2+auto"]
    assert (2 * lists_of(c) <= NUM_SMS) == cluster              # K2 with a one-slot workspace: 2-CTA cluster iff 2 x lists <= 148


for _B in (NUM_SMS // 2, NUM_SMS // 2 + 1):
    case(f"cluster-policy-b{_B}", _B, 2,
         (lambda B: lambda: (*(a[:B] for a in synth_batch(800, 600, NUM_SMS + 1, 3800)), priors(800, 600)))(_B),
         functools.partial(check_cluster_policy, cluster=_B == NUM_SMS // 2), variants=["k2+auto"], depth=1)


# ------------------------------------------------------------------------------- C. per-list capacities
SIZES = [(640, 640), (800, 600)]


def warp_queue_plan(N):
    """Per-warp first-scan candidate counts: image 0 gets WQ_CAP - 16 + w (so WQ_CAP - 1 .. WQ_CAP + 2 appear), image 1 cycles
    through 0, 1, WQ_CAP, WQ_CAP + 1 and every prior the warp owns."""
    owned = warp_owned(N)
    w = np.arange(K3_THREADS // 32)
    img0 = WQ_CAP - 16 + w
    img1 = np.choose(w % 5, [np.zeros_like(w), np.ones_like(w), np.full_like(w, WQ_CAP), np.full_like(w, WQ_CAP + 1), owned])
    return img0, img1, owned


def make_warp_queue(w, h):
    rng = np.random.Generator(np.random.PCG64(4000 + w))
    pri = priors(w, h); N = pri.shape[0]
    s = below(rng, (2, N), 0.05)
    warp = scan_warp(np.arange(N))
    for b, plan in enumerate(warp_queue_plan(N)[:2]):
        for q, n in enumerate(plan):
            idx = rng.permutation(np.nonzero(warp == q)[0])[:n]
            s[b, idx] = unique_scores(rng, n, 0.05, 1.0) if n else s[b, idx]
        tail = np.nonzero(warp < 0)[0]
        idx = tail[rng.uniform(size=tail.size) < 0.2]
        s[b, idx] = unique_scores(rng, idx.size, 0.05, 1.0) if idx.size else s[b, idx]
    return (*two_class(rand_loc(rng, 2, N), s), pri)


def check_warp_queue(c):
    img0, img1, owned = warp_queue_plan(c.N)
    got0, got1 = warp_counts(c.scores()[0], c.conf_t), warp_counts(c.scores()[1], c.conf_t)
    assert np.array_equal(got0, img0) and np.array_equal(got1, img1)
    assert {WQ_CAP - 1, WQ_CAP, WQ_CAP + 1, WQ_CAP + 2} <= set(got0.tolist())
    assert {0, 1, WQ_CAP, WQ_CAP + 1} <= set(got1.tolist())
    full = got1 == owned
    assert full.any() and (owned[full] > WQ_CAP).all()          # warps whose every prior is a candidate


for _w, _h in SIZES:
    case(f"warp-queue-{_w}x{_h}", 2, 2, functools.partial(make_warp_queue, _w, _h), check_warp_queue)


def make_exact_candidates(w, h, n, seed, hi=1.0):
    """Exactly n candidates per list, unique scores, at random priors."""
    rng = np.random.Generator(np.random.PCG64(seed))
    pri = priors(w, h); N = pri.shape[0]
    s = below(rng, (2, N), 0.05)
    for b in range(2):
        s[b, rng.permutation(N)[:n]] = unique_scores(rng, n, 0.05, hi)
    return (*two_class(rand_loc(rng, 2, N), s), pri)


def check_exact_candidates(c, n):
    s = c.scores()
    cand = s > np.float32(c.conf_t)
    assert (cand.sum(1) == n).all()
    assert all(np.unique(s[b][cand[b]]).size == n for b in range(c.B))


for _w, _h in SIZES:
    for _n in (REG_KEYS - 1, REG_KEYS, REG_KEYS + 1):
        case(f"reg-keys-{_n}-{_w}x{_h}", 2, 2, functools.partial(make_exact_candidates, _w, _h, _n, 4100 + _n),
             functools.partial(check_exact_candidates, n=_n))


def make_big_bucket(w, h, ties):
    """`ties` equal scores at the top of every list, 6,000 unique scores far below them."""
    rng = np.random.Generator(np.random.PCG64(4200 + ties))
    pri = priors(w, h); N = pri.shape[0]
    s = below(rng, (2, N), 0.05)
    for b in range(2):
        idx = rng.permutation(N)
        s[b, idx[:ties]] = np.float32(0.9)
        s[b, idx[ties:ties + 6000]] = unique_scores(rng, 6000, 0.05, 0.5)
    return (*two_class(rand_loc(rng, 2, N), s), pri)


def check_big_bucket(c, ties):
    for b in range(c.B):
        assert (c.scores()[b] == np.float32(0.9)).sum() == ties
        for fused in (True, False):
            k, placed, biggest = bucket_profile(c.scores()[b], c.conf_t, c.nms_top_k, fused)
            assert biggest == ties and placed <= key_cap(c.nms_top_k, c.N)     # reached without the radix-select fallback


for _w, _h in SIZES:
    for _t in (BIG_BUCKET, BIG_BUCKET + 1):
        case(f"big-bucket-{_t}-{_w}x{_h}", 2, 2, functools.partial(make_big_bucket, _w, _h, _t), functools.partial(check_big_bucket, ties=_t))


def make_keepers(w, h, seed):
    """Spaced level-0 priors (every third in both directions) score high and barely overlap, so NMS keeps thousands of boxes;
    10 % of the other priors are lower candidates."""
    rng = np.random.Generator(np.random.PCG64(seed))
    pri = priors(w, h); N = pri.shape[0]
    keep = spaced_level0(w, h, 3)
    loc = rand_loc(rng, 2, N)
    loc[:, keep] *= np.float32(0.3)
    s = below(rng, (2, N), 0.05)
    rest = np.setdiff1d(np.arange(N), keep)
    for b in range(2):
        s[b, keep] = unique_scores(rng, keep.size, 0.5, 1.0)
        low = rest[rng.uniform(size=rest.size) < 0.1]
        s[b, low] = unique_scores(rng, low.size, 0.05, 0.5)
    return (*two_class(loc, s), pri)


def check_keepers(c):
    edge = KEPT_SMEM_ROWS[c.nms_top_k]
    assert edge - 1 <= c.top_k <= edge + 2                      # within two rows of the shared-memory / workspace edge
    assert (c.ref[1][:, 1] == c.top_k).any()                    # a list really fills all top_k kept rows


for _w, _h in SIZES:
    for _ntk in (5000, 3000):
        _edge = KEPT_SMEM_ROWS[_ntk]
        for _tk in ((_edge - 1, _edge, _edge + 1, _edge + 2) if _ntk == 5000 else (_edge - 1, _edge, _edge + 1)):
            case(f"kept-rows-{_tk}-ntk{_ntk}-{_w}x{_h}", 2, 2, functools.partial(make_keepers, _w, _h, 4300 + _w), check_keepers,
                 top_k=_tk, nms_top_k=_ntk)


def check_max_nms_top_k(c):
    assert c.nms_top_k == MAX_NMS_TOP_K
    assert ((c.scores() > np.float32(c.conf_t)).sum(1) >= MAX_NMS_TOP_K).all()


for _w, _h in SIZES:
    case(f"nms-top-k-max-{_w}x{_h}", 2, 2, functools.partial(make_exact_candidates, _w, _h, 9000, 4400 + _w), check_max_nms_top_k,
         nms_top_k=MAX_NMS_TOP_K)


# ------------------------------------------------------------------------------- D. the strict threshold
def make_strict(thr):
    """Scores exactly float32(conf_thresh) (never candidates) and one ulp above it (always candidates), each in the first scan and
    past it, at priors that barely overlap; 300 higher candidates elsewhere."""
    rng = np.random.Generator(np.random.PCG64(int(thr * 1000) + 4500))
    pri = priors(800, 600); N = pri.shape[0]
    t = np.float32(thr); up = np.nextafter(t, np.float32(1.0))
    fw2, fh2 = synth.feature_maps(800, 600)[2]
    lvl2 = sum(a * b for a, b in synth.feature_maps(800, 600)[:2])
    gy, gx = np.meshgrid(np.arange(0, fh2, 3), np.arange(0, fw2, 3), indexing="ij")
    tail = lvl2 + (gy * fw2 + gx).ravel()                       # level 2 (stride 16): past the first scan at 800 x 600
    head = spaced_level0(800, 600, 4)
    s = below(rng, (2, N), t)
    for b in range(2):
        h, tl = rng.permutation(head), rng.permutation(tail)
        s[b, h[:150]] = up; s[b, h[150:300]] = t
        s[b, tl[:40]] = up; s[b, tl[40:80]] = t
        hi = np.setdiff1d(rng.permutation(N)[:400], np.concatenate([h[:300], tl[:80]]))[:300]
        s[b, hi] = unique_scores(rng, hi.size, 0.5, 1.0)
    return (*two_class(rand_loc(rng, 2, N), s), pri)


def check_strict(c):
    t = np.float32(c.conf_t); up = np.nextafter(t, np.float32(1.0))
    s = c.scores()
    for b in range(c.B):
        for part in (slice(0, SCAN_PRIORS), slice(SCAN_PRIORS, None)):
            assert (s[b, part] == t).sum() >= 40 and (s[b, part] == up).sum() >= 40
        kept = c.ref[2][b, 1][:c.ref[1][b, 1]]
        at_up = kept[s[b, kept] == up]
        assert (at_up < SCAN_PRIORS).any() and (at_up >= SCAN_PRIORS).any()         # one-ulp candidates are output in both parts
    loc, conf, pri = c.inputs
    loose = oracle_detect(loc, conf, pri, (2, 0, c.top_k, float(np.nextafter(t, np.float32(0.0))), c.nms_t))
    assert not np.array_equal(loose[0], c.ref[0])               # a `>=` threshold would change the output


STRICT = {thr: case(f"strict-threshold-{thr}", 2, 2, functools.partial(make_strict, thr), check_strict, conf_t=thr) for thr in (0.05, 0.3)}


# ------------------------------------------------------------------------------- runner
ALL_VARIANTS = dict(VARIANTS, **{"auto": (-1, -1), "k2+auto": (0, -1)})       # (detect_fused, k3_cluster)
_OPTION_DEFAULTS = (("detect_fused", "FDT_DETECT_FUSED", -1), ("k3_cluster", "FDT_K3_CLUSTER", -1),
                    ("detect_depth", "FDT_DETECT_DEPTH", 4), ("host_chunk", "FDT_HOST_CHUNK", 16))
GUARD = -7.0


@pytest.fixture()
def lib():
    """The library; every option a case sets is back at its process default (environment or built-in) afterwards."""
    from fdt_b200 import _lib
    yield _lib
    for name, env, dflt in _OPTION_DEFAULTS:
        e = os.environ.get(env)
        _lib.set_option(name, int(e) if e else dflt)


def use_variant(lib, variant):
    if variant in VARIANTS:
        set_variant(lib, variant)
    else:
        fused, cluster = ALL_VARIANTS[variant]
        lib.set_option("detect_fused", fused)
        lib.set_option("k3_cluster", cluster)


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def run_case(lib, c, variant, nms_top_k=None):
    """One fdt_detect call of case c; the output sits inside a guard band that must stay untouched."""
    loc, conf, pri = c.inputs
    use_variant(lib, variant)
    B, N, C = conf.shape
    ws = new_ws(lib, B, N, C, c.depth)
    n = B * C * c.top_k * 5
    buf = torch.full((n + 8,), GUARD, device="cuda")
    out = buf[4:4 + n].view(B, C, c.top_k, 5)
    counts = torch.full((B, C), -5, dtype=torch.int32, device="cuda")
    kept = torch.full((B, C, c.top_k), -5, dtype=torch.int64, device="cuda")
    c_detect(lib, cu(loc), cu(conf), cu(pri), ws, out, counts, kept, top_k=c.top_k, nms_top_k=nms_top_k or c.nms_top_k,
             conf_t=c.conf_t, nms_t=c.nms_t)
    torch.cuda.synchronize()
    assert status(lib, ws) == 0
    g = buf.cpu().numpy()
    assert np.all(g[:4] == GUARD) and np.all(g[4 + n:] == GUARD), f"{variant}: write outside the output"
    return out, counts, kept


@pytest.mark.parametrize("c", CASES, ids=lambda c: c.id)
def test_case_reaches_its_edge(c):
    """CPU: each generator reaches the kernel edge its case is named for."""
    c.check()


@pytest.mark.gpu
@pytest.mark.parametrize("c,variant", [(c, v) for c in CASES for v in c.variants], ids=lambda x: x.id if isinstance(x, Case) else x)
def test_detect_edge_case(lib, c, variant):
    c.check()
    got = run_case(lib, c, variant)
    for g, w, name in zip(got, c.ref, ("out", "counts", "kept_prior")):
        assert np.array_equal(g.cpu().numpy(), w), f"{name} differs ({c.id}, {variant})"


@pytest.mark.gpu
def test_nms_top_k_past_the_limit_is_refused(lib):
    c = CASES[[x.id for x in CASES].index("nms-top-k-max-800x600")]
    for variant in ("fused", "k2+single"):
        with pytest.raises(NotImplementedError, match="nms_top_k"):
            run_case(lib, c, variant, nms_top_k=MAX_NMS_TOP_K + 1)


@pytest.mark.gpu
@pytest.mark.parametrize("thr", list(STRICT))
def test_strict_threshold_candidate_counts(lib, thr):
    """Stage 1 alone counts exactly the scores > float32(conf_thresh): none at the threshold, all one ulp above it."""
    c = STRICT[thr]
    loc, conf, pri = c.inputs
    B, N, C = conf.shape
    L = lib.lib()
    ws = torch.empty(L.fdt_detect_workspace_bytes(B, N, C), dtype=torch.uint8, device="cuda")
    st = lib.stream_ptr()
    lib.check(L.fdt_detect_threshold_compact(cu(conf).data_ptr(), B, N, C, thr, ws.data_ptr(), ws.numel(), st))
    cnt = torch.empty(B, dtype=torch.int32, device="cuda")
    lib.check(L.fdt_detect_candidate_counts(ws.data_ptr(), ws.numel(), B, N, C, cnt.data_ptr(), st))
    assert np.array_equal(cnt.cpu().numpy(), (conf[..., 1] > np.float32(thr)).sum(1).astype(np.int32))


# ------------------------------------------------------------------------------- E. the other entry points at 800 x 600
HOST_B, HOST_CHUNK = 20, 16


@functools.lru_cache(maxsize=None)
def host_inputs():
    return synth_batch(800, 600, HOST_B, 4600)


@functools.lru_cache(maxsize=None)
def heads_inputs():
    loc_maps, conf_maps, neg_max = synth.head_maps(2, 800, 600, 4700)
    return loc_maps, conf_maps, neg_max, priors(800, 600)


def test_other_entry_points_reach_their_edges():
    """CPU: the host batch leaves a remainder chunk; the 800 x 600 head maps have ceil'd coarse levels and one map position per prior."""
    assert HOST_B > HOST_CHUNK and HOST_B % HOST_CHUNK == 4
    loc_maps, conf_maps, _, pri = heads_inputs()
    assert [m.shape[2:] for m in conf_maps][4:] == [(10, 13), (5, 7)]          # [H, W]: 600/64, 800/64, 600/128, 800/128 rounded up
    assert sum(m.shape[2] * m.shape[3] for m in conf_maps) == pri.shape[0] == 40040


@pytest.mark.gpu
@pytest.mark.parametrize("pin", [True, False], ids=["pinned", "pageable"])
def test_host_buffers_chunk_and_remainder(lib, pin):
    """fdt_detect_host with B = 20 and 16-image chunks: one chunk of 16 and a remainder of 4."""
    import fdt_b200.layers as layers
    lib.set_option("host_chunk", HOST_CHUNK)
    loc, conf = host_inputs()
    pri = priors(800, 600)
    t = [torch.from_numpy(np.ascontiguousarray(a)) for a in (loc, conf, pri)]
    if pin:
        t = [x.pin_memory() for x in t]
    got = layers.Detect(2, 0, 750, 0.05, 0.3)(*t, return_aux=True)
    for g, w, name in zip(got, oracle_detect(loc, conf, pri), ("out", "counts", "kept_prior")):
        assert g.device.type == "cpu" and np.array_equal(g.numpy(), w), name


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["k2+single", "k2+cluster", "auto"])
def test_head_maps_with_ceiled_levels(lib, variant):
    """Detect.detect_heads at 800 x 600 (coarse maps 13 x 10 and 7 x 5) equals the oracle on the materialised tensors."""
    from fdt_b200.layers import Detect
    use_variant(lib, variant)
    loc_maps, conf_maps, neg_max, pri = heads_inputs()
    got = Detect(2, 0, 750, 0.05, 0.3).detect_heads([cu(m) for m in loc_maps], [cu(m) for m in conf_maps], cu(pri), neg_max,
                                                     return_aux=True)
    rl, rc = orc.heads_to_loc_conf(loc_maps, conf_maps, neg_max, softmax=True)
    for g, w, name in zip(got, oracle_detect(rl, rc, pri), ("out", "counts", "kept_prior")):
        assert np.array_equal(g.cpu().numpy(), w), name
