"""The IoU tracker (csrc/tracker.cu: k_track_mask, k_track_resolve, k_track_step) at the frame sizes, frame counts and candidate
depths where its kernel paths switch.

Every case is a seeded generator plus a regime check that asserts, on the inputs alone, that the case sits on the side of a kernel
edge it claims.  Where the edge is behavioural (refusal depth, drops, ties, thresholds) the check runs `mirror`, a small numpy
restatement of the association order that records, per frame and active track, its ranked candidate list and the rank of the
candidate it finally gets; the mirror's tracks_finished must equal the C oracle's, so the mirror is itself checked.  The regime
checks run without a GPU (test_case_reaches_its_edge).  On the GPU every case runs offline (tracker.iou_track, FDT_TRACK_FORCE_SLOW
0 and 1) and online (StreamTracker through run_streams / check_video), and must be bit-identical to the C oracle.

The kernel constants the cases aim at are named in the first block below; each case brackets its edge with values computed from
them."""
import math
from fractions import Fraction

import numpy as np
import pytest

from fdt_b200 import _lib
from oracle import oracle as orc

# ------------------------------------------------------------------------------- kernel constants (csrc/tracker.cu)
TR_THREADS = 1024                # tracker.cu:30   one thread per track / detection of a frame
OFF_CHUNK = 512                  # tracker.cu:31   frame offsets staged per chunk; reloaded at f = 512, 1023, 1534, ...
ROW_EXTRA = 4                    # tracker.cu:78   NaN flag, 4 best candidates (uint16), candidate count; re-rank after 4 refusals
SMEM_LIMIT = 232448 - 1024       # fdt_common.cuh:48 FDT_SMEM_MAX - 1024 = tracker.cu:89 TR_SMEM_LIMIT


def resolve_smem(W, prefetch):
    """tracker.cu:81-88 (resolve_smem): dynamic shared memory of k_track_resolve / k_track_step for cap = 32 * W rows."""
    cap = 32 * W
    s = ((2 if prefetch else 1) * cap * (W + ROW_EXTRA) * 4 + 15) // 16 * 16
    s += 8 * ((3 if prefetch else 2) * cap * 5 + 2 * cap)
    return s + 4 * 10 * cap


def _max_w(prefetch):
    W = 1
    while resolve_smem(W + 1, prefetch) <= SMEM_LIMIT:
        W += 1
    return W


PREFETCH_MAX_ROWS = 32 * _max_w(1)   # tracker.cu:823  frame f+1 staged with cp.async while frame f is resolved (608)
MAX_ROWS = 32 * _max_w(0)            # tracker.cu:98   TR_MAX_D: the most rows per frame, offline and online (864)
W_PF, W_MAX = PREFETCH_MAX_ROWS // 32, MAX_ROWS // 32
assert MAX_ROWS <= TR_THREADS


def W_of(frames):
    return max(1, -(-max(np.asarray(f).reshape(-1, 5).shape[0] for f in frames) // 32))


def reloads(F):
    """Frames at which k_track_resolve reloads its offsets (tracker.cu:523: at f - c0 >= OFF_CHUNK, c0 = f - 1)."""
    out, c0 = [], 0
    for f in range(F):
        if f - c0 >= OFF_CHUNK:
            c0 = f - 1
            out.append(f)
    return out


# ------------------------------------------------------------------------------- the association order, restated in numpy
def values(dets, tb, use_iou):
    """iou_f64 / distance_f64 (tracker.cu:38-62, oracle track_value) of detections dets[D, 4] against one track box: the same
    operand order; the quarter root is libm's pow, like the oracle's.  Larger = better (minus the distance)."""
    a, b = dets, tb
    if use_iou:
        w = np.maximum(np.minimum(a[:, 2], b[2]) - np.maximum(a[:, 0], b[0]), 0.0)
        h = np.maximum(np.minimum(a[:, 3], b[3]) - np.maximum(a[:, 1], b[1]), 0.0)
        inter = w * h
        uni = (a[:, 2] - a[:, 0]) * (a[:, 3] - a[:, 1]) + (b[2] - b[0]) * (b[3] - b[1]) - inter
        with np.errstate(invalid="ignore", divide="ignore"):
            return inter / uni
    adx, ady, bdx, bdy = a[:, 2] - a[:, 0], a[:, 3] - a[:, 1], b[2] - b[0], b[3] - b[1]
    dx = (b[2] + b[0]) / 2 - (a[:, 2] + a[:, 0]) / 2
    dy = (b[3] + b[1]) / 2 - (a[:, 3] + a[:, 1]) / 2
    dz = ((adx - bdx) + (ady - bdy)) / 2
    dis = dz * dz + dx * dx + dy * dy
    return -np.array([math.pow(x, 0.25) for x in dis.tolist()])


def mirror(frames, sigma_iou=0.4, sigma_h=0.6, t_min=5, use_iou=True, sigma_dis=8):
    """iouTracke_cal.py:126-155 / :174-176 in numpy.  -> (tracks_finished, log); log[f] = per active track in order
    (ranked candidate list, their values, outcome): outcome = the rank taken, "unmatched" or "dropped".  Candidates rank by value, then
    detection index (the order k_track_mask and rank_candidates keep); a track takes the best one no earlier track took."""
    thr = sigma_iou if use_iou else -sigma_dis
    active, done, log = [], [], []
    for f, fr in enumerate(frames):
        d = np.asarray(fr, np.float64).reshape(-1, 5)
        D = d.shape[0]
        taken = np.zeros(D, bool)
        upd, lf = [], []
        for tr in active:
            v = values(d[:, :4], tr["last"], use_iou) if D else np.zeros(0)
            assert not np.isnan(v).any(), "the mirror does not model NaN values"
            cand = np.where(v > thr)[0]
            ranked = cand[np.lexsort((cand, -v[cand]))].tolist()
            rv = v[ranked].tolist()
            if taken.all():
                lf.append((ranked, rv, "dropped"))
                continue
            free = [j for j in ranked if not taken[j]]
            if free:
                j = free[0]
                taken[j] = True
                lf.append((ranked, rv, ranked.index(j)))
                tr["rows"].append(d[j, :4].tolist()); tr["last"] = d[j, :4]; tr["max"] = max(tr["max"], d[j, 4])
                upd.append(tr)
            else:
                lf.append((ranked, rv, "unmatched"))
                if tr["max"] > sigma_h and len(tr["rows"]) > t_min:
                    done.append(tr)
        for j in np.where(~taken)[0]:
            upd.append(dict(rows=[d[j, :4].tolist()], last=d[j, :4], max=d[j, 4], start=f + 1))
        active = upd
        log.append(lf)
    done += [tr for tr in active if tr["max"] > sigma_h and len(tr["rows"]) >= t_min]
    return [{"bboxes": t["rows"], "max_score": float(t["max"]), "start_frame": t["start"]} for t in done], log


def ranks(log):
    return [o for lf in log for _, _, o in lf if isinstance(o, int)]


def outcomes(log, kind):
    return sum(o == kind for lf in log for _, _, o in lf)


# ------------------------------------------------------------------------------- generators
def walk(sizes, seed, n_objects=None, width=1280.0, height=720.0, sigma=1.5):
    """Boxes doing pixel random walks; frame f shows sizes[f] of them in a random order (float32 rows like detect_face)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    n = n_objects or max(max(sizes), 1)
    side = rng.uniform(10, 60, (n, 2))
    ctr = np.stack([rng.uniform(30, width - 30, n), rng.uniform(30, height - 30, n)], 1)
    frames = []
    for D in sizes:
        ctr = np.clip(ctr + rng.normal(0, sigma, ctr.shape), 0, [width, height])
        vis = rng.permutation(n)[:D]
        sc = rng.uniform(0.4, 1.0, D)
        frames.append(np.concatenate([ctr[vis] - side[vis] / 2, ctr[vis] + side[vis] / 2, sc[:, None]], 1).astype(np.float32))
    return frames


def frame_size_case(R, seed):
    """A short video whose largest frames have exactly R rows (several in a row, so tracks of R rows meet R candidates), one frame
    of 32 * (W - 1) + 1 rows (the last mask word holds one bit) and small frames around them."""
    W = -(-R // 32)
    sizes = [20, 25, 30, R, R, R, 32 * (W - 1) + 1, R, 40, 5, R, R, 10]
    return walk(sizes, seed, n_objects=R + 16, sigma=2.0)


def reload_case(F, big, seed, at):
    """F frames of a few rows, with crowded frames of `big` rows at the frames in `at` (around the offset reloads)."""
    sizes = [big if f in at else 1 + (f * 7) % 12 for f in range(F)]
    return walk(sizes, seed, n_objects=big + 8, width=900.0, height=600.0, sigma=1.0)


def filler(n, x0=20000.0, step=80.0):
    """n small boxes on a grid, far apart (IoU 0 and distance > 8 to each other and to anything near the origin)."""
    k = np.arange(n)
    x, y = x0 + (k % 40) * step, x0 + (k // 40) * step
    return np.stack([x, y, x + 10, y + 10, np.full(n, 0.9)], 1)


def mix(rows, extra, seed):
    """rows + extra filler rows, in a seeded random order."""
    a = np.concatenate([np.asarray(rows, np.float64).reshape(-1, 5), extra], 0)
    return a[np.random.Generator(np.random.PCG64(seed)).permutation(a.shape[0])]


def pile_case(n_tracks, n_dets, pad_rows, seed):
    """n_tracks identical boxes (tracks that share one preference order), then n_dets concentric boxes 1 px apart: the t-th
    track in active order gets its t-th choice, and tracks past n_dets are dropped.  Repeated so every pile meets both identical
    (IoU 1 / distance 0 ties) and concentric candidates; filler rows pad the frames to pad_rows (W = pad_rows / 32)."""
    c = 5000.0
    ident = np.array([[c - 50, c - 50, c + 50, c + 50, 0.9]] * n_tracks)
    conc = np.array([[c - 50 - k, c - 50 - k, c + 50 + k, c + 50 + k, 0.7] for k in range(n_dets)])
    fill = filler(max(pad_rows - max(n_tracks, n_dets), 0))
    seq = [ident, ident, conc, ident, conc[::-1], ident, np.zeros((0, 5)), ident, conc]
    return [mix(fr, fill, seed + i) for i, fr in enumerate(seq)]


def tie_case(n_tracks, use_iou, pad_rows, seed):
    """n_tracks identical track boxes; candidates in groups of 4 placed symmetrically around them (shifted by +-s in x and in y:
    equal IoUs below 1 and equal distances), s = 1, 2, 3, 4: ties inside the mask's top 4 and at ranks 4..15."""
    c, h = 3000.0, 20.0
    tb = np.array([[c - h, c - h, c + h, c + h, 0.9]] * n_tracks)
    grp = []
    for s in (1.0, 2.0, 3.0, 4.0):
        for dx, dy in ((s, 0), (-s, 0), (0, s), (0, -s)):
            grp.append([c - h + dx, c - h + dy, c + h + dx, c + h + dy, 0.8])
    fill = filler(max(pad_rows - n_tracks, 0))
    seq = [tb, tb, np.array(grp), tb, np.array(grp[::-1]), tb, np.array(grp)]
    return [mix(fr, fill, seed + i) for i, fr in enumerate(seq)]


def lane_video(scripts, F, use_iou):
    """Independent lanes 1000 px apart; scripts[i](f) -> (box [x1, y1, x2, y2] relative to the lane, score) or None."""
    frames = []
    for f in range(F):
        rows = []
        for i, s in enumerate(scripts):
            r = s(f)
            if r is not None:
                b, sc = r
                rows.append([b[0] + 1000 * i, b[1], b[2] + 1000 * i, b[3], sc])
        frames.append(np.array(rows, np.float64).reshape(-1, 5))
    return frames


F32_06 = float(np.float32(0.6))          # 0.6000000238418579 > sigma_h = 0.6


def threshold_case(use_iou):
    """Equality at every strict comparison.  IoU: [0,0,5,1] -> [0,0,2,1] is intersection 2 / union 5 = 0.4 == sigma_iou (not
    matched), -> [0,0,4,1] 0.8 (matched).  Distance: a centre shift of 64 px is dis = 4096 = 8^4, distance == sigma_dis (not
    matched), 63 px is matched.  Lengths 5 and 6 end in a frame (len > t_min) or at the flush (len >= t_min); max_score exactly
    0.6 (float64) against float32 0.6 widened."""
    F = 14
    if use_iou:
        base, cut, keep = [0, 0, 5, 1], [0, 0, 2, 1], [0, 0, 4, 1]
    else:
        base, cut, keep = [0, 0, 10, 10], [64, 0, 74, 10], [63, 0, 73, 10]

    def ends_at(n, sc=0.9):                  # a track of length n, then the edge box at frame n (not matched -> it ends there)
        return lambda f: (base if f < n else cut, sc) if f <= n + 1 else None

    def tail(n, sc=0.9):                     # a track of length n ending at the flush
        return lambda f: (base, sc) if f >= F - n else None

    scripts = [ends_at(5), ends_at(6), tail(5), tail(4), ends_at(7, 0.6), ends_at(7, F32_06), tail(6, 0.6), tail(6, F32_06),
               lambda f: (keep if f % 2 else base, 0.9) if f < 9 else None]
    return lane_video(scripts, F, use_iou)


def nan_case(seed):
    """Dummy rows [0,0,0,0,0.4] inside a W_MAX video: a frame of MAX_ROWS - 1 rows + a dummy, then one of MAX_ROWS rows with a
    dummy (0/0 IoU: the NaN flag sends the whole frame down the warp-sequential path), and two dummy-only frames."""
    fr = walk([MAX_ROWS - 1, MAX_ROWS - 1, MAX_ROWS - 1, 30, 30], seed, n_objects=MAX_ROWS + 8)
    dummy = np.array([[0, 0, 0, 0, 0.4]])
    a = np.concatenate([fr[1], dummy]); b = np.concatenate([dummy, fr[2]])
    return [fr[0], a, b, dummy, dummy, fr[3], fr[4], b]


def capacity_case():
    """Online, max_dets_per_frame = 40 (cap = 64): frames of 41..64 rows, one of cap + 1 rows at step 9."""
    sizes = [41 + (k * 5) % 24 for k in range(24)]
    fr = walk(sizes, 77, n_objects=80, width=400.0, height=300.0)
    fr[9] = walk([65], 78, n_objects=80, width=400.0, height=300.0)[0]
    return fr


def finish_all_case(cap):
    """cap boxes for 7 frames (tracks of length 7), then cap boxes far from all of them: every track finishes in one step
    (fin_count == cap); those boxes stay for 6 frames, so the flush finishes cap tracks too."""
    a = filler(cap, x0=100.0, step=100.0)
    b = filler(cap, x0=100.0 + 50000.0, step=100.0)
    return [a] * 7 + [b] * 6


# name -> (frames, tracker kwargs, regime check)
CASES = {}


def case(name, frames, kw=None, check=None):
    CASES[name] = (frames, kw or {}, check)


def _rows(frames):
    return [np.asarray(f).reshape(-1, 5).shape[0] for f in frames]


for R, s in ((PREFETCH_MAX_ROWS - 1, 1), (PREFETCH_MAX_ROWS, 2), (PREFETCH_MAX_ROWS + 1, 3), (32 * (W_PF + 1), 4),
             (MAX_ROWS - 32, 5), (MAX_ROWS, 6)):
    case(f"rows{R}", lambda R=R, s=s: frame_size_case(R, 100 + s),
         check=lambda fr, R=R: (max(_rows(fr)) == R and _rows(fr).count(R) >= 3 and 32 * (W_of(fr) - 1) + 1 in _rows(fr)
                                and (R <= PREFETCH_MAX_ROWS) == (resolve_smem(W_of(fr), 1) <= SMEM_LIMIT)))

AROUND = set(range(510, 515)) | set(range(1021, 1027))
case("reload_noprefetch_F1030", lambda: reload_case(1030, 32 * W_PF + 32, 201, AROUND),
     check=lambda fr: W_of(fr) > W_PF and reloads(len(fr)) == [512, 1023] and all(_rows(fr)[f] > 32 * W_PF for f in AROUND))
case("reload_prefetch_F1030", lambda: reload_case(1030, PREFETCH_MAX_ROWS, 201, AROUND),
     check=lambda fr: W_of(fr) == W_PF and reloads(len(fr)) == [512, 1023] and all(_rows(fr)[f] == PREFETCH_MAX_ROWS for f in AROUND))
for F in (OFF_CHUNK, OFF_CHUNK + 1):
    case(f"reload_F{F}", lambda F=F: reload_case(F, 32 * W_PF + 32, 202 + F, set(range(F - 4, F))),
         check=lambda fr, F=F: len(fr) == F and W_of(fr) > W_PF and reloads(F) == ([512] if F > OFF_CHUNK else []))


def pile_check(n_tracks, n_dets):
    def chk(fr, log):
        r = ranks(log)
        need = n_tracks - 1                       # the last of n_tracks identical tracks takes its last choice
        assert max(r) == need, (max(r), need)
        if n_tracks > n_dets:
            assert outcomes(log, "dropped") > 0
    return chk


for n in (4, 5, 8, 9, 40):
    for pad, tag in ((0, "W_small"), (32 * W_PF + 32, "W20"), (MAX_ROWS, "Wmax")):
        for use_iou in (True, False):
            case(f"pile{n}_{tag}_{'iou' if use_iou else 'dist'}", lambda n=n, pad=pad: pile_case(n, n, pad, 300 + n),
                 dict(use_iou=use_iou, sigma_h=0.0, t_min=0), pile_check(n, n))
def drop_case(n_tracks, n_dets, seed):
    """n_tracks identical boxes, then n_dets identical boxes (IoU 1 / distance 0 ties: track t takes detection t): the tracks
    past n_dets find every detection taken and are dropped; no filler, so nothing else is left for them."""
    c = 5000.0
    box = [c - 50, c - 50, c + 50, c + 50]
    ident = lambda n, sc: np.array([box + [sc]] * n)
    seq = [ident(n_tracks, 0.9), ident(n_tracks, 0.8), ident(n_dets, 0.7), ident(n_tracks, 0.9), ident(n_dets, 0.95)]
    return [mix(fr, np.zeros((0, 5)), seed + i) for i, fr in enumerate(seq)]


for nt, nd, tag in ((12, 7, "W_small"), (32 * W_PF + 32, 32 * W_PF - 40, "W20"), (MAX_ROWS, MAX_ROWS - 100, "Wmax")):
    for use_iou in (True, False):
        case(f"pile_drop_{tag}_{'iou' if use_iou else 'dist'}", lambda nt=nt, nd=nd: drop_case(nt, nd, 350),
             dict(use_iou=use_iou, sigma_h=0.0, t_min=0), pile_check(nt, nd))


def tie_check(fr, log, use_iou):
    """A track takes a candidate whose value (IoU below 1 / distance above 0) equals another candidate's, so the lower detection
    index decides: once inside the mask's top 4 and once at rank >= 4 (after the re-rank)."""
    got = set()
    for lf in log:
        for ranked, rv, o in lf:
            if isinstance(o, int) and 0 < abs(rv[o]) and (abs(rv[o]) < 1 or not use_iou) and rv.count(rv[o]) > 1:
                got.add(o >= 4)
    assert got == {False, True}, got


for use_iou in (True, False):
    for pad, tag in ((0, "W_small"), (32 * W_PF + 32, "W20")):
        case(f"ties_{tag}_{'iou' if use_iou else 'dist'}", lambda use_iou=use_iou, pad=pad: tie_case(14, use_iou, pad, 400),
             dict(use_iou=use_iou, sigma_h=0.0, t_min=0), lambda fr, log, u=use_iou: tie_check(fr, log, u))


def threshold_check(fr, log, use_iou, kw):
    sig = kw.get("sigma_iou", 0.4) if use_iou else -kw.get("sigma_dis", 8)
    at_edge = 0
    for f in range(1, len(fr)):
        a, b = np.asarray(fr[f - 1], np.float64), np.asarray(fr[f], np.float64)
        for row in a:
            v = values(b[:, :4], row[:4], use_iou)
            at_edge += int((v == sig).sum())
    assert at_edge > 0                                                # a value exactly at the threshold
    tr, _ = mirror(fr, **kw)
    lens = sorted(len(t["bboxes"]) for t in tr)
    assert 5 in lens and 6 in lens                                   # len == t_min at the flush kept, len > t_min in a frame kept
    assert any(t["max_score"] == F32_06 for t in tr) and all(t["max_score"] != 0.6 for t in tr)


for use_iou in (True, False):
    case(f"threshold_{'iou' if use_iou else 'dist'}", lambda use_iou=use_iou: threshold_case(use_iou), dict(use_iou=use_iou),
         lambda fr, log, u=use_iou: threshold_check(fr, log, u, dict(use_iou=u)))
case("nan_Wmax", lambda: nan_case(500),
     check=lambda fr: W_of(fr) == W_MAX and max(_rows(fr)) == MAX_ROWS and any(
         (np.asarray(f)[:, :4] == 0).all(1).any() and np.asarray(f).shape[0] == MAX_ROWS for f in fr))


BEHAVIOURAL = sorted(k for k in CASES if k.startswith(("pile", "ties", "threshold")))
_FRAMES = {}


def frames_of(name):
    if name not in _FRAMES:
        _FRAMES[name] = CASES[name][0]()
    return _FRAMES[name]


def same_tracks(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x["start_frame"] == y["start_frame"] and x["max_score"] == y["max_score"]
        assert x["bboxes"] == y["bboxes"]                      # float64 boxes bit-exact, same append order


# ------------------------------------------------------------------------------- regime checks (no GPU)
@pytest.mark.parametrize("name", sorted(CASES))
def test_case_reaches_its_edge(name):
    fr = frames_of(name)
    _, kw, check = CASES[name]
    if name in BEHAVIOURAL:
        tr, log = mirror(fr, **kw)
        same_tracks(tr, orc.iou_track(fr, **kw))                # the mirror is the oracle's association order
        check(fr, log)
    else:
        assert check(fr)


def test_constants_match_the_kernel_limits():
    assert (PREFETCH_MAX_ROWS, MAX_ROWS) == (608, 864)
    assert resolve_smem(W_MAX, 0) == 224640 and resolve_smem(W_MAX + 1, 0) > SMEM_LIMIT
    assert reloads(1535) == [512, 1023, 1534]


def test_one_row_limit_for_every_entry_point_without_a_gpu():
    """MAX_ROWS rows per frame are accepted and MAX_ROWS + 1 refused by the size queries, init / step / flush and the offline
    call, before any CUDA call (so this runs without a device)."""
    import ctypes as C
    L = _lib.lib()
    for n in (MAX_ROWS, MAX_ROWS + 1):                     # the size queries first: they touch no memory
        ok = n <= MAX_ROWS
        assert (L.fdt_track_stream_state_bytes(1, n) > 0) == ok and (L.fdt_track_stream_workspace_bytes(1, n) > 0) == ok
        assert (L.fdt_iou_track_workspace_bytes(10, 100, n) > 0) == ok
    # The calls below get placeholder pointers (address 256, never allocated): every one must be refused by the row limit
    # before it enqueues a memset or a launch, which is what they check.  If an entry point checked the limit after its first
    # CUDA call, the device would write to address 256; keep the limit checks ahead of any CUDA call.
    st, big, p = C.c_void_p(256), 1 << 40, [C.c_void_p(256)] * 8
    assert L.fdt_track_stream_init(st, big, 1, MAX_ROWS + 1, 0, 0.4, 0.6, 5, None) == _lib.FDT_E_UNSUPPORTED
    assert str(MAX_ROWS) in _lib.last_error()
    assert L.fdt_track_stream_step(st, 1, MAX_ROWS + 1, *p[:3], *p[:7], st, big, None) == _lib.FDT_E_UNSUPPORTED
    assert L.fdt_track_stream_flush(st, 1, MAX_ROWS + 1, None, *p[:6], None) == _lib.FDT_E_UNSUPPORTED
    for metric in (0, 1):
        assert L.fdt_iou_track_metric(p[0], p[0], 3, 2000, MAX_ROWS + 1, metric, 0.4, 0.6, 5, *p[:5], p[0], big,
                                      None) == _lib.FDT_E_UNSUPPORTED
    with pytest.raises(NotImplementedError):
        _lib.check(L.fdt_track_stream_init(st, big, 1, MAX_ROWS + 1, 0, 0.4, 0.6, 5, None))


def test_libm_quarter_root_reference_is_exact_on_fourth_powers():
    """The oracle's `dis ** 0.25` gives k for dis = k^4, the values the distance threshold cases sit on."""
    k = np.arange(0, 1 << 13, dtype=np.float64)
    z = np.zeros_like(k)
    d = orc.calculate_distance_f64(np.stack([k * k, z, k * k, z], 1), np.zeros((1, 4)))[:, 0]
    assert np.array_equal(d, k)


# ------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def tracker():
    from fdt_b200 import tracker as T
    return T


@pytest.fixture(scope="module")
def stream_helpers():
    from tests.test_tracker_stream_gpu import check_video, run_streams
    return run_streams, check_video


@pytest.mark.gpu
@pytest.mark.parametrize("slow", ["0", "1"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_offline_equals_oracle(tracker, name, slow, monkeypatch):
    monkeypatch.setenv("FDT_TRACK_FORCE_SLOW", slow)
    fr = frames_of(name)
    kw = CASES[name][1]
    same_tracks(tracker.iou_track(fr, **kw), orc.iou_track(fr, **kw))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_online_equals_oracle(tracker, stream_helpers, name):
    run_streams, check_video = stream_helpers
    fr = frames_of(name)
    kw = CASES[name][1]
    st, ids, recs = run_streams(tracker, [fr], kw=kw)
    assert st.cap == 32 * W_of(fr)
    check_video(tracker, st, 0, fr, ids[0], recs[0], **kw)


@pytest.mark.gpu
def test_online_capacity_is_cap_not_max_dets_per_frame(tracker):
    """max_dets_per_frame = 40 -> cap = 64: frames of 41..64 rows are tracked, the frame of 65 rows is skipped and flagged."""
    fr = capacity_case()
    st = tracker.StreamTracker(1, 40, keep_history=True)
    assert st.cap == 64
    for s, f in enumerate(fr):
        dets, off = tracker.pack_frames([f])
        out = st.step(dets, off)
        rt = out["row_track"].cpu().numpy()
        if s == 9:
            assert f.shape[0] == st.cap + 1 and st.status() == _lib.TRACK_STATUS_OVERFLOW and (rt == -1).all()
        else:
            assert 40 < f.shape[0] <= st.cap and (rt >= 0).all()
    st.flush()
    with pytest.raises(RuntimeError, match="cap=64"):
        st.check()
    same_tracks(st.tracks_finished(0), orc.iou_track(fr[:9] + fr[10:]))


@pytest.mark.gpu
@pytest.mark.parametrize("cap", [64, MAX_ROWS])
def test_online_step_and_flush_finish_cap_tracks(tracker, cap):
    fr = finish_all_case(cap)
    st = tracker.StreamTracker(1, cap, keep_history=True)
    counts = []
    for f in fr:
        dets, off = tracker.pack_frames([f])
        counts.append(int(st.step(dets, off)["fin_count"][0]))
    fl = st.flush()
    assert counts == [0] * 7 + [cap] + [0] * 5 and int(fl["fin_count"][0]) == cap
    assert sorted(fl["fin_index"][0].cpu().numpy().tolist()) == list(range(cap, 2 * cap))
    st.check()
    same_tracks(st.tracks_finished(0), orc.iou_track(fr))


@pytest.mark.gpu
def test_more_streams_than_sms_at_the_largest_cap(tracker, stream_helpers):
    """149 streams at cap = MAX_ROWS: one 864-thread CTA with 224,640 B of shared memory per SM, so more CTAs than SMs."""
    run_streams, check_video = stream_helpers
    V = 149
    videos = [walk([1 + (v * 13 + k * 7) % 40 for k in range(6 + v % 5)], 900 + v, n_objects=48) for v in range(V)]
    for v in (0, 74, 148):
        videos[v][2] = walk([MAX_ROWS], 990 + v, n_objects=MAX_ROWS)[0]
    st, ids, recs = run_streams(tracker, videos, [v % 3 for v in range(V)])
    assert st.cap == MAX_ROWS
    for v in (0, 1, 74, 147, 148):
        check_video(tracker, st, v, videos[v], ids[v], recs[v])
    for v in range(V):
        same_tracks(st.tracks_finished(v), tracker.iou_track(videos[v]))


@pytest.mark.gpu
def test_row_limit_accepted_and_refused(tracker):
    ok = walk([MAX_ROWS, MAX_ROWS], 61, n_objects=MAX_ROWS)
    same_tracks(tracker.iou_track(ok), orc.iou_track(ok))
    bad = walk([MAX_ROWS + 1, 3], 62, n_objects=MAX_ROWS + 1)
    for use_iou in (True, False):
        with pytest.raises(NotImplementedError):
            tracker.iou_track(bad, use_iou=use_iou)
    tracker.StreamTracker(1, MAX_ROWS)
    with pytest.raises(NotImplementedError):
        tracker.StreamTracker(1, MAX_ROWS + 1)


def _exact_side(x, y_lo, y_hi):
    """True when y_hi is the correctly rounded x ** 0.25 of the neighbours y_lo < y_hi (exact rationals)."""
    m = (Fraction(y_lo) + Fraction(y_hi)) / 2
    return m ** 4 < Fraction(x)


@pytest.mark.gpu
def test_device_quarter_root_is_correctly_rounded():
    """calculate_distance's `dis ** 0.25` on the device (fdt_qroot_cr, shared with the tracker) is correctly rounded: exact on
    fourth powers, and over a seeded sample of 2^24 within one ulp of libm's pow and equal to it for more than 99 %; wherever the
    two differ, exact rational arithmetic must show the device's value to be the correctly rounded one.  CUDA's pow missed k for
    491 of the k^4 below and about a quarter of the sample."""
    from fdt_b200.utils import calc_performance as cp
    k = np.arange(0, 1 << 13, dtype=np.float64)
    z = np.zeros_like(k)
    assert np.array_equal(cp.calculate_distance(np.stack([k * k, z, k * k, z], 1), np.zeros((1, 4)))[:, 0], k)
    q = np.arange(1, 4097, dtype=np.float64) / 64                   # (q^2)^2 with fractional q, exact too
    assert np.array_equal(cp.calculate_distance(np.stack([q * q, 0 * q, q * q, 0 * q], 1), np.zeros((1, 4)))[:, 0], q)
    rng = np.random.Generator(np.random.PCG64(2024))
    n_diff = n_wrong = n = 0
    for it in range(4):
        xa = rng.uniform(-1e3, 1e3, 2048) * np.exp(rng.uniform(-30, 30, 2048))
        xb = rng.uniform(-1e3, 1e3, 2048)
        A, B = np.stack([xa, 0 * xa, xa, 0 * xa], 1), np.stack([xb, 0 * xb, xb, 0 * xb], 1)
        dev, ref = cp.calculate_distance(A, B), orc.calculate_distance_f64(A, B)
        n += dev.size
        for i, j in np.argwhere(dev != ref):
            dx = (float(xb[j]) + float(xb[j])) / 2 - (float(xa[i]) + float(xa[i])) / 2
            x = dx * dx                                              # dis as the kernel forms it (dz = dy = 0); not dx ** 2 (pow)
            a, b = float(dev[i, j]), float(ref[i, j])
            assert abs(np.frexp(a)[1] - np.frexp(b)[1]) <= 1 and np.nextafter(a, b) == b, (x, a, b)
            n_wrong += _exact_side(x, min(a, b), max(a, b)) != (a > b)
            n_diff += 1
    assert n_diff < n // 100 and n_wrong == 0, (n_diff, n_wrong)
