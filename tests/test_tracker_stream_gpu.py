"""GPU tests of the online multi-stream tracker (tracker.StreamTracker, fdt_track_stream_*): for every stream, its steps and its
flush must reproduce the offline tracker on that stream's frames bit for bit -- the C oracle's tracks_finished, and row ids that
group the rows exactly like the offline track_dets."""
import numpy as np
import pytest
import torch

from fdt_b200 import synth
from oracle import oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def tracker():
    from fdt_b200 import tracker as T
    return T


def same_tracks(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x["start_frame"] == y["start_frame"] and x["max_score"] == y["max_score"]
        assert x["bboxes"] == y["bboxes"]                      # float64 boxes bit-exact, same append order


def run_streams(T, videos, starts=None, V=None, kw=None):
    """Feed video k to stream k from step starts[k] on, one frame per step, and flush it right after its last frame.
    -> (tracker, per video: row ids in packed-row order, finish records {fin_index: (id, start, len, max)})."""
    kw = kw or {}
    V = V or len(videos)
    starts = starts or [0] * len(videos)
    ends = [s + len(f) for s, f in zip(starts, videos)]
    max_d = max([max([np.asarray(fr).reshape(-1, 5).shape[0] for fr in f] or [1]) for f in videos] + [1])
    st = T.StreamTracker(V, max_dets_per_frame=max(max_d, 1), keep_history=True, **kw)
    ids = [[] for _ in videos]
    recs = [{} for _ in videos]

    def collect(out, v, rows=None):
        n = int(out["fin_count"][v])                           # (out: host copies)
        for k in range(n):
            recs[v][int(out["fin_index"][v, k])] = (int(out["fin_track"][v, k]), int(out["fin_start"][v, k]),
                                                     int(out["fin_len"][v, k]), float(out["fin_max"][v, k]))
        if rows is not None:
            ids[v].append(rows)

    for s in range(max(ends)):
        adv = np.zeros(V, bool)
        frames = [np.zeros((0, 5))] * V
        for v, f in enumerate(videos):
            if starts[v] <= s < ends[v]:
                adv[v] = True
                frames[v] = f[s - starts[v]]
        dets, off = T.pack_frames(frames)
        out = st.step(dets, off, adv)
        out = {k: t.cpu().numpy() for k, t in out.items()}
        rt = out["row_track"]
        for v in range(len(videos)):
            if adv[v]:
                collect(out, v, rt[off[v]:off[v + 1]])
            else:
                assert int(out["fin_count"][v]) == 0 and (rt[off[v]:off[v + 1]] == -1).all()
        done = np.array([e == s + 1 for e in ends] + [False] * (V - len(videos)))
        if done.any():
            fo = {k: t.cpu().numpy() for k, t in st.flush(done).items()}
            for v in np.where(done)[0]:
                collect(fo, v)
    st.check()
    return st, [np.concatenate(r) if r else np.zeros(0, np.int64) for r in ids], recs


def check_video(T, st, v, frames, ids, recs, **kw):
    ref = orc.iou_track(frames, **kw)
    same_tracks(st.tracks_finished(v), ref)
    dets, off = T.pack_frames(frames)
    t_off, t_dets, t_start, t_max = (x.cpu().numpy() for x in T.iou_track_raw(dets, off, **kw))
    assert sorted(recs) == list(range(len(t_start)))
    for i in range(len(t_start)):                              # the rows of finished track i carry its id, and only they do
        tid, start, ln, mx = recs[i]
        rows = t_dets[t_off[i]:t_off[i + 1]]
        assert (start, ln, mx) == (int(t_start[i]), len(rows), float(t_max[i]))
        assert np.array_equal(np.where(ids == tid)[0], np.sort(rows))
    assert (ids >= 0).all() and ids.shape[0] == off[-1]


VIDEOS = [
    dict(F=400, seed=21, d_lo=1, d_hi=300, n_objects=300, empty_every=133),             # config-4 shape, shorter
    dict(F=300, seed=22, d_lo=100, d_hi=120, n_objects=120, empty_every=0, sigma=6.0),  # crowded, many conflicts
    dict(F=300, seed=23, d_lo=1, d_hi=3, n_objects=3, empty_every=7),
    dict(F=40, seed=24, d_lo=700, d_hi=750, n_objects=750, empty_every=0),              # Detect's top_k = 750 per frame
]


@pytest.mark.parametrize("slow", ["0", "1"])
def test_streams_vs_oracle(tracker, slow, monkeypatch):
    monkeypatch.setenv("FDT_TRACK_FORCE_SLOW", slow)
    videos = [synth.tracker_frames(**kw) for kw in VIDEOS]
    if slow == "1":
        videos = [v[:120] for v in videos]
    starts = [0, 17, 5, 60]                                      # streams of different lengths, starting and ending at different steps
    st, ids, recs = run_streams(tracker, videos, starts)
    for v, f in enumerate(videos):
        check_video(tracker, st, v, f, ids[v], recs[v])


@pytest.mark.parametrize("kw,sigma_dis", [
    (dict(F=300, seed=51, d_lo=1, d_hi=300, n_objects=300, empty_every=100), 8),
    (dict(F=200, seed=52, d_lo=80, d_hi=120, n_objects=120, empty_every=0, sigma=6.0), 20),
    (dict(F=200, seed=53, d_lo=1, d_hi=4, n_objects=4, empty_every=9), 2),
])
def test_streams_distance_mode(tracker, kw, sigma_dis):
    f = synth.tracker_frames(**kw)
    videos = [f, f[:150], synth.tracker_frames(**dict(kw, seed=kw["seed"] + 100))]
    st, ids, recs = run_streams(tracker, videos, [0, 30, 3], kw=dict(use_iou=False, sigma_dis=sigma_dis))
    for v, fr in enumerate(videos):
        check_video(tracker, st, v, fr, ids[v], recs[v], use_iou=False, sigma_dis=sigma_dis)


def test_edge_frames_dummy_empty_identical_duplicated(tracker):
    f = synth.tracker_frames(F=200, seed=31, d_lo=1, d_hi=30, n_objects=30, empty_every=0)
    f[10] = np.zeros((0, 5))                                     # truly empty frame: every active track silently dropped (Q5)
    f[20] = np.array([[0, 0, 0, 0, 0.4]]); f[21] = np.array([[0, 0, 0, 0, 0.4]])   # dummy frames: NaN IoU
    f[50] = f[49].copy()                                         # identical frames
    f[60] = np.concatenate([f[60], f[60][:3]])                   # duplicated detections
    g = [np.zeros((0, 5))] * 3 + f[:80]
    for args in (dict(), dict(sigma_iou=0.1, sigma_h=0.0, t_min=0), dict(sigma_iou=0.7, sigma_h=0.9, t_min=2)):
        st, ids, recs = run_streams(tracker, [f, g], [0, 11], kw=args)
        check_video(tracker, st, 0, f, ids[0], recs[0], **args)
        check_video(tracker, st, 1, g, ids[1], recs[1], **args)


def test_empty_frame_versus_not_advanced(tracker):
    f = synth.tracker_frames(F=60, seed=32, d_lo=5, d_hi=20, n_objects=20, empty_every=0)
    with_gap = f[:30] + [np.zeros((0, 5))] + f[30:]
    # stream 0: frame 30 is truly empty; stream 1: the same video with no frame at that step (not advanced) = the video without it
    st = tracker.StreamTracker(2, 32, keep_history=True)
    for s in range(len(with_gap)):
        dets, off = tracker.pack_frames([with_gap[s], with_gap[s]])
        st.step(dets, off, [True, s != 30])
    st.flush()
    same_tracks(st.tracks_finished(0), orc.iou_track(with_gap))
    same_tracks(st.tracks_finished(1), orc.iou_track(f))
    assert orc.iou_track(with_gap) != orc.iou_track(f)


def test_stream_independence_and_more_streams_than_sms(tracker):
    kw = dict(d_lo=1, d_hi=60, n_objects=60, empty_every=50)
    videos = [synth.tracker_frames(F=60 + (v % 7) * 5, seed=1000 + v, **kw) for v in range(200)]
    st, ids, recs = run_streams(tracker, videos, [v % 11 for v in range(200)])
    for v in (0, 1, 63, 100, 147, 148, 199):
        check_video(tracker, st, v, videos[v], ids[v], recs[v])
    for v in range(200):
        same_tracks(st.tracks_finished(v), orc.iou_track(videos[v]))
    alone, ids1, recs1 = run_streams(tracker, [videos[63]], [63 % 11], V=1)
    assert recs1[0] == recs[63] and np.array_equal(ids1[0], ids[63])
    st64, ids64, recs64 = run_streams(tracker, videos[:65], [v % 11 for v in range(65)])
    assert recs64[63] == recs[63] and np.array_equal(ids64[63], ids[63])


def test_slot_reused_after_flush(tracker):
    a = synth.tracker_frames(F=80, seed=61, d_lo=1, d_hi=40, n_objects=40, empty_every=0)
    b = synth.tracker_frames(F=90, seed=62, d_lo=1, d_hi=40, n_objects=40, empty_every=0)
    st = tracker.StreamTracker(2, 40, keep_history=True)
    outs = []
    for s, fr in enumerate(a + b):
        dets, off = tracker.pack_frames([fr, b[s % len(b)]])
        outs.append(st.step(dets, off))
        if s == len(a) - 1:
            st.flush([True, False])
    st.flush()
    same_tracks(st.tracks_finished(0), orc.iou_track(b))          # the reused slot = a fresh tracker on b
    fresh = tracker.StreamTracker(1, 40, keep_history=True)
    for s, fr in enumerate(b):
        dets, off = tracker.pack_frames([fr])
        o = fresh.step(dets, off)
        assert np.array_equal(o["row_track"].cpu().numpy(), outs[len(a) + s]["row_track"][:off[1]].cpu().numpy())
    fresh.flush()
    same_tracks(fresh.tracks_finished(0), st.tracks_finished(0))


def test_over_capacity_skips_only_that_stream(tracker):
    f = [synth.tracker_frames(F=30, seed=70 + v, d_lo=1, d_hi=30, n_objects=30, empty_every=0) for v in range(3)]
    big = synth.tracker_frames(F=1, seed=79, d_lo=40, d_hi=40, n_objects=40, empty_every=0)[0]     # 40 rows > cap = 32
    st = tracker.StreamTracker(3, 30, keep_history=True)
    for s in range(30):
        frames = [f[0][s], f[1][s], f[2][s]]
        if s == 12:
            frames[1] = big
        dets, off = tracker.pack_frames(frames)
        out = st.step(dets, off)
        if s == 12:
            assert st.status() == 4
            assert (out["row_track"][off[1]:off[2]] == -1).all() and int(out["fin_count"][1]) == 0
    st.flush()
    with pytest.raises(RuntimeError, match="max_dets_per_frame"):
        st.check()
    same_tracks(st.tracks_finished(0), orc.iou_track(f[0]))
    same_tracks(st.tracks_finished(2), orc.iou_track(f[2]))
    same_tracks(st.tracks_finished(1), orc.iou_track(f[1][:12] + f[1][13:]))     # the skipped frame never happened for stream 1


def test_call_not_matching_the_state_changes_nothing(tracker):
    from fdt_b200 import _lib
    f = synth.tracker_frames(F=20, seed=81, d_lo=1, d_hi=20, n_objects=20, empty_every=0)
    st = tracker.StreamTracker(2, 20, keep_history=True)
    for s in range(20):
        dets, off = tracker.pack_frames([f[s], f[s]])
        st.step(dets, off)
        if s == 9:                                                # V = 1 against a 2-stream state
            d = torch.from_numpy(dets).cuda(); o = torch.from_numpy(off[:2]).cuda()
            junk = st._records(); rt = torch.empty(d.shape[0], dtype=torch.int64, device="cuda")
            _lib.check(_lib.lib().fdt_track_stream_step(
                st._state.data_ptr(), 1, 20, d.data_ptr(), o.data_ptr(), None, rt.data_ptr(), junk["fin_count"].data_ptr(),
                junk["fin_index"].data_ptr(), junk["fin_track"].data_ptr(), junk["fin_start"].data_ptr(), junk["fin_len"].data_ptr(),
                junk["fin_max"].data_ptr(), st._ws.data_ptr(), st._ws.numel(), _lib.stream_ptr()))
            assert st.status() == 8
    st.flush()
    same_tracks(st.tracks_finished(0), orc.iou_track(f))
    same_tracks(st.tracks_finished(1), orc.iou_track(f))


@pytest.mark.parametrize("tag", ["a", "b"])
def test_golden_clips_through_step_detections(tracker, golden, tag):
    """The frames.npz clips fed frame by frame from Detect-shaped output (iouTracke_cal.py:117-155 online) reproduce the fixture."""
    g = golden("frames")
    F, top_k, seed, w, h, shrink = g[f"{tag}_cfg"]
    det = torch.from_numpy(synth.clip_detections(int(F), int(top_k), int(seed))).cuda()
    st = tracker.StreamTracker(1, keep_history=True)
    for f in range(int(F)):
        st.step_detections(det[f:f + 1], float(w), float(h), 0.4, float(shrink))
    st.flush()
    st.check()
    tr = st.tracks_finished(0)
    assert [len(t["bboxes"]) for t in tr] == g[f"{tag}_len"].tolist() and [t["start_frame"] for t in tr] == g[f"{tag}_start"].tolist()
    assert np.array_equal(np.array([t["max_score"] for t in tr]), g[f"{tag}_max"])
    assert np.array_equal(np.array([b for t in tr for b in t["bboxes"]], np.float64).reshape(-1, 4), g[f"{tag}_bboxes"])


def test_step_detections_many_cameras_and_cuda_graph(tracker):
    """64 cameras from one [64, 2, top_k, 5] Detect output per step; one step_detections captured in a CUDA graph and replayed per
    frame equals eager, and every camera equals the offline tracker on its own clip."""
    V, F, K = 64, 40, 12
    clips = [synth.clip_detections(F, K, 500 + v) for v in range(V)]
    seq = torch.from_numpy(np.stack(clips, 1)).cuda()              # [F, V, 2, K, 5]
    eager = tracker.StreamTracker(V, 64, keep_history=True)
    graphed = tracker.StreamTracker(V, 64)
    inp = seq[0].clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):                                    # warm up outside the capture
        scratch = tracker.StreamTracker(V, 64)
        scratch.step_detections(inp, 640.0, 480.0)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gout = graphed.step_detections(inp, 640.0, 480.0)
    for f in range(F):
        e = eager.step_detections(seq[f], 640.0, 480.0)
        inp.copy_(seq[f])
        graph.replay()
        n = int(e["frame_off"][-1])
        assert torch.equal(e["frame_off"], gout["frame_off"]) and torch.equal(e["row_track"][:n], gout["row_track"][:n])
        assert torch.equal(e["fin_count"], gout["fin_count"])
        for key in ("fin_index", "fin_track", "fin_start", "fin_len", "fin_max"):
            for v in range(V):
                c = int(e["fin_count"][v])
                assert torch.equal(e[key][v, :c], gout[key][v, :c])
    eager.flush()
    eager.check(); graphed.check()
    for v in (0, 31, 63):
        ref = orc.detections_to_frames(clips[v], 640.0, 480.0, 0.4, 1.0)
        same_tracks(eager.tracks_finished(v), orc.iou_track(ref))
