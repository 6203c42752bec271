#!/usr/bin/env python
"""bench.py -- frames/s of Detect (decode + top-k + NMS) at 640x640, batch 64 per GPU (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--mode random|clustered] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one Detect pass over one batch of B=64 synthetic head outputs per GPU (weak scaling: every rank owns its own
64 images; for N>1 the step includes the gather of the fixed-shape detections block to rank 0, the only exchange the path
has).  Prints ONE JSON line (rank 0).

  value     frames/s, inputs resident in HBM: K = --steps steps issued back to back on ONE stream over 3 rotating input sets
            (165 MB per GPU > 126 MB of L2) and `depth` rotating output buffers, after W = --warmup (at least 3) untimed steps
            issued the same way; timed on the device with one CUDA-event pair around the K steps, barrier + synchronize on both
            sides; max over ranks.  Consecutive calls overlap on the device (workspace ring, fdt_detect in include/fdt_b200.h);
            completion stays in stream order.
  latency   the same step timed one at a time (own event pair, 256 MiB L2 flush + spin before it).
  e2e       frames/s through the public API with pinned HOST tensors: a stream of batches through Detect.submit(...).result()
            (fdt_detect_host_submit / _wait, two batches in flight; every batch's H2D copies, kernels and results inside the
            timed region, wall clock), beside the one-batch-at-a-time Detect.__call__ (`sync_call`) and the host's own pinned
            H2D rate measured in the same run.
  roofline  dominant kernel = the fused k_sort_nms, i.e. the step itself (k_detect_begin is one block); the two-kernel path is
            timed beside it through the stage entry points.
  cpu_baseline  the C oracle port (oracle/, the checker) on the host cores, bounded sample.
  secondary (N=1) BASELINE configs 3, 4, 5 -- MultiBoxLoss B=32, the IoU tracker over 10k frames, Detect B=512 @1024^2 -- each
            with a parity bit against the oracle, outside the headline timed region.
  gather_check (N>1) the fused gathered block on rank 0 == NCCL all-gather of every rank's local Detect output, byte for byte.
--impl reference times the CPU port with all host threads as the reference arm.
--dump-outputs DIR writes the detections block [B x N_GPUs, 2, top_k, 5] (float32) that the last timed step returned to
DIR/detections.npy; the synthetic inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import glob
import json
import os
import collections
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np

B_PER_GPU = 64
WIDTH = HEIGHT = 640
TOP_K, NMS_TOP_K, CONF_T, NMS_T = 750, 5000, 0.05, 0.3
SEED = 20262
ROTATE = 3                                                # input sets per GPU (3 x 54.9 MB > L2)
METRIC = "frames/sec for Detect (decode+top-k+NMS) @640^2 batch 64; % HBM roofline"      # BASELINE.json metric, both arms


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="random", choices=["random", "clustered"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed path returned in its last timed step to DIR/<name>.npy (float32), "
                         "to compare two builds output for output; the inputs depend on the arguments only")
    ap.add_argument("--depth", type=int, default=0, help="workspace slots (calls that may overlap on the device); 0 = library default")
    ap.add_argument("--gather", default="peer", choices=["peer", "peer-inline", "peer-barrier", "peer-all", "nccl"],
                    help="N>1: peer = rows stored into rank 0's gathered block by the NMS kernel over NVLink, completion signalled through "
                         "symmetric memory (fused gather), rank 0's await kernels on a stream of their own; peer-inline = the await "
                         "kernels in the calls' stream; peer-barrier = the stores followed by a symmetric-memory barrier; "
                         "peer-all = into every rank's block, signalled (fused all-gather); nccl = all_gather after the kernel")
    return ap.parse_args()


def workload_config(mode, n_gpus):
    """identical for both arms (the driver compares the dicts)"""
    return {"workload": f"Detect batch {B_PER_GPU}/GPU @{WIDTH}x{HEIGHT} (34,125 priors), conf_thresh {CONF_T}, "
                        f"top_k {TOP_K}, nms_top_k {NMS_TOP_K}, NMS {NMS_T}; synthetic heads mode={mode} seed={SEED}",
            "global_batch": B_PER_GPU * n_gpus, "priors": 34125, "classes": 2,
            "parallelism": f"batch-sharded x{n_gpus}, detections gathered on rank 0" if n_gpus > 1 else "batch-sharded x1"}


GATHER_NOTE = {"peer-inline": "gather to rank 0 fused into k_sort_nms (16-byte NVLink peer stores into a ring of 4 gathered blocks; completion "
                              "signalled through symmetric memory, rank 0's await kernel enqueued behind every call in the same stream)",
               "peer": "gather to rank 0 fused into k_sort_nms (16-byte NVLink peer stores into a ring of 4 gathered blocks; completion "
                       "signals through symmetric memory; rank 0 awaits the signals of the LAST call of a timed block -- epochs are monotonic, "
                       "it covers every call of the block -- with a one-block kernel on a stream of its own that the timed stream waits for "
                       "before the end of the timed region; no rank waits inside the NMS kernel)",
               "peer-barrier": "gather to rank 0 fused into k_sort_nms (NVLink peer stores + symmetric-memory barrier)",
               "peer-all": "all-gather fused into k_sort_nms (NVLink peer stores into every rank's block, signalled)",
               "nccl": "NCCL all-gather of detections after the kernel"}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profile_summary():
    """What the newest ncu summary under profiles/ (profiles/r*_detect_summary*.json, written by tools/ncu_summary.py from an
    `ncu --set full` capture and the launch list of this command) says about the dominant kernel: DRAM bytes per launch and its
    share of the step's kernel time."""
    best = None
    for path in glob.glob(os.path.join(ROOT, "profiles", "r*_detect_summary*.json")):
        try:
            with open(path) as f:
                d = json.load(f)
            if best is None or d.get("order", 0) >= best[1].get("order", 0):
                best = (path, d)
        except Exception:                                         # noqa: BLE001
            pass
    if best is None:
        return {"traffic": None, "traffic_source": "no ncu summary under profiles/", "kernel_share_of_step": None, "share_source": None}
    rel, d = os.path.relpath(best[0], ROOT), best[1]
    return {"traffic": float(d["dram_bytes_read"]) + float(d["dram_bytes_write"]), "traffic_source": rel + ": " + d.get("traffic_note", ""),
            "kernel_share_of_step": d.get("kernel_share_of_step"), "share_source": rel + ": " + d.get("share_note", "")}


def dump_outputs(out_dir, arrays):
    """arrays: name -> float32 / float64 ndarray, written as out_dir/<name>.npy"""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def host_threads():
    """all hardware threads this process may use (torchrun exports OMP_NUM_THREADS=1, which must not throttle the CPU arm)"""
    try:
        return len(os.sched_getaffinity(0))
    except Exception:                                             # noqa: BLE001
        return os.cpu_count() or 1


def cpu_oracle_rate(loc, conf, pri, budget_s, early_exit, threads=0):
    """frames/s of the C oracle port on the host cores; repeats the batch until ~budget_s of wall time."""
    from oracle import oracle as orc
    det = orc.Detect(2, 0, TOP_K, CONF_T, NMS_T)
    det.early_exit = early_exit
    threads = threads if threads > 0 else host_threads()
    det.n_threads = threads
    det(loc[:2], conf[:2], pri)                                   # page in
    n, t0 = 0, time.perf_counter()
    while True:
        det(loc, conf, pri)
        n += loc.shape[0]
        dt = time.perf_counter() - t0
        if dt >= budget_s or n >= 64 * 64:
            break
    return n / dt, n, dt, threads


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.stop_flag, self.ok = [], set(), threading.Event(), False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:                                    # noqa: BLE001
            self.err = repr(e)
        self.active = False

    NAMES = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
             0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
             0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def sample(self):
        nv = self.nv
        mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:                                         # noqa: BLE001
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        if self.active:
            self.samples.append(mhz)
            for bit, name in self.NAMES.items():
                if r & bit and name != "gpu_idle":
                    self.reasons.add(name)

    def run(self):
        while self.ok and not self.stop_flag.is_set():
            try:
                self.sample()
            except Exception:                                     # noqa: BLE001
                pass
            time.sleep(0.0005)

    def result(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "error": getattr(self, "err", "nvml unavailable")}
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def run_reference(args):
    """Reference arm: the reference's CPU algorithm (C oracle port, run to completion like box_utils.nms)
    on the host cores with all threads; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from fdt_b200 import synth
    pri = synth.priors_numpy(WIDTH, HEIGHT)
    loc, conf = synth.detect_inputs(B_PER_GPU, pri, SEED, CONF_T, args.mode)
    from oracle import oracle as orc
    det = orc.Detect(2, 0, TOP_K, CONF_T, NMS_T)
    det.early_exit = False
    cores = host_threads()
    det.n_threads = cores
    for _ in range(max(args.warmup, 1)):
        det(loc, conf, pri)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = det(loc, conf, pri)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"detections": out})
    fps = args.steps * B_PER_GPU / dt
    line = {"impl": "reference", "metric": METRIC, "value": fps,
            "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args.mode, args.gpus),
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                             "sample": f"{args.steps} x the full B={B_PER_GPU} batch, C oracle (oracle/fdt_oracle.c), "
                                       f"OpenMP over images, NMS run to completion as the reference does"},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ secondary workloads (N = 1)
def _timed_isolated(torch, fn, flush, reps, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush.zero_()
        torch.cuda._sleep(250_000)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(statistics.median(ts))


def secondary_workloads(torch, dev, flush, peak):
    """BASELINE.json configs 3, 4 and 5 on one GPU, device-timed (isolated calls, L2 flushed), each checked against the oracle."""
    from fdt_b200 import _lib, synth
    from fdt_b200 import tracker as T
    from fdt_b200.layers import Detect
    from fdt_b200.layers.modules.multibox_loss import pack_targets
    from oracle import oracle as orc
    L = _lib.lib()
    st = _lib.stream_ptr()
    out = {}
    # ---- config 3: MultiBoxLoss forward, B=32, N=34,125, G ~ U{0..200}
    try:
        B = 32
        pri = synth.priors_numpy(640, 640); N = pri.shape[0]
        loc, conf, targets = synth.multibox_inputs(B, pri, 3030, 0, 200)
        l, c, p = (torch.from_numpy(a).to(dev) for a in (loc, conf, pri))
        tg = [torch.from_numpy(t).to(dev) for t in targets]
        gt, off, total = pack_targets(tg, dev)
        losses = torch.empty(2, device=dev); norm = torch.empty(1, device=dev)
        loc_t = torch.empty((B, N, 4), device=dev); conf_t = torch.empty((B, N), dtype=torch.int64, device=dev)
        sel = torch.empty((B, N), dtype=torch.uint8, device=dev)
        ws = _lib.workspace(L.fdt_multibox_workspace_bytes(B, N, 2, total), dev, "bench-mbl")

        def fwd():
            _lib.check(L.fdt_multibox_loss_forward(l.data_ptr(), c.data_ptr(), p.data_ptr(), gt.data_ptr(), off.data_ptr(), total,
                                                   B, N, 2, 0.35, 3, 0, 0.1, 0.2, losses.data_ptr(), norm.data_ptr(),
                                                   loc_t.data_ptr(), conf_t.data_ptr(), sel.data_ptr(), None, ws.data_ptr(),
                                                   ws.numel(), st))
        ms = _timed_isolated(torch, fwd, flush, 15)
        ref = orc.multibox_loss(loc, conf, pri, targets, 0.35, 3, False)
        got = losses.cpu().numpy()
        ok = bool(np.array_equal(conf_t.cpu().numpy(), ref["conf_t"]) and
                  np.array_equal(sel.cpu().numpy().astype(bool), (ref["conf_t"] > 0) | ref["neg"]) and
                  abs(got[0] - ref["loss_l"]) <= 1e-5 * abs(ref["loss_l"]) and abs(got[1] - ref["loss_c"]) <= 1e-5 * abs(ref["loss_c"]))
        G = int(sum(t.shape[0] for t in targets))
        alg = B * 48 * N + 20 * G
        out["multibox_loss_b32"] = {"workload": "MultiBoxLoss match/encode + mining + loss forward, B=32, N=34,125, G~U{0..200} (BASELINE config 3)",
                                    "ms": ms, "value": B / (ms * 1e-3), "unit": "images/s", "algorithmic_bytes": alg,
                                    "roofline_frac": alg / (ms * 1e-3) / 1e9 / peak, "gt_boxes": G,
                                    "parity": "ok" if ok else "MISMATCH",
                                    "parity_how": "whole batch vs the C oracle: match labels and mined mask bit-exact, both losses within 1e-5 relative"}
        del l, c, loc_t, conf_t, sel
    except Exception as e:                                        # noqa: BLE001
        out["multibox_loss_b32"] = {"error": repr(e)}
    # ---- config 4: IoU tracker, 10,000 frames x U{1..300} detections
    try:
        frames = synth.tracker_frames(F=10000, seed=4040, d_lo=1, d_hi=300, n_objects=300, empty_every=1000)
        dets, off = T.pack_frames(frames)
        d = torch.from_numpy(dets).to(dev); o = torch.from_numpy(off).to(dev)
        F = len(frames); total = int(off[-1]); max_d = int(np.diff(off).max())
        n = torch.zeros(1, dtype=torch.int64, device=dev); t_off = torch.zeros(total + 2, dtype=torch.int64, device=dev)
        t_dets = torch.zeros(total, dtype=torch.int64, device=dev); t_start = torch.zeros(total + 1, dtype=torch.int64, device=dev)
        t_max = torch.zeros(total + 1, dtype=torch.float64, device=dev)
        ws = _lib.workspace(L.fdt_iou_track_workspace_bytes(F, total, max_d), dev, "bench-trk")

        def run():
            _lib.check(L.fdt_iou_track(d.data_ptr(), o.data_ptr(), F, total, max_d, 0.4, 0.6, 5, n.data_ptr(), t_off.data_ptr(),
                                       t_dets.data_ptr(), t_start.data_ptr(), t_max.data_ptr(), ws.data_ptr(), ws.numel(), st))
        ms = _timed_isolated(torch, run, flush, 3, warm=1)
        tr = T.iou_track(frames)
        t0 = time.perf_counter(); ref = orc.iou_track(frames); cpu_s = time.perf_counter() - t0
        same = len(tr) == len(ref) and all(a["bboxes"] == b["bboxes"] and a["start_frame"] == b["start_frame"] and
                                           a["max_score"] == b["max_score"] for a, b in zip(tr, ref))
        out["iou_tracker_10k"] = {"workload": "IoU tracker association, 10,000 frames x U{1..300} detections (BASELINE config 4)",
                                  "ms": ms, "value": F / (ms * 1e-3), "unit": "frames/s", "detections": total, "tracks": len(tr),
                                  "algorithmic_bytes": 28 * total, "roofline_frac": 28 * total / (ms * 1e-3) / 1e9 / peak,
                                  "note": "latency-bound serial chain over the frames (SURVEY 8d); replicas only across GPUs",
                                  "cpu_port_frames_per_s_1_thread": F / cpu_s,
                                  "parity": "ok" if same else "MISMATCH",
                                  "parity_how": "all 10,000 frames vs the C oracle: track membership, order, start frames and max scores bit-exact"}
    except Exception as e:                                        # noqa: BLE001
        out["iou_tracker_10k"] = {"error": repr(e)}
    # ---- config 5 on one GPU: Detect B=512 @1024x1024 (N=87,360), device-generated inputs (1.07 GB)
    try:
        B = 512
        pri = synth.priors_numpy(1024, 1024); N = pri.shape[0]
        g = torch.Generator(device=dev); g.manual_seed(5)
        loc = torch.randn((B, N, 4), device=dev, generator=g) * 0.5
        s1 = torch.sigmoid(torch.randn((B, N), device=dev, generator=g) * 2.0 - 4.5)
        conf = torch.stack([1 - s1, s1], -1).contiguous()
        del s1
        det = Detect(2, 0, TOP_K, CONF_T, NMS_T)
        p = torch.from_numpy(pri).to(dev)
        res = [None]

        def run5():
            res[0] = det(loc, conf, p)
        ms = _timed_isolated(torch, run5, flush, 6)
        sample = 6
        ref = orc.Detect(2, 0, TOP_K, CONF_T, NMS_T)
        ref.early_exit = True
        want = ref(loc[:sample].cpu().numpy(), conf[:sample].cpu().numpy(), pri)
        ok = bool(np.array_equal(res[0][:sample].cpu().numpy(), want))
        alg = B * (24 * N + 30000) + 16 * N
        out["detect_b512_1024"] = {"workload": "Detect B=512 @1024x1024 (N=87,360) on one GPU (BASELINE config 5 unsharded; device-generated inputs)",
                                   "ms": ms, "value": B / (ms * 1e-3), "unit": "frames/s", "algorithmic_bytes": alg,
                                   "roofline_frac": alg / (ms * 1e-3) / 1e9 / peak,
                                   "parity": "ok" if ok else "MISMATCH",
                                   "parity_how": f"first {sample} images vs the C oracle, bit-exact (scores may tie: both sides order ties by prior index)"}
        del loc, conf
    except Exception as e:                                        # noqa: BLE001
        out["detect_b512_1024"] = {"error": repr(e)}
    return out


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import fdt_b200  # noqa: F401
    from fdt_b200 import _lib, synth
    from fdt_b200.layers import Detect

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    _lib.check(_lib.lib().fdt_device_check(local))
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    pri_np = synth.priors_numpy(WIDTH, HEIGHT)
    N = pri_np.shape[0]
    # ROTATE input sets per GPU: 3 x 54.9 MB = 165 MB > 126 MB of L2, so back-to-back steps read their inputs from HBM
    sets = []
    for r in range(ROTATE):
        l_np, c_np = synth.detect_inputs(B_PER_GPU, pri_np, SEED + rank + 1000 * r, CONF_T, args.mode)
        if r == 0:
            loc_np, conf_np = l_np, c_np
        sets.append((torch.from_numpy(l_np).to(dev), torch.from_numpy(c_np).to(dev)))
    pri = torch.from_numpy(pri_np).to(dev)
    cur = [0]                                            # step counter: which input set / output buffer the next step uses

    def inputs():
        return sets[cur[0] % ROTATE]
    det = Detect(2, 0, TOP_K, CONF_T, NMS_T)
    B, C = B_PER_GPU, 2
    L = _lib.lib()
    depth = args.depth if args.depth > 0 else _lib.DETECT_DEPTH
    depth = max(1, min(4, depth))
    ws = torch.empty(L.fdt_detect_workspace_bytes_depth(B, N, C, depth), dtype=torch.uint8, device=dev)
    n_out = max(depth, 2)
    outs = [torch.empty((B, C, TOP_K, 5), dtype=torch.float32, device=dev) for _ in range(n_out)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)              # > 126 MB L2
    st = _lib.stream_ptr()

    def stage1():
        _lib.check(L.fdt_detect_threshold_compact(inputs()[1].data_ptr(), B, N, C, CONF_T, ws.data_ptr(), ws.numel(), st))

    def stage2():
        _lib.check(L.fdt_detect_sort_nms(inputs()[0].data_ptr(), pri.data_ptr(), B, N, C, TOP_K, NMS_TOP_K, NMS_T, 0.1, 0.2,
                                         outs[0].data_ptr(), None, None, ws.data_ptr(), ws.numel(), st))

    gather = args.gather if world > 1 else None
    peer = None
    gathered = None
    if world > 1 and gather in ("peer", "peer-inline", "peer-barrier", "peer-all"):
        try:
            from fdt_b200.sharding import PeerGatherDetect
            peer = PeerGatherDetect(det, B, dest="all" if gather == "peer-all" else 0,
                                    signal={"peer-barrier": "barrier", "peer": "kernel-side"}.get(gather, "kernel"))
        except Exception as e:                          # noqa: BLE001  (symmetric memory unavailable: keep the NCCL gather)
            if rank == 0:
                print(f"peer gather unavailable ({e!r}); using NCCL all_gather", file=sys.stderr)
            gather = "nccl"
    if world > 1 and gather == "nccl":
        gathered = [torch.empty((world * B, C, TOP_K, 5), dtype=torch.float32, device=dev) for _ in range(n_out)]
    last_block = [None]

    def step():
        # N=1: the public C-ABI call.  N>1: the same call with the gather fused into the NMS kernel (or followed by NCCL).
        lc = inputs()
        args12 = (lc[0].data_ptr(), lc[1].data_ptr(), pri.data_ptr(), B, N, C, TOP_K, NMS_TOP_K, CONF_T, NMS_T, 0.1, 0.2)
        if world == 1 or gather == "nccl":
            o = outs[cur[0] % n_out]
            _lib.check(L.fdt_detect(*args12, o.data_ptr(), None, None, ws.data_ptr(), ws.numel(), st))
            if world > 1:
                dist.all_gather_into_tensor(gathered[cur[0] % n_out], o)
                last_block[0] = gathered[cur[0] % n_out]
            else:
                last_block[0] = o
        else:
            hdl, buf = peer.hdls[peer.turn], peer.bufs[peer.turn]
            peer.turn = (peer.turn + 1) % peer.RING
            ptrs, n_dst = peer.dest_ptrs(hdl)
            if peer.signal == "kernel":
                peer.epoch += 1
                root = -1 if peer.dest == "all" else 0
                call = L.fdt_detect_gather_store if peer.await_stream is not None else L.fdt_detect_gather_signal
                _lib.check(call(*args12, ptrs, n_dst, int(peer.sig_hdl.buffer_ptrs_dev), world, rank, root, peer.epoch, peer.RING, rank * B,
                                ws.data_ptr(), ws.numel(), st))
                peer._last_ws = ws                  # (kernel-side: rank 0 awaits when the rows are needed, peer.wait_ready())
            else:
                _lib.check(L.fdt_detect_peers(*args12, ptrs, n_dst, rank * B, ws.data_ptr(), ws.numel(), st))
                hdl.barrier()
            last_block[0] = buf
        cur[0] += 1

    spin_cycles = 250_000
    torch.cuda._sleep(spin_cycles)
    for _ in range(max(args.warmup, 3)):                # untimed steps, issued back to back like the timed ones
        step()
    torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()
    # ---- throughput: the K = --steps timed steps back to back over the rotating input sets, one event pair around them, barrier +
    #      synchronize on both sides
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    wall0 = time.perf_counter()
    sampler.active = True
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(2_000_000)                        # ~1 ms of GPU spin: the host gets ahead, the pair sees device time only
    e0.record()
    for _ in range(args.steps):
        step()
    if peer is not None:
        peer.wait_ready()                               # (await kernels on their own stream: the timed stream waits for the last one)
    e1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - wall0
    if world > 1:
        dist.barrier()
    t = torch.tensor([float(e0.elapsed_time(e1))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)        # max over ranks
    total_ms = float(t.item())
    if args.dump_outputs and rank == 0:
        # the detections block the last timed step returned (N > 1: rank 0's gathered block of every rank's images)
        dump_outputs(args.dump_outputs, {"detections": last_block[0].cpu().numpy()})
    # ---- N>1: the gathered block the timed path produced must equal the NCCL all-gather of the ranks' local outputs
    gather_check = None
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        cur[0] = 0
        step()                                          # one more step on input set 0
        if peer is not None:
            peer.wait_ready()
        torch.cuda.synchronize()
        dist.barrier()
        fused = last_block[0].clone()
        local_out = det(sets[0][0], sets[0][1], pri)
        ref_block = torch.empty((world * B, C, TOP_K, 5), dtype=torch.float32, device=dev)
        dist.all_gather_into_tensor(ref_block, local_out)
        torch.cuda.synchronize()
        same = True
        if rank == 0 or gather in ("peer-all", "nccl"):
            same = bool(torch.equal(fused.view(torch.int32), ref_block.view(torch.int32)))
        if peer is not None:
            try:
                peer.check()
            except RuntimeError as e:
                same = False
                print(f"rank {rank}: {e}", file=sys.stderr)
        t = torch.tensor([1 if same else 0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        gather_check = "ok" if int(t.item()) == 1 else "MISMATCH"
    # ---- latency: the same step in isolation (own event pair; L2 flushed and the GPU spinning while the host enqueues it)
    n_lat = max(10, min(args.steps, 30))
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(n_lat)]
    for i in range(n_lat):
        flush.zero_()                                   # L2 flush, outside the event pairs
        torch.cuda._sleep(spin_cycles)
        ev[i][0].record()
        step()
        if peer is not None:
            peer.wait_ready()
        ev[i][1].record()
    torch.cuda.synchronize()
    if sampler.ok:
        try:
            sampler.sample()
        except Exception:                               # noqa: BLE001
            pass
    sampler.active = False
    sampler.stop_flag.set()
    step_ms = [e[0].elapsed_time(e[1]) for e in ev]
    unfused = None
    if world == 1:
        # for reference: the two-kernel path (K2 threshold/compaction grid + k_sort_nms reading its keys), stage entry points.
        # (a) k_sort_nms isolated: stage 1, then an event pair around the stage-2 launch, L2 flushed before the step
        k3 = []
        for _ in range(max(10, min(args.steps, 30))):
            flush.zero_()
            torch.cuda._sleep(spin_cycles)
            stage1()
            a, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            stage2()
            b2.record()
            torch.cuda.synchronize()
            k3.append(a.elapsed_time(b2))
            cur[0] += 1
        # (b) K stage-2 launches back to back on one prepared workspace slot (they overlap on the device), average per launch
        reps = []
        for _ in range(5):
            stage1()
            torch.cuda.synchronize()
            a, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(1_000_000)
            a.record()
            for _ in range(args.steps):
                stage2()
            b2.record()
            torch.cuda.synchronize()
            reps.append(a.elapsed_time(b2) / args.steps)
            cur[0] += 1
        unfused = {"k_sort_nms_ms_isolated": float(statistics.median(k3)), "k_sort_nms_ms_back_to_back": float(statistics.median(reps)),
                   "note": "two-kernel path through fdt_detect_threshold_compact + fdt_detect_sort_nms (head-map input and fdt_set_option('detect_fused', 0) "
                           "still take it): k_sort_nms alone, isolated and as K overlapping launches on one prepared slot"}
    lat_ms = float(np.mean(step_ms))
    if world > 1:
        t = torch.tensor([lat_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        lat_ms = float(t[0].item())
    ms_per_step = total_ms / args.steps
    value = world * B * args.steps / (total_ms * 1e-3)

    peak, peak_src = peaks()
    roofline = None
    if world == 1:
        step_bytes = B * (24 * N + C * TOP_K * 5 * 4) + 16 * N         # SURVEY 8(d): 849,000 B/image (conf 8 N + loc 16 N + rows) + priors once
        prof = profile_summary()
        roofline = {"bound": "hbm", "kernel": "k_sort_nms<DETECT, fused> (threshold + select/sort + decode + lazy NMS + output rows: the whole step but the "
                                              "one-block sequencing kernel k_detect_begin)",
                    "achieved": step_bytes / (ms_per_step * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                    "frac": step_bytes / (ms_per_step * 1e-3) / 1e9 / peak,
                    "traffic": prof.get("traffic"), "traffic_source": prof.get("traffic_source"),
                    "peak_source": peak_src,
                    "kernel_ms": ms_per_step, "kernel_ms_isolated": lat_ms,
                    "frac_isolated": step_bytes / (lat_ms * 1e-3) / 1e9 / peak,
                    "kernel_share_of_step": prof.get("kernel_share_of_step"), "share_source": prof.get("share_source"),
                    "kernel_timing": "kernel_ms = average launch duration over the timed region (K launches issued back to back on one stream, "
                                     "overlapping on the device; median block / K); kernel_ms_isolated = one call alone with its own event pair, L2 flushed",
                    "algorithmic_bytes_per_launch": step_bytes,
                    "unfused_path": unfused,
                    "note": "NMS is O(K^2) IoU work on SM ALUs/LSU, not a streaming kernel; frac is bytes/time as the spec asks"}

    # ---- end to end through the public API with pinned host tensors
    loc_h, conf_h, pri_h = (torch.from_numpy(a).pin_memory() for a in (loc_np, conf_np, pri_np))
    IN_FLIGHT = int(os.environ.get("FDT_BENCH_IN_FLIGHT", "2"))

    def e2e_stream(steps):
        """`steps` batches through Detect.submit with IN_FLIGHT of them in flight; every batch's copies, kernels and results are
        inside the caller's timed region (the queue is empty before and after)."""
        pend = collections.deque()
        last = None
        for _ in range(steps):
            pend.append(det.submit(loc_h, conf_h, pri_h))
            if len(pend) > IN_FLIGHT:
                last = pend.popleft().result()
        while pend:
            last = pend.popleft().result()
        return last

    for _ in range(5):
        o = det(loc_h, conf_h, pri_h)
    e2e_stream(5)
    e2e_steps = max(20, min(args.steps, 100))
    if world > 1:
        dist.barrier()
    per = []
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        t1 = time.perf_counter()
        o = det(loc_h, conf_h, pri_h)                   # returns after the detections landed in host memory
        per.append(time.perf_counter() - t1)
    sync_dt = time.perf_counter() - t0
    if world > 1:
        dist.barrier()
    # like the device-timed value: the block of e2e_steps batches is repeated and the MEDIAN repeat is reported (the host side of
    # this path -- PCIe, the CPU that enqueues the copies -- takes a while to settle on a fresh box)
    E2E_REPEATS = 7
    e2e_dts = []
    for _ in range(E2E_REPEATS):
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        o = e2e_stream(e2e_steps)
        e2e_dts.append(time.perf_counter() - t0)
    if world > 1:
        t = torch.tensor(e2e_dts + [sync_dt], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)              # every repeat: max over ranks
        e2e_dts, sync_dt = [float(x) for x in t[:-1].tolist()], float(t[-1].item())
    e2e_dt = float(statistics.median(e2e_dts))
    # the host's pinned H2D rate in this run: what bounds e2e from below
    h2d_bytes = int(conf_h.numel() * 4)
    stage_dev = torch.empty_like(conf_h, device=dev)
    stage_dev.copy_(conf_h, non_blocking=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(10):
        stage_dev.copy_(conf_h, non_blocking=True)
    torch.cuda.synchronize()
    h2d_gbs = 10 * conf_h.numel() * 4 / (time.perf_counter() - t0) / 1e9
    floor_ms = h2d_bytes / (h2d_gbs * 1e9) * 1e3
    e2e = {"value": world * B * e2e_steps / e2e_dt, "unit": "frames/s",
           "h2d_bytes_per_step": h2d_bytes,
           "h2d_note": "conf is copied (cudaMemcpyAsync from pinned memory, chunks of 16 images overlapping the kernels); the pinned loc tensor "
                       "(%d bytes) is NOT copied: k_sort_nms gathers only the rows NMS decodes (<= 1024 x 16 B per image and round) from host "
                       "memory over PCIe; the prior set (%d bytes, a constant of the model) is uploaded once and stays resident" % (int(loc_h.numel() * 4), int(pri_h.numel() * 4)),
           "host_input_bytes_per_step": int(loc_h.numel() * 4 + conf_h.numel() * 4),
           "d2h_bytes_per_step": int(o.numel() * 4), "steps": e2e_steps, "ms_per_step": 1e3 * e2e_dt / e2e_steps,
           "in_flight": IN_FLIGHT,
           "repeats_ms_per_step": [1e3 * d / e2e_steps for d in e2e_dts], "reported": "median repeat",
           "sync_call": {"value": world * B * e2e_steps / sync_dt, "ms_per_step": 1e3 * sync_dt / e2e_steps,
                         "ms_per_step_median": 1e3 * statistics.median(per), "ms_per_step_max": 1e3 * max(per),
                         "api": "fdt_b200.layers.Detect.__call__(pinned CPU tensors) -> fdt_detect_host (one batch at a time: submit + wait)"},
           "pinned_h2d_gbs_this_host": h2d_gbs, "pcie_floor_ms": floor_ms,
           "frac_of_pcie_floor": floor_ms / (1e3 * e2e_dt / e2e_steps),
           "scope": "single-process public API" if world == 1 else "per-rank, no gather (every rank runs Detect on host tensors independently)",
           "api": "fdt_b200.layers.Detect.submit(pinned CPU tensors).result() -> fdt_detect_host_submit / _wait, %d batches in flight "
                  "(a stream of video batches); wall clock over all %d batches of a repeat, queue empty at both ends" % (IN_FLIGHT, e2e_steps)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        if gather_check == "MISMATCH":
            sys.exit(3)
        return

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        fps, n, dt, cores = cpu_oracle_rate(loc_np, conf_np, pri_np, budget_s=10.0, early_exit=False)
        cpu = {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
               "sample": f"{n} images ({n // B} x the B={B} batch) in {dt:.1f} s, C oracle port with OpenMP over images, "
                         f"NMS run to completion as box_utils.nms does (the reference itself is a Python loop, ~1-2 frames/s)"}
    secondary = None
    if world == 1 and not args.no_secondary:
        del sets
        secondary = secondary_workloads(torch, dev, flush, peak)

    launches_per_step = 2 + (1 if (world > 1 and peer is not None and peer.signal == "kernel") else 0)
    line = {"metric": METRIC,
            "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args.mode, world),
            "l2": f"inputs larger than L2: {ROTATE} rotating input sets per GPU ({ROTATE * 54.9:.0f} MB > 126 MB), steps issued back to back on one stream",
            "timing": {"steps": args.steps, "ms": total_ms,
                       "how": "one CUDA-event pair around the K steps on the launching stream, barrier + synchronize on both sides, "
                              "max over ranks", "workspace_depth": depth,
                       "overlap": "consecutive calls overlap on the device (workspace ring of `depth` slots; completion in stream order)"},
            "latency": {"ms_per_step": lat_ms, "frames_per_s": world * B / (lat_ms * 1e-3), "steps": n_lat,
                        "how": "each step alone with its own event pair; 256 MiB L2 flush + 0.1 ms GPU spin before it (outside the pair)"},
            "clocks": sampler.result(), "e2e": e2e,
            "gpu_launches": launches_per_step * args.steps,      # k_detect_begin, k_sort_nms<fused> (+ k_gather_await on rank 0)
            "gpu_launches_per_step": launches_per_step,
            "wall_s_timed_region": wall}
    if world > 1:
        line["gather"] = GATHER_NOTE[gather]
        line["gather_check"] = gather_check
    if roofline:
        line["roofline"] = roofline
    if cpu:
        line["cpu_baseline"] = cpu
    if secondary:
        line["secondary"] = secondary
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    if gather_check == "MISMATCH":
        sys.exit(3)


if __name__ == "__main__":
    main()
