#!/usr/bin/env python
"""Headline benchmark: frames/sec through the four trackers (BASELINE.json metric) on synthetic frames.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|eager] [--config all4|players|pose|court|ball]
                  [--batch B] [--res 1080p|4k|720p] [--strong [--frames N]] [--dump-outputs DIR]

One *step* = one batch of `--batch` frames through the hot path of the selected trackers (default all four:
PlayerTracker YOLOv8n-detect, PlayerKeypointsTracker YOLOv8n-pose 13x3 @1280, KeypointsTracker YOLOv8n-pose 12x3 @640,
BallTracker TrackNet 27->8).  BASELINE.json configs: [1] = default; [2] = --config pose --batch 128;
[3] = --config ball --batch 256 under torchrun on 2 GPUs; [4] = --res 4k --batch 64 under torchrun on 8 GPUs.
N > 1 (torchrun, one rank per GPU): every rank runs its own shard of frames (weak scaling, no data-path collective;
NCCL only broadcasts the weights at init and gathers detection counts at the end).
--strong: a FIXED job of --frames frames goes through `TrackingRunner.run()` (the reference's entry point) sharded over the
ranks by contiguous ranges, with the result all_gather and the rank-0 host stages (polygon filter, ByteTrack, result
objects) INSIDE the timed region ("scaling": "strong").

Printed JSON (rank 0, one line): value (device-resident frames), e2e (pinned host frames through the tracker API, H2D
and result D2H inside the timed region), roofline (dominant kernel, event-timed live), cpu_baseline (the CPU oracle on
this box's host cores, bounded sample), clocks.  `--impl reference` times that CPU oracle as the main arm (the
reference's own Python path cannot travel to the GPU box: ultralytics/supervision are not installed anywhere; oracle/
restates it -- DESIGN.md, oracle).  `--impl eager` times the same oracle networks in PyTorch eager mode on the GPU
(cuDNN, TF32: the reference's own GPU numerics and the library baseline for the conv kernels).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

RES = {"1080p": (1080, 1920), "4k": (2160, 3840), "720p": (720, 1280)}


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(tflops_burst=d.get("bf16_tflops"), tflops_sustained=d.get("bf16_tflops_sustained"),
                    hbm_gbs=d.get("hbm_gbs"), source="measured")
    return dict(tflops_burst=1590.0, tflops_sustained=1400.0, hbm_gbs=6650.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])), mx.append(float(r[2]))
            except Exception:  # noqa: BLE001
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------------------
CONFIGS = {  # --config -> tracker names (bench keys)
    "all4": ("players", "pose", "court", "ball"), "players": ("players",), "pose": ("pose",), "court": ("court",),
    "ball": ("ball",),
}
KIND = {"players": "detect", "pose": "pose13", "court": "court12", "ball": "tracknet"}
YOLO_ARGS = {"detect": (640, 0.5, [0], 300), "pose13": (1280, 0.25, [0], 300), "court12": (640, 0.5, None, 12)}
METRIC = "frames/sec through trackers.runner (all 4 trackers)"


def workload_name(args, world):
    names = {"all4": "all four trackers", "players": "PlayerTracker (YOLOv8n-detect) only",
             "pose": "PlayerKeypointsTracker (YOLOv8n-pose 13x3 @1280) only",
             "court": "KeypointsTracker (YOLOv8n-pose 12x3 @640) only", "ball": "BallTracker (TrackNet 27->8) only"}
    base = {("all4", "1080p", 32): "configs[1]", ("pose", "1080p", 128): "configs[2]", ("ball", "1080p", 256): "configs[3]",
            ("all4", "4k", 64): "configs[4]"}.get((args.config, args.res, args.batch), "variant")
    return (f"{names[args.config]}, synthetic {args.res} frames, batch_size={args.batch} per GPU (BASELINE.json {base}); "
            f"YOLOv8n detect@384x640 + pose13x3@1280 + court12x3@640 + TrackNet 27->8@288x512 as selected, seeded "
            f"random weights")


# ------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle (port of the reference's CPU path) on the host cores, bounded sample
# ------------------------------------------------------------------------------------------------------------
def cpu_threads() -> int:
    """Threads given to the CPU oracle: every host core up to 64 (beyond that PyTorch's CPU convolutions on these
    small networks get slower, not faster)."""
    return max(1, min(os.cpu_count() or 1, 64))


class CpuOracle:
    """The reference's CPU path for the selected trackers: oracle networks + the reference's own pre-processing calls
    (cv2 / PIL), built once; `step(n)` pushes n frames through every selected tracker (ball: n + 7 frames = n windows)
    and returns seconds per frame per tracker."""

    def __init__(self, hw, trackers, seed=1234, nmax=8):
        from oracle import tracknet as OT
        from oracle import weights as OW
        from oracle import yolov8 as OY
        from padel_analytics_b200 import synth

        torch.set_num_threads(cpu_threads())
        self.OT, self.hw, self.trackers = OT, hw, trackers
        H, W = hw
        self.frames = [f.numpy() for f in synth.make_frames(nmax + 7, H, W, seed=seed)]
        self.yolo = {k: OY.YOLO(OW.load_yolo(OW.make_yolo(KIND[k]))) for k in trackers if k != "ball"}
        if "ball" in trackers:
            self.net = OW.load_tracknet(OW.make_tracknet())
            self.med = synth.make_median(H, W, seed=seed).numpy()

    @torch.no_grad()
    def step(self, n):
        import cv2
        from PIL import Image

        per = {}
        H, W = self.hw
        for k in self.trackers:
            t0 = time.perf_counter()
            if k == "ball":
                self.OT.run_ball_oracle(self.net, self.frames[:n + 7], self.med, (W, H), batch_size=min(n, 8))
            else:
                imgsz, conf, classes, max_det = YOLO_ARGS[KIND[k]]
                if k == "players":  # players_tracker.py:346-359
                    sample = [cv2.cvtColor(f, cv2.COLOR_BGR2RGB) for f in self.frames[:n]]
                else:  # players_keypoints_tracker.py:260-292 / keypoints_tracker.py:190-245
                    sample = [Image.fromarray(cv2.cvtColor(f, cv2.COLOR_BGR2RGB)).resize((imgsz, imgsz))
                              for f in self.frames[:n]]
                self.yolo[k].predict(sample, conf=conf, iou=0.7, imgsz=imgsz, classes=classes, max_det=max_det)
            per[k] = (time.perf_counter() - t0) / n
        return per


def run_reference_arm(args, rank, world):
    """`--impl reference`: the CPU oracle on the host cores, same config / metric / unit.  Per step every selected
    tracker processes 8 frames at batch 8 (the reference's default batch sizes, config.py:23,31,38,45) -- ball: 15 frames
    = 8 windows; frames/s = 1 / sum over trackers of seconds per frame, like the GPU arm's single pass over all of
    them.  Rank 0 alone runs; the other ranks exit."""
    if rank != 0:
        return
    n = 8
    ora = CpuOracle(RES[args.res], CONFIGS[args.config], nmax=n)
    for _ in range(min(args.warmup, 1)):
        ora.step(n)
    vals, pers = [], []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        per = ora.step(n)
        pers.append(per)
        vals.append(1.0 / sum(per.values()))
    dt = time.perf_counter() - t0
    v = statistics.median(vals)
    per = {k: round(statistics.median(p[k] for p in pers), 4) for k in pers[0]}
    sample = (f"per step: {n} frames per selected YOLO tracker at batch {n} + {n + 7} frames ({n} windows) ball; "
              f"per-frame times summed over the trackers; median of {args.steps} steps")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(v, 4), "unit": "frames/s", "n_gpus": 0,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt / args.steps * 1e3, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args, 1) + " -- CPU oracle (port of the reference's CPU path)",
                   "per_frame_s": per, "value_spread": [round(min(vals), 4), round(max(vals), 4)]},
        "cpu_baseline": {"value": round(v, 4), "unit": "frames/s", "cores": cpu_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": round(v, 4), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), file=JSON_OUT, flush=True)


def run_eager_arm(args, rank, world):
    """`--impl eager`: the oracle networks (what ultralytics / the reference's TrackNet run) in PyTorch eager mode on
    one B200 with cuDNN TF32 convolutions -- the reference's own GPU numerics, and the library baseline the hand-written
    conv kernels are measured against.  Timed per step: network forward (+ torchvision NMS for the YOLO heads) of every
    selected tracker on a resident, already pre-processed batch (the reference pre-processes on the CPU: cv2 / PIL)."""
    if rank != 0:
        return
    import cv2
    from PIL import Image

    from oracle import tracknet as OT
    from oracle import weights as OW
    from oracle import yolov8 as OY
    from padel_analytics_b200 import synth

    dev = torch.device("cuda", 0)
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.benchmark = True
    B, (H, W) = args.batch, RES[args.res]
    trackers = CONFIGS[args.config]
    frames = [f.numpy() for f in synth.make_frames(8, H, W)]
    work = []
    for k in trackers:
        if k == "ball":
            net = OW.load_tracknet(OW.make_tracknet()).to(dev)
            xw = torch.from_numpy(OT.assemble_windows(frames[:8], synth.make_median(H, W).numpy())).float()
            x = xw[:1].repeat(B, 1, 1, 1).to(dev)
            work.append((k, lambda net=net, x=x: net(x), 227.606e9))
        else:
            imgsz, conf, classes, max_det = YOLO_ARGS[KIND[k]]
            net = OW.load_yolo(OW.make_yolo(KIND[k], cls_mean={"players": -5.0, "pose": -5.7, "court": None}[k])).to(dev)
            yolo = OY.YOLO(OW.load_yolo(OW.make_yolo(KIND[k])))
            sample = ([cv2.cvtColor(f, cv2.COLOR_BGR2RGB) for f in frames[:1]] if k == "players" else
                      [Image.fromarray(cv2.cvtColor(f, cv2.COLOR_BGR2RGB)).resize((imgsz, imgsz)) for f in frames[:1]])
            yolo.predict(sample, conf=conf, iou=0.7, imgsz=imgsz, classes=classes, max_det=max_det)
            x = yolo.last_preprocessed.repeat(B, 1, 1, 1).to(dev)
            nc = net.nc
            work.append((k, lambda net=net, x=x, conf=conf, classes=classes, max_det=max_det, nc=nc:
                         OY.non_max_suppression(net(x), conf, 0.7, classes, max_det, nc), None))
    per = {}
    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            for _, fn, _ in work:
                fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(args.steps):
            for _, fn, _ in work:
                fn()
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        for k, fn, _ in work:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(3):
                fn()
            b.record()
            torch.cuda.synchronize()
            per[k] = round(a.elapsed_time(b) / 3, 3)
    ms = max(e0.elapsed_time(e1), wall * 1e3) / args.steps
    v = B / (ms / 1e3)
    print(json.dumps({
        "impl": "eager", "metric": METRIC, "value": round(v, 2), "unit": "frames/s", "n_gpus": 1, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 storage, TF32 convolutions (cuDNN, torch defaults)", "data": "synthetic",
        "config": {"workload": workload_name(args, 1) + " -- PyTorch eager CUDA (cuDNN) of the oracle networks + "
                               "torchvision NMS on a resident pre-processed batch",
                   "ms_per_model": per},
        "gpu_launches": 0,
    }), file=JSON_OUT, flush=True)


# ------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------
def build_trackers(B, hw, ckpts, dev, which=("players", "pose", "court", "ball")):
    from padel_analytics_b200 import synth
    from padel_analytics_b200.trackers import BallTracker, KeypointsTracker, PlayerKeypointsTracker, PlayerTracker
    from padel_analytics_b200.trackers import sv_compat as sv

    H, W = hw
    vi = sv.VideoInfo(width=W, height=H, fps=30.0, total_frames=None)
    poly = sv.PolygonZone(np.array([[W // 10, H // 10], [9 * W // 10, H // 10], [9 * W // 10, 9 * H // 10],
                                    [W // 10, 9 * H // 10]]), frame_resolution_wh=(W, H))
    med = synth.make_median(H, W).numpy()
    make = {
        "players": lambda: PlayerTracker(ckpts["detect"], poly, batch_size=B),
        "pose": lambda: PlayerKeypointsTracker(ckpts["pose13"], 1280, batch_size=B, load_path=None, save_path=None),
        "court": lambda: KeypointsTracker(ckpts["court12"], batch_size=B, model_type="yolo"),
        "ball": lambda: BallTracker(ckpts["tracknet"], None, batch_size=B, median=med),
    }
    tr = {k: make[k]() for k in which}
    for t in tr.values():
        t.video_info_post_init(vi)
    return tr, med


# The contract is ONE JSON line on stdout: everything else this process prints (tracker banners, library chatter)
# is sent to stderr, the JSON line goes to the real stdout.
JSON_OUT = sys.stdout


def make_ckpts(which, rank, world, dev):
    """Seeded synthetic checkpoints, generated on rank 0 and broadcast over NCCL (the only init-time collective)."""
    import torch.distributed as dist

    from oracle import weights as OW

    ckpts = None
    if rank == 0:
        # sparse heads: a handful of players per frame like a real padel rally (the dense defaults are for parity tests)
        mk = {"detect": lambda: OW.make_yolo("detect", cls_mean=-5.0), "pose13": lambda: OW.make_yolo("pose13", cls_mean=-5.7),
              "court12": lambda: OW.make_yolo("court12"), "tracknet": OW.make_tracknet}
        # the heads are standardised with CPU convolutions whose last bits depend on the thread count: one thread makes
        # the weights, and so every output, the same on any host
        threads = torch.get_num_threads()
        torch.set_num_threads(1)
        try:
            ckpts = {KIND[k]: mk[KIND[k]]() for k in which}
        finally:
            torch.set_num_threads(threads)
    if world > 1:
        box = [ckpts]
        dist.broadcast_object_list(box, src=0, device=dev)
        ckpts = box[0]
    return ckpts


DUMP_BYTES = 64 << 20


def dump_outputs(out, path: Path):
    """What a caller of the fused pass receives for one batch, as float64 tables with one row per object, written to
    path/<tracker>.npy.  `frame` is the index within the batch (ball: the tracker's frame number).
      players: frame, x1, y1, x2, y2, confidence, class_id, tracker id (-1: none)
      pose:    frame, then x, y of the 13 keypoints of one player
      court:   frame, then x, y of the 12 keypoints ordered by id
      ball:    frame, x, y, visibility
    Tables above DUMP_BYTES together keep the same seeded sample of rows on every run."""
    rows = {
        "players": [[f, *p.xyxy, p.confidence, p.class_id, -1 if p.id is None else p.id]
                    for f, ps in enumerate(out.get("players", [])) for p in ps],
        "pose": [[f, *(v for k in pk.player_keypoints for v in k.xy)]
                 for f, pks in enumerate(out.get("pose", [])) for pk in pks],
        "court": [[f, *(v for k in kps.keypoints for v in k.xy)] for f, kps in enumerate(out.get("court", [])) if len(kps)],
        "ball": [[f, *xyv] for f, xyv in out.get("ball", {}).items()],
    }
    width = {"players": 8, "pose": 27, "court": 25, "ball": 4}
    tables = {k: np.array(v, dtype=np.float64).reshape(-1, width[k]) for k, v in rows.items() if k in out}
    total = sum(t.nbytes for t in tables.values())
    if total > DUMP_BYTES:
        rng = np.random.default_rng(0)
        tables = {k: t[np.sort(rng.choice(len(t), len(t) * DUMP_BYTES // total, replace=False))]
                  for k, t in tables.items()}
    path.mkdir(parents=True, exist_ok=True)
    for k, t in tables.items():
        np.save(path / f"{k}.npy", t)


def run_strong(args, rank, world, local, dev):
    """--strong: a fixed job of args.frames frames through TrackingRunner.run() -- contiguous shards, ball halo,
    fixed-capacity all_gather, rank-0 polygon filter + ByteTrack + result objects -- all inside the timed region."""
    import torch.distributed as dist

    from padel_analytics_b200 import _lib as L
    from padel_analytics_b200 import synth
    from padel_analytics_b200.trackers import TrackingRunner
    from padel_analytics_b200.trackers import sv_compat as sv
    from padel_analytics_b200.trackers.runner import ball_shard_frames, shard_range

    which = CONFIGS[args.config]
    B, (H, W), N = args.batch, RES[args.res], args.frames
    ckpts = make_ckpts(which, rank, world, dev)
    NB = 4  # distinct pinned batches the synthetic "video" cycles through
    pool = [synth.make_frames(B, H, W, start=i * B, device=dev).cpu().pin_memory() for i in range(NB)]

    def source(lo, hi):  # ready (n,H,W,3) pinned batches covering frames lo..hi-1 (content cycles, length exact)
        pos, i = lo, 0
        while pos < hi:
            n = min(B, hi - pos)
            yield pool[i % NB][:n]
            pos, i = pos + n, i + 1

    tr, _ = build_trackers(B, (H, W), ckpts, dev, which)  # engines are built once, like loading the models once
    run = TrackingRunner(list(tr.values()), video_info=sv.VideoInfo(width=W, height=H, fps=30.0, total_frames=N))

    def one_pass():
        run.restart()  # empty results, ByteTrack reset: run() would skip trackers that already hold predictions
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        l0 = L.lib().pb_launch_count()
        t0 = time.perf_counter()
        tm = dict(run.run(frame_source=source, total_frames=N))
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([wall], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.barrier()
            wall = t.item()
        nobj = sum(len(t.results) for t in tr.values())
        return wall, tm, L.lib().pb_launch_count() - l0, nobj

    one_pass()  # warm-up: kernels, tensor maps, allocator
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    walls, tms, launches, nobj = [], [], 0, 0
    for _ in range(args.steps):
        w_, tm, launches, nobj = one_pass()
        walls.append(w_)
        tms.append(tm)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        wall = statistics.median(walls)
        tm = tms[walls.index(sorted(walls)[len(walls) // 2])]
        lo, hi = shard_range(N, 0, world)
        flo, fhi = ball_shard_frames(N, lo, hi)
        print(json.dumps({
            "metric": METRIC, "value": round(N / wall, 2), "unit": "frames/s", "n_gpus": world, "steps": len(walls),
            "warmup": 1, "ms_per_step": round(wall * 1e3, 2), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f16 storage, f32 accumulate", "data": "synthetic",
            "config": {"workload": workload_name(args, world) + f"; STRONG scaling: one fixed job of {N} frames through "
                                   f"TrackingRunner.run(), a step = the whole job",
                       "frames": N, "parallelism": f"contiguous frame shards over {world} GPU(s); all_gather of "
                                                   f"fixed-capacity detection records; rank-0 host stages inside the timed region",
                       "rank0_frames_read": fhi - flo, "objects_assembled_on_rank0": nobj,
                       "rank0_seconds": {k: round(v, 4) for k, v in tm.items() if k.startswith("_")},
                       "l2": "inputs (%d MB/batch) and activations exceed L2; no flush" % (B * H * W * 3 // 1000000)},
            "e2e": {"value": round(N / wall, 2), "unit": "frames/s", "h2d_bytes_per_step": (fhi - flo) * H * W * 3,
                    "d2h_bytes_per_step": None,
                    "note": "this mode IS end to end: pinned host batches in, result objects out, wall clock"},
            "gpu_launches": int(launches), "clocks": clocks,
        }), file=JSON_OUT, flush=True)


def main():
    sys.stdout = sys.stderr
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "eager"])
    ap.add_argument("--config", default="all4", choices=list(CONFIGS))
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--res", default="1080p", choices=list(RES))
    ap.add_argument("--strong", action="store_true", help="fixed job through TrackingRunner.run(), gather inside the timing")
    ap.add_argument("--frames", type=int, default=4096, help="--strong: frames of the fixed job")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-host", action="store_true", help="cProfile the timed region's host side (stderr)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the tracker outputs of the last timed step as DIR/<tracker>.npy (float64 tables)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.strong):
        ap.error("--dump-outputs covers the default fused pass only (--impl ours, no --strong)")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if args.impl == "eager":
        run_eager_arm(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch.distributed as dist

    # The only oracle import of the product arm: oracle.weights CONSTRUCTS the seeded synthetic checkpoints (a stand-in
    # for torch.load of real .pt files, none of which exist offline) before anything is timed.  No oracle code computes
    # anything inside the warm-up or timed regions; the trackers below run on libpadel_b200.so only.
    from padel_analytics_b200 import _lib as L
    from padel_analytics_b200 import synth
    from padel_analytics_b200.engine import ops

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    if args.strong:
        run_strong(args, rank, world, local, dev)
        if world > 1:
            dist.destroy_process_group()
        return

    which = CONFIGS[args.config]
    ckpts = make_ckpts(which, rank, world, dev)
    B = args.batch
    hw = RES[args.res]
    H, W = hw
    trackers, med = build_trackers(B, hw, ckpts, dev, which)
    ball = trackers.get("ball")

    # frames: NBUF distinct batches resident in HBM (+ pinned host copies for the e2e leg); each batch (B*H*W*3 bytes
    # = 199 MB at 1080p/32) alone exceeds the 126 MB L2 and activations are GBs, so no L2 flush is needed.
    NBUF = 3
    dev_batches = [synth.make_frames(B, H, W, start=rank * 100000 + i * B, device=dev) for i in range(NBUF)]
    host_batches = [b.cpu().pin_memory() for b in dev_batches]
    from padel_analytics_b200.trackers.runner import FusedPass

    # The measured path is the fused single pass (trackers/runner.py::FusedPass, what TrackingRunner.run() takes): one
    # upload per batch shared by the selected trackers, their device work enqueued back to back, host post-processing
    # overlapped.
    fused = FusedPass(trackers, hw, B, total_frames=10 ** 9)  # steady state: the tail flush is never reached
    if ball is not None:
        ball._pipe.push_frames(dev_batches[0][:7])  # prime the 8-frame window so every step yields B windows

    def run_steps(batches, steps):
        nd, out = 0, None
        for out in fused.run(batches[i % NBUF] for i in range(steps)):
            nd += sum(len(p) for k in ("players", "pose") if k in out for p in out[k])
        return nd, out

    import gc

    def timed(batches, steps):
        gc.collect()
        gc.freeze()  # keep the (large, static) engine object graph out of the cyclic collector's way
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = L.lib().pb_launch_count()
        t0 = time.perf_counter()
        e0.record()
        if os.environ.get("PADEL_B200_NCU") == "1":  # `ncu --profile-from-start off`: capture the timed region only
            torch.cuda.profiler.start()
        nd, out = run_steps(batches, steps)
        if os.environ.get("PADEL_B200_NCU") == "1":
            torch.cuda.synchronize()
            torch.cuda.profiler.stop()
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms, wall * 1e3], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.barrier()
            ms, wall = t[0].item(), t[1].item() / 1e3
        return ms, wall, L.lib().pb_launch_count() - l0, nd, out

    run_steps(dev_batches, args.warmup)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if args.profile_host:
        import cProfile
        import pstats

        pr = cProfile.Profile()
        pr.enable()
    ms_dev, wall_dev, launches, ndet, last = timed(dev_batches, args.steps)
    if args.profile_host:
        pr.disable()
        pstats.Stats(pr, stream=sys.stderr).sort_stats("cumulative").print_stats(35)
    if args.dump_outputs and rank == 0:
        dump_outputs(last, Path(args.dump_outputs))
    run_steps(host_batches, 2)
    ms_e2e, wall_e2e, _, _, _ = timed(host_batches, args.steps)
    clocks = sampler.stop() if rank == 0 else None

    frames_total = B * args.steps * world
    value = frames_total / (max(ms_dev, wall_dev * 1e3) / 1e3)
    e2e = frames_total / (max(ms_e2e, wall_e2e * 1e3) / 1e3)

    # roofline of the dominant kernel: algorithmic FLOPs of every conv launch of one step divided by the event-timed
    # duration of those launches (per-op CUDA events on the launch stream, median of 5 repeats, rank 0 only)
    roof = None
    if rank == 0:
        progs = []
        if ball is not None:
            progs.append(("tracknet", ball.tracknet.prog))
        for k in ("players", "pose", "court"):
            if k in trackers:
                for st in trackers[k].model._progs.values():
                    progs.append((k, st["prog"]))
        per_kernel = {}
        per_model = {}
        all_ms = 0.0
        for name, p in progs:
            t = ops.time_program_ops(p, repeats=5)
            kn = p.op_kernels()
            for ti, k, f, by in zip(t, kn, p.flops, p.bytes):
                e = per_kernel.setdefault(k, {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "launches": 0})
                e["ms"] += ti
                e["flops"] += f
                e["bytes"] += by
                e["launches"] += 1
            cm = sum(ti for ti, kd in zip(t, p.kinds) if kd == "conv")
            cf = sum(f for f, kd in zip(p.flops, p.kinds) if kd == "conv")
            all_ms += sum(t)
            for _ in range(2):
                p.run()
            torch.cuda.synchronize()
            pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            pe0.record()
            for _ in range(5):
                p.run()
            pe1.record()
            torch.cuda.synchronize()
            per_model[name] = {"conv_ms": round(cm, 3), "all_ops_ms": round(sum(t), 3),
                               "program_ms_back_to_back": round(pe0.elapsed_time(pe1) / 5, 3),
                               "gflop_per_frame": round(cf / B / 1e9, 3), "tflops": round(cf / cm / 1e9, 1)}
        pk = _peaks()
        dom = max((k for k in per_kernel if k.startswith("conv")), key=lambda k: per_kernel[k]["ms"])
        d = per_kernel[dom]
        achieved = d["flops"] / (d["ms"] / 1e3) / 1e12
        conv_ms = sum(v["ms"] for k, v in per_kernel.items() if k.startswith("conv"))
        conv_fl = sum(v["flops"] for k, v in per_kernel.items() if k.startswith("conv"))
        traffic = None
        for cand in ("r02_tracknet_dram_bytes.json", "r01_tracknet_dram_bytes.json"):
            tf = ROOT / "profiles" / cand
            if tf.exists() and dom == "conv_halo_kernel" and ball is not None:
                traffic = json.loads(tf.read_text())
                break
        roof = {"bound": "tensor", "kernel": dom, "achieved": round(achieved, 1), "peak": pk["tflops_sustained"],
                "peak_kind": f"{pk['source']} cuBLAS bf16 sustained (fp16 runs at the same tensor-core rate)",
                "unit": "TFLOP/s", "frac": round(achieved / pk["tflops_sustained"], 4),
                "traffic": (traffic or {}).get("dram_gb_per_step_tracknet_halo_launches"),
                "traffic_note": (traffic or {}).get("note"),
                "launches_per_step": d["launches"], "kernel_ms_per_step": round(d["ms"], 3),
                "timing": "median of 5 per-op CUDA-event timings",
                "algorithmic_gflop_per_step": round(d["flops"] / 1e9, 1),
                "algorithmic_act_gb_per_step": round(d["bytes"] / 1e9, 2),
                "all_conv_kernels": {"ms_per_step": round(conv_ms, 3), "tflops": round(conv_fl / conv_ms / 1e9, 1),
                                     "frac": round(conv_fl / conv_ms / 1e9 / pk["tflops_sustained"], 4)},
                "program_ms_per_step": round(all_ms, 3),
                "per_kernel": {k: {"ms": round(v["ms"], 3), "launches": v["launches"],
                                   "tflops": round(v["flops"] / v["ms"] / 1e9, 1) if v["flops"] else 0.0,
                                   "gbs": round(v["bytes"] / v["ms"] / 1e6, 1)} for k, v in per_kernel.items()},
                "per_model": per_model}

    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        ora = CpuOracle(hw, which, nmax=4)
        ora.step(1)
        per = ora.step(4)
        cpu = {"value": round(1.0 / sum(per.values()), 4), "unit": "frames/s", "cores": cpu_threads(), "kind": "port",
               "sample": "4 frames per selected YOLO tracker (batch 4) + 11 frames (4 windows) ball on the host cores, "
                         "after one warm-up frame; per-frame times summed over the trackers",
               "per_frame_s": {k: round(v, 4) for k, v in per.items()}}

    if world > 1:
        cnt = torch.tensor([ndet], device=dev)
        gathered = [torch.zeros_like(cnt) for _ in range(world)]
        dist.all_gather(gathered, cnt)  # detection counts gathered to every rank (tiny)
        ndet = int(sum(int(g.item()) for g in gathered))

    if rank == 0:
        h2d = B * H * W * 3  # one pinned-host -> device upload per batch, shared by the selected trackers
        d2h = sum(int(np.prod(st[k]["host"][0][0].shape)) * 4 for t in ("players", "pose", "court") if t in trackers
                  for st in trackers[t].model._progs.values() for k in st if isinstance(k, tuple))
        d2h += (B + 7) * 16 if ball is not None else 0
        print(json.dumps({
            "metric": METRIC, "value": round(value, 2),
            "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(max(ms_dev, wall_dev * 1e3) / args.steps, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16 storage, f32 accumulate", "data": "synthetic",
            "config": {"workload": workload_name(args, world),
                       "global_batch": B * world,
                       "l2": f"inputs ({h2d // 1000000} MB/batch) and activations exceed L2; no flush",
                       "parallelism": f"frames sharded over {world} GPU(s), no data-path collective",
                       "detections_in_timed_region": ndet,
                       "pass": "fused single pass (what TrackingRunner.run() takes): one upload per batch shared by the "
                               "selected trackers, one batch of look-ahead, YOLO chains on their own streams, native "
                               "ByteTrack / result objects on the host overlapped with the next batch"},
            "e2e": {"value": round(e2e, 2), "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": round(max(ms_e2e, wall_e2e * 1e3) / args.steps, 3)},
            "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu, "clocks": clocks,
            "timing": {"device_ms_per_step": round(ms_dev / args.steps, 3), "wall_ms_per_step": round(wall_dev * 1e3 / args.steps, 3),
                       "e2e_device_ms_per_step": round(ms_e2e / args.steps, 3),
                       "e2e_wall_ms_per_step": round(wall_e2e * 1e3 / args.steps, 3)},
        }), file=JSON_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
