"""Whole-program device time of the four conv programs (CUDA events around `reps` back-to-back runs, no per-op
events in between, so programmatic dependent launch can overlap consecutive kernels).
Usage: python scripts/prog_times.py [B] [reps]"""
import sys

import torch

sys.path.insert(0, ".")
import bench
from oracle import weights as OW
from padel_analytics_b200 import synth

B = int(sys.argv[1]) if len(sys.argv) > 1 else 32
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
ckpts = {k: OW.make_yolo(k) for k in ("detect", "pose13", "court12")}
ckpts["tracknet"] = OW.make_tracknet()
tr, med = bench.build_trackers(B, (1080, 1920), ckpts, "cuda")
fr = synth.make_frames(B, 1080, 1920, device="cuda")
for k in ("players", "pose", "court"):
    tr[k].detect_sample(fr)
progs = {"ball": tr["ball"].tracknet.prog}
for k in ("players", "pose", "court"):
    progs[k] = list(tr[k].model._progs.values())[0]["prog"]
print("B", B)
for name, p in progs.items():
    for _ in range(3):
        p.run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        p.run()
    e1.record()
    torch.cuda.synchronize()
    print(f"{name:8s} {e0.elapsed_time(e1) / reps:8.3f} ms per program run ({p.num_ops} ops)", flush=True)
