"""Generate tests/golden/*.npz by running the UNMODIFIED reference code (only possible where /root/reference exists).

    python tests/golden/make_golden.py

ball_ref.npz  — the reference BallTracker.predict_frames TrackNet stage (ball_tracker.py:373-523) on 21 synthetic
                frames with a seeded TrackNet at a reduced heat-map size (HEIGHT=32, WIDTH=64 are class attributes the
                reference lets a subclass override): ensemble heat-maps fed to predict_modified and the x/y/visibility
                it returned, captured by wrapping `predict_modified`.  (predict_frames then dies with KeyError 'Frame',
                SURVEY App. E q6 — the TrackNet stage has completed by then.)
tracknet_ref.npz — reference TrackNet forward on one seeded input (models.py:45-74).
yolo_glue_ref.npz — the reference's OWN PlayerKeypointsTracker.predict_sample / KeypointsTracker.predict_sample /
                PlayerTracker.predict_sample (players_keypoints_tracker.py:271-322, keypoints_tracker.py:199-262,
                players_tracker.py:341-380) driven with the oracle YOLO as the `ultralytics.YOLO` stub, on the three
                rally.mp4 crops under tests/golden/rally/: what the reference's glue (processor, predict arguments,
                ratio scaling, id mapping, object construction) makes of a given model output.  ultralytics itself
                stays unpinned (absent); for PlayerTracker the `supervision` names are bound to this repo's sv_compat
                (supervision is absent too), so only the reference's own lines are pinned there.  The oracle YOLO
                results the glue was given are stored with it (oracle_*).
"""
import sys
import tempfile
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from oracle import ref_harness, weights as OW  # noqa: E402
from padel_analytics_b200 import synth  # noqa: E402

OUT = Path(__file__).resolve().parent
sys.path.insert(0, str(OUT.parent))
from fixtures import court_conf_for_single_detection, glue_ckpt, rally_frames  # noqa: E402


def main():
    ref_harness.import_reference()
    import trackers.ball_tracker.ball_tracker as rbt
    from trackers.ball_tracker.models import TrackNet

    torch.manual_seed(0)
    ck = OW.make_tracknet()
    with tempfile.TemporaryDirectory() as td:
        path = Path(td) / "tracknet.pt"
        torch.save(ck, path)

        class SmallBall(rbt.BallTracker):
            HEIGHT, WIDTH = 32, 64

        T, B, H, W = 21, 4, 90, 160
        frames = synth.make_frames(T, H, W, seed=7)
        med = synth.make_median(H, W, seed=7).numpy()
        bt = SmallBall(str(path), None, batch_size=B, median=med)
        bt.video_info_post_init(SimpleNamespace(width=W, height=H, fps=30))
        cap = {"ens": [], "x": [], "y": [], "vis": []}
        orig = rbt.predict_modified

        def spy(**kw):
            out = orig(**kw)
            cap["ens"].append(kw["y_pred"].clone())
            cap["x"] += out["x"]
            cap["y"] += out["y"]
            cap["vis"] += out["visibility"]
            return out

        rbt.predict_modified = spy
        try:
            bt.predict_frames((f.numpy() for f in frames), total_frames=T)
        except KeyError as e:  # q6
            assert str(e) == "'Frame'"
        finally:
            rbt.predict_modified = orig
        ens = torch.cat(cap["ens"])[:, 0].numpy()
        assert ens.shape[0] == T and len(cap["x"]) == T
        np.savez_compressed(OUT / "ball_ref.npz", ens=ens.astype(np.float32), x=np.array(cap["x"]),
                            y=np.array(cap["y"]), vis=np.array(cap["vis"]), T=T, B=B, H=H, W=W, seed=7,
                            net_h=32, net_w=64)
        print("ball_ref:", ens.shape, "visible frames", int(np.sum(cap["vis"])), list(zip(cap["x"], cap["y"]))[:8])

    # ---- InpaintNet stage (ball_tracker.py:525-673): the reference hard-codes .cuda(); redirect it to the CPU ----
    from oracle import inpaint as OI

    torch.Tensor.cuda = lambda self, *a, **k: self
    ick = OI.make_inpaintnet()
    with tempfile.TemporaryDirectory() as td:
        tpath, ipath = Path(td) / "tracknet.pt", Path(td) / "inpaint.pt"
        torch.save(ck, tpath)
        torch.save(ick, ipath)

        # default 288x512 heat-maps (COOR_TH depends on them); the TrackNet outputs are replaced by a crafted trajectory
        # with gaps so that the inpaint mask, the InpaintNet blend, both thresholds and the ensemble all do real work
        T, B, H, W = 44, 8, 360, 640
        frames = synth.make_frames(T, H, W, seed=9)
        med = synth.make_median(H, W, seed=9).numpy()
        bt = rbt.BallTracker(str(tpath), str(ipath), batch_size=B, median=med)
        bt.video_info_post_init(SimpleNamespace(width=W, height=H, fps=30))
        rng = np.random.default_rng(3)
        tx = (100 + 11 * np.arange(T) + rng.integers(-3, 4, T)).astype(int)
        ty = (120 + 60 * np.sin(np.arange(T) / 5.0) + rng.integers(-3, 4, T)).astype(int)
        tv = np.ones(T, dtype=int)
        for lo, hi in ((0, 3), (9, 13), (20, 21), (30, 37)):
            tv[lo:hi] = 0
        tx[tv == 0] = 0
        ty[tv == 0] = 0
        ty[26] = 10  # a visible point above the th_h line next to nothing
        cursor = {"n": 0}
        orig = rbt.predict_modified

        def fake(**kw):
            n = kw["y_pred"].shape[0]
            lo = cursor["n"]
            cursor["n"] += n
            return {"x": tx[lo:lo + n].tolist(), "y": ty[lo:lo + n].tolist(), "visibility": tv[lo:lo + n].tolist()}

        rbt.predict_modified = fake
        try:
            balls = bt.predict_frames((f.numpy() for f in frames), total_frames=T)
        finally:
            rbt.predict_modified = orig
        assert len(balls) == T and cursor["n"] == T
        np.savez_compressed(OUT / "inpaint_ref.npz", x=tx, y=ty, vis=tv,
                            X=np.array([b.xy[0] for b in balls]), Y=np.array([b.xy[1] for b in balls]),
                            V=np.array([b.visibility for b in balls]), T=T, B=B, H=H, W=W, seq_len=16,
                            net_h=288, net_w=512)
        print("inpaint_ref: tracknet vis", int(tv.sum()), "-> inpainted vis", int(sum(b.visibility for b in balls)),
              [b.xy for b in balls][:14])

    yolo_glue_golden()

    net = TrackNet(27, 8)
    net.load_state_dict(ck["model"])
    net.eval()
    g = torch.Generator().manual_seed(11)
    x = torch.rand((1, 27, 32, 64), generator=g)
    with torch.no_grad():
        y = net(x)
    np.savez_compressed(OUT / "tracknet_ref.npz", y=y.numpy(), seed=11)
    print("tracknet_ref:", y.shape, float(y.mean()))


def yolo_glue_golden():
    """Reference tracker classes (unmodified) + oracle YOLO -> tests/golden/yolo_glue_ref.npz."""
    import trackers.keypoints_tracker.keypoints_tracker as rkt
    import trackers.players_keypoints_tracker.players_keypoints_tracker as rpk
    import trackers.players_tracker.players_tracker as rpt
    from oracle import yolov8 as OY
    from padel_analytics_b200.trackers import sv_compat

    frames = rally_frames()
    H, W = frames[0].shape[:2]
    out = {"H": H, "W": W, "n": len(frames)}
    # the oracle YOLO results the reference glue consumed (oracle_<tracker>_{boxes,kpts}_<frame>): the test feeds them
    # to the product glue, whose exact comparison must not depend on how the host's CPU convolutions round
    calls = []
    predict = OY.YOLO.predict

    def spy(self, *a, **k):
        res = predict(self, *a, **k)
        calls.append([(r.boxes.data.numpy().copy(), None if r.keypoints is None else r.keypoints.data.numpy().copy())
                      for r in res])
        return res

    def keep(name, i, res):
        out[f"oracle_{name}_boxes_{i}"], kp = res
        if kp is not None:
            out[f"oracle_{name}_kpts_{i}"] = kp

    OY.YOLO.predict = spy
    with tempfile.TemporaryDirectory() as td:
        paths = {}
        for kind in ("detect", "pose13", "court12"):
            paths[kind] = str(Path(td) / f"{kind}.pt")
            torch.save(glue_ckpt(kind), paths[kind])
        # --- PlayerKeypointsTracker (needs >= 3 players per frame, SURVEY App. E q4)
        pk = rpk.PlayerKeypointsTracker(paths["pose13"], 640, batch_size=len(frames), load_path=None, save_path=None)
        preds = pk.predict_sample(frames)
        for i, p in enumerate(preds):
            arr = np.array([[kp.xy for kp in player.player_keypoints] for player in p.players_keypoints], dtype=np.float64)
            assert arr.shape[0] >= 3 and arr.shape[1:] == (13, 2), arr.shape
            out[f"pose_{i}"] = arr
            keep("pose", i, calls[-1][i])
        out["pose_names"] = np.array([kp.name for kp in preds[0].players_keypoints[0].player_keypoints])
        # --- KeypointsTracker: exactly one detection per frame (q5) -> per-frame CONF via a subclass attribute
        net = OW.load_yolo(glue_ckpt("court12"))
        confs = []
        for i, f in enumerate(frames):
            conf = court_conf_for_single_detection(net, f)
            confs.append(conf)
            cls = type("CourtOne", (rkt.KeypointsTracker,), {"CONF": conf})
            kt = cls(paths["court12"], batch_size=1, model_type="yolo")
            (kp,) = kt.predict_sample([f])
            keep("court", i, calls[-1][0])
            ks = sorted(kp.keypoints, key=lambda k: k.id)
            assert [k.id for k in ks] == list(range(12))
            out[f"court_{i}"] = np.array([k.xy for k in ks], dtype=np.float64)
        out["court_conf"] = np.array(confs)
        # --- PlayerTracker: supervision names bound to sv_compat (Detections.from_ultralytics, PolygonZone, ByteTrack)
        rpt.sv = sv_compat
        try:
            poly = sv_compat.PolygonZone(np.array([[0, 0], [W, 0], [W, H], [0, H]]),
                                         frame_resolution_wh=(W, H))
            pt = rpt.PlayerTracker(paths["detect"], poly, batch_size=len(frames))
            pt.video_info_post_init(sv_compat.VideoInfo(width=W, height=H, fps=25.0, total_frames=len(frames)))
            preds = pt.predict_sample(frames)
            for i, p in enumerate(preds):
                out[f"players_{i}"] = np.array([[*pl.xyxy, pl.confidence, pl.class_id, -1 if pl.id is None else pl.id]
                                                for pl in p.players], dtype=np.float64).reshape(-1, 7)
                keep("players", i, calls[-1][i])
        finally:
            rpt.sv = sys.modules["supervision"]
            OY.YOLO.predict = predict
    # --- KeypointsTracker(model_type="resnet") (keypoints_tracker.py:158-167,276-312): torchvision's resnet50 is
    # installed, only the `pretrained=True` download must be avoided (the state dict is loaded over it anyway)
    import torchvision
    from oracle import resnet as OR

    with tempfile.TemporaryDirectory() as td:
        rpath = str(Path(td) / "resnet.pt")
        torch.save(OR.make_resnet50_court(), rpath)
        orig_r50 = rkt.models.resnet50
        rkt.models.resnet50 = lambda pretrained=True: orig_r50(weights=None)
        try:
            kt = rkt.KeypointsTracker(rpath, batch_size=2, model_type="resnet")
            preds = kt.predict_frames(iter(frames))
        finally:
            rkt.models.resnet50 = orig_r50
        out["resnet"] = np.array([[k.xy for k in sorted(p.keypoints, key=lambda k: k.id)] for p in preds], dtype=np.float64)
        assert out["resnet"].shape == (len(frames), 12, 2)
    np.savez_compressed(OUT / "yolo_glue_ref.npz", **out)
    print("yolo_glue_ref:", {k: (v.shape if hasattr(v, "shape") else v) for k, v in out.items()})


if __name__ == "__main__":
    if "--yolo-glue-only" in sys.argv:
        ref_harness.import_reference()
        yolo_glue_golden()
    else:
        main()
