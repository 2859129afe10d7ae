"""CPU: the oracle against golden vectors produced by the reference's own code (tests/golden/make_golden.py), and
self-consistency of the restatements."""
from pathlib import Path

import cv2
import numpy as np
import pytest
import torch
from PIL import Image

from oracle import tracknet as OT
from oracle import weights as OW
from oracle import yolov8 as OY
from padel_analytics_b200 import synth
from padel_analytics_b200.engine import resample

GOLD = Path(__file__).resolve().parent / "golden"


def test_tracknet_forward_matches_reference_golden():
    g = np.load(GOLD / "tracknet_ref.npz")
    net = OW.load_tracknet(OW.make_tracknet())
    x = torch.rand((1, 27, 32, 64), generator=torch.Generator().manual_seed(int(g["seed"])))
    with torch.no_grad():
        y = net(x)
    # same torch ops in the same order, but the seeded weights and the forward run on CPU convolutions whose last bits
    # depend on the host's thread count (up to ~6e-6 here); bit-identical only on a host like the golden's
    assert np.abs(y.numpy() - g["y"]).max() < 5e-5


def test_ball_stage_matches_reference_golden():
    g = np.load(GOLD / "ball_ref.npz")
    T, B, H, W = (int(g[k]) for k in ("T", "B", "H", "W"))
    nh, nw = int(g["net_h"]), int(g["net_w"])
    frames = [f.numpy() for f in synth.make_frames(T, H, W, seed=int(g["seed"]))]
    med = synth.make_median(H, W, seed=int(g["seed"])).numpy()
    net = OW.load_tracknet(OW.make_tracknet())
    o = OT.run_ball_oracle(net, frames, med, (W, H), batch_size=B, width=nw, height=nh)
    # fp32 CPU conv results differ at the 1e-6 level between oneDNN call sequences; everything after the network
    # (ensemble arithmetic, threshold, contours, integer coordinates) is compared exactly below
    assert np.abs(o["ens"].numpy() - g["ens"]).max() < 5e-5
    assert torch.equal(OT.ensemble_reference_loop(o["preds"], T, 7), o["ens"])  # batching-independent
    assert o["x"] == g["x"].tolist() and o["y"] == g["y"].tolist() and o["vis"] == g["vis"].tolist()
    # closed form == stateful loop, and the library-free CCL == cv2 path, on the golden heat-maps
    assert torch.equal(OT.ensemble_closed_form(o["preds"], T), o["ens"])
    for n in range(T):
        m = (g["ens"][n] > 0.5)
        assert tuple(OT.heatmap_to_bbox((m * 255).astype("uint8"))) == tuple(OT.largest_component_bbox(m))


@pytest.mark.parametrize("T,bs", [(8, 4), (9, 8), (15, 3), (16, 5), (30, 8)])
def test_ensemble_closed_form_equals_loop(T, bs):
    p = torch.rand((T - 7, 8, 6, 10), generator=torch.Generator().manual_seed(T))
    assert torch.equal(OT.ensemble_reference_loop(p, T, bs), OT.ensemble_closed_form(p, T))


def test_ccl_restatement_matches_cv2_random():
    rng = np.random.default_rng(0)
    for _ in range(150):
        m = (rng.random((24, 40)) < rng.choice([0.01, 0.05, 0.2, 0.4, 0.6])).astype(np.uint8)
        assert tuple(OT.heatmap_to_bbox(m * 255)) == tuple(OT.largest_component_bbox(m))


def test_yolov8_restatement_param_counts():
    # published ultralytics figures (M params): v8n 3.16, v8s 11.17, v8m 25.90 (incl. the 16-weight DFL conv)
    for scale, expect in (("n", 3.157), ("s", 11.167), ("m", 25.903)):
        n = sum(p.numel() for p in OY.YoloV8(scale, 80).parameters()) / 1e6
        assert abs(n - expect) < 0.01, (scale, n)
    assert OY.YoloV8("n", 1, (13, 3))(torch.zeros(1, 3, 64, 64)).shape == (1, 4 + 1 + 39, 84)


def test_letterbox_geometry_and_tables_match_cv2():
    rng = np.random.default_rng(1)
    for (h, w) in ((1080, 1920), (720, 1280), (2160, 3840)):
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        ref = OY.letterbox(img, 640, auto=True)
        g = resample.letterbox_geometry(h, w, 640)
        assert ref.shape[:2] == (g["Hn"], g["Wn"]) == (384, 640)
        xo, xc = resample.cv2_linear_tables(w, g["rw"])
        yo, yc = resample.cv2_linear_tables(h, g["rh"])
        x1, y1 = np.minimum(xo + 1, w - 1), np.minimum(yo + 1, h - 1)
        I = img.astype(np.int32)
        rows = I[:, xo] * xc[:, 0][None, :, None] + I[:, x1] * xc[:, 1][None, :, None]
        out = (((yc[:, 0][:, None, None] * (rows[yo] >> 4)) >> 16) + ((yc[:, 1][:, None, None] * (rows[y1] >> 4)) >> 16) + 2) >> 2
        assert np.array_equal(out.astype(np.uint8), ref[g["top"]:g["top"] + g["rh"], g["left"]:g["left"] + g["rw"]])
        assert np.all(ref[: g["top"]] == 114)


def test_pil_tables_match_pillow():
    rng = np.random.default_rng(2)
    img = rng.integers(0, 256, (270, 480, 3), dtype=np.uint8)
    for (ow, oh) in ((128, 72), (320, 320), (600, 300)):
        bh, kh, _ = resample.pil_bicubic_tables(480, ow)
        bv, kv, _ = resample.pil_bicubic_tables(270, oh)
        I = img.astype(np.int64)
        tmp = np.zeros((270, ow, 3), np.int64)
        for xx in range(ow):
            x0, n = bh[xx]
            tmp[:, xx] = (I[:, x0:x0 + n] * kh[xx, :n][None, :, None]).sum(1)
        tmp = np.clip((tmp + (1 << 21)) >> 22, 0, 255)
        out = np.zeros((oh, ow, 3), np.int64)
        for yy in range(oh):
            y0, n = bv[yy]
            out[yy] = (tmp[y0:y0 + n] * kv[yy, :n][:, None, None]).sum(0)
        out = np.clip((out + (1 << 21)) >> 22, 0, 255).astype(np.uint8)
        assert np.array_equal(out, np.array(Image.fromarray(img).resize((ow, oh))))


def test_seeded_weights_are_deterministic_and_useful():
    a, b = OW.make_yolo("court12"), OW.make_yolo("court12")
    assert all(torch.equal(a["model"][k], b["model"][k]) for k in a["model"])
    frames = [f.numpy() for f in synth.make_frames(1, 360, 640, start=2)]
    yolo = OY.YOLO(OW.load_yolo(a))
    sample = [Image.fromarray(cv2.cvtColor(f, cv2.COLOR_BGR2RGB)).resize((640, 640)) for f in frames]
    res = yolo.predict(sample, conf=0.5, iou=0.7, imgsz=640, max_det=12)
    assert len(res) == 1 and res[0].keypoints.xy.shape[1:] == (12, 2)


def test_inpaint_stage_matches_reference_golden():
    """oracle/inpaint.py against the reference's own BallTracker inpainting pass (tests/golden/inpaint_ref.npz)."""
    from oracle import inpaint as OI

    g = np.load(GOLD / "inpaint_ref.npz")
    net = OI.load_inpaintnet(OI.make_inpaintnet())
    out, mask = OI.inpaint_stage(net, g["x"].tolist(), g["y"].tolist(), g["vis"].tolist(), (int(g["W"]), int(g["H"])),
                                 int(g["seq_len"]), (int(g["net_h"]), int(g["net_w"])), batch_size=int(g["B"]))
    assert sum(mask) > 5 and sum(g["vis"].tolist()) < len(mask)  # the mask and the gaps are exercised
    assert out["X"] == g["X"].tolist() and out["Y"] == g["Y"].tolist() and out["Visibility"] == g["V"].tolist()


def test_tracker_glue_reproduces_reference_golden():
    """tests/golden/yolo_glue_ref.npz was produced by the UNMODIFIED reference tracker classes (predict_sample of
    PlayerKeypointsTracker / KeypointsTracker / PlayerTracker) driving the oracle YOLO on the committed rally.mp4 crops.
    The product trackers' host glue (processor semantics, predict arguments, ratio scaling, id mapping, result objects)
    fed with the same oracle results must reproduce it EXACTLY; the GPU tests then only have to show engine == oracle.
    The golden also stores the oracle results the reference glue was given.  The glue is fed those, because the seeded
    checkpoints and the oracle run on CPU convolutions whose last bits depend on the host's thread count; the oracle
    recomputed here must match them to that rounding."""
    import cv2
    from PIL import Image

    from fixtures import GOLDEN, court_conf_for_single_detection, glue_ckpt, rally_frames
    from oracle import yolov8 as OY
    from padel_analytics_b200.trackers import sv_compat as sv
    from padel_analytics_b200.trackers.keypoints_tracker import KeypointsTracker
    from padel_analytics_b200.trackers.players_keypoints_tracker import PlayerKeypoints, PlayerKeypointsTracker
    from padel_analytics_b200.trackers.players_tracker import PlayerTracker

    g = np.load(GOLDEN / "yolo_glue_ref.npz")
    frames = rally_frames()
    H, W = frames[0].shape[:2]
    assert (H, W, len(frames)) == (int(g["H"]), int(g["W"]), int(g["n"]))
    rgb = [cv2.cvtColor(f, cv2.COLOR_BGR2RGB) for f in frames]
    pil = [Image.fromarray(f).resize((640, 640)) for f in rgb]

    def stored(kind, i, like):
        """The stored oracle result of frame i, as the Result `like` (the recomputed one) is laid out."""
        kp = f"oracle_{kind}_kpts_{i}"
        return OY.Result(OY.Boxes(torch.from_numpy(g[f"oracle_{kind}_boxes_{i}"])),
                         OY.Keypoints(torch.from_numpy(g[kp])) if kp in g.files else None, like.names, like.orig_shape)

    def same_detections(res, ref):
        """Same detections; box edges to 0.1 px (the seeded heads' multi-modal DFL edges are ill-conditioned, see
        tests/parity.py: last-bit changes of the weights move them by up to ~0.01 px), scores and keypoints to 1e-3."""
        assert len(res) == len(ref)
        for r, s in zip(res, ref):
            assert r.boxes.data.shape == s.boxes.data.shape
            assert torch.allclose(r.boxes.xyxy, s.boxes.xyxy, rtol=0, atol=0.1)
            assert torch.allclose(r.boxes.data[:, 4:], s.boxes.data[:, 4:], rtol=0, atol=1e-3)
            assert (r.keypoints is None) == (s.keypoints is None)
            if s.keypoints is not None:
                assert torch.allclose(r.keypoints.data, s.keypoints.data, rtol=0, atol=1e-3)

    # pose (players_keypoints_tracker.py:271-322)
    pk = object.__new__(PlayerKeypointsTracker)  # no CUDA here: skip the engine, keep the class constants
    pk.train_image_size = 640
    res = OY.YOLO(OW.load_yolo(glue_ckpt("pose13"))).predict(pil, conf=pk.CONF, iou=pk.IOU, imgsz=640, classes=[0])
    ref = [stored("pose", i, r) for i, r in enumerate(res)]
    same_detections(res, ref)
    out = pk.postprocess(ref, (H, W))
    assert list(g["pose_names"]) == PlayerKeypoints.KEYPOINTS_NAMES
    for i, p in enumerate(out):
        arr = np.array([[kp.xy for kp in pl.player_keypoints] for pl in p.players_keypoints], dtype=np.float64)
        assert np.array_equal(arr, g[f"pose_{i}"]), f"pose frame {i}"
        assert [kp.id for kp in p.players_keypoints[0].player_keypoints] == list(range(13))

    # court (keypoints_tracker.py:199-262), one detection per frame by construction of the golden
    net = OW.load_yolo(glue_ckpt("court12"))
    kt = object.__new__(KeypointsTracker)
    for i, f in enumerate(frames):
        conf = float(g["court_conf"][i])
        assert abs(court_conf_for_single_detection(net, f) - conf) < 1e-5
        res = OY.YOLO(net).predict([pil[i]], conf=conf, iou=kt.IOU, imgsz=kt.TRAIN_IMAGE_SIZE, max_det=kt.NUMBER_KEYPOINTS)
        ref = [stored("court", i, res[0])]
        same_detections(res, ref)
        (kp,) = kt.postprocess(ref, (H, W))
        assert [k.id for k in kp.keypoints] == list(range(12))
        assert np.array_equal(np.array([k.xy for k in kp.keypoints]), g[f"court_{i}"]), f"court frame {i}"

    # players (players_tracker.py:341-380) with this repo's supervision stand-ins on both sides
    pt = object.__new__(PlayerTracker)
    pt.polygon_zone = sv.PolygonZone(np.array([[0, 0], [W, 0], [W, H], [0, H]]), frame_resolution_wh=(W, H))
    pt.video_info_post_init(sv.VideoInfo(width=W, height=H, fps=25.0, total_frames=len(frames)))
    res = OY.YOLO(OW.load_yolo(glue_ckpt("detect"))).predict(rgb, conf=pt.CONF, iou=pt.IOU, imgsz=pt.IMGSZ, classes=[0])
    ref = [stored("players", i, r) for i, r in enumerate(res)]
    same_detections(res, ref)
    for i, p in enumerate(pt.postprocess(ref)):
        arr = np.array([[*pl.xyxy, pl.confidence, pl.class_id, -1 if pl.id is None else pl.id] for pl in p.players],
                       dtype=np.float64).reshape(-1, 7)
        assert np.array_equal(arr, g[f"players_{i}"]), f"players frame {i}"


def test_resnet_oracle_reproduces_reference_golden():
    """oracle/resnet.py (pipeline restatement around torchvision's resnet50) vs the golden produced by the unmodified
    reference KeypointsTracker(model_type="resnet").predict_frames on the rally.mp4 crops."""
    from fixtures import GOLDEN, rally_frames
    from oracle import resnet as OR

    g = np.load(GOLDEN / "yolo_glue_ref.npz")
    got = OR.predict(OR.load(OR.make_resnet50_court()), rally_frames())
    # the reference multiplies float32 sigmoid outputs by the integer frame size (float32 products)
    assert np.abs(got - g["resnet"]).max() < 1e-3
