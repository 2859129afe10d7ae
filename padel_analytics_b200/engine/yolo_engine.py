"""YOLOv8 detect / pose inference on the B200 kernels behind the `ultralytics.YOLO(...).predict()` surface the
reference trackers use:
    /root/reference/trackers/players_tracker/players_tracker.py:303,338-339,351-359
    /root/reference/trackers/players_keypoints_tracker/players_keypoints_tracker.py:238,285-292
    /root/reference/trackers/keypoints_tracker/keypoints_tracker.py:169,238-245
Graph = ultralytics yolov8{,-pose}.yaml layers 0..22 (third-party; SURVEY.md App. A.2), executed as a static list of
fused conv kernels over preallocated NHWC fp16 buffers; concat / chunk / residual / upsample are channel-slice
reads and writes (no copies except the two nearest-upsamples and SPPF pooling).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from .. import _lib as L
from . import ops, resample


# ---- result containers with the attribute surface the trackers (and sv.Detections.from_ultralytics) touch ----------
@dataclass
class Boxes:
    data: torch.Tensor  # (N,6) xyxy, conf, cls  (CPU float32)

    @property
    def xyxy(self):
        return self.data[:, :4]

    @property
    def conf(self):
        return self.data[:, 4]

    @property
    def cls(self):
        return self.data[:, 5]

    @property
    def id(self):
        return None

    def __len__(self):
        return self.data.shape[0]


@dataclass
class Keypoints:
    data: torch.Tensor  # (N,K,D)

    @property
    def xy(self):
        return self.data[..., :2]

    @property
    def conf(self):
        return self.data[..., 2] if self.data.shape[-1] == 3 else None


@dataclass
class Result:
    boxes: Boxes
    keypoints: Keypoints | None
    names: dict
    orig_shape: tuple


class ResultBlock:
    """The Results of consecutive frames as ONE dense array: rows (n, cap, 6 + K*D) float32 = [x1, y1, x2, y2, conf,
    cls, keypoints...] per detection (score-sorted, rows at and beyond counts[i] are padding) + counts (n,) int32.
    A read-only sequence of `Result`s (built on demand, views into the block) for code written against ultralytics'
    list of Results; the trackers' post-processing and the multi-GPU gather read the arrays directly -- at thousands
    of frames per second a Python object per frame and tracker is the expensive part of the host side."""

    __slots__ = ("rows", "counts", "kpt_shape", "names", "orig_shape", "_t")

    def __init__(self, rows: np.ndarray, counts: np.ndarray, kpt_shape, names, orig_shape):
        self.rows, self.counts, self.kpt_shape, self.names, self.orig_shape = rows, counts, kpt_shape, names, orig_shape
        self._t = None

    def __len__(self):
        return self.rows.shape[0]

    @property
    def keypoints(self) -> np.ndarray | None:
        """(n, cap, K, D) view of the keypoint columns"""
        if not self.kpt_shape:
            return None
        n, cap = self.rows.shape[:2]
        return self.rows[..., 6:].reshape(n, cap, *self.kpt_shape)

    def __getitem__(self, i):
        if isinstance(i, slice):
            a, b, step = i.indices(len(self))
            if step != 1:
                raise IndexError("ResultBlock: contiguous slices only")
            return ResultBlock(self.rows[a:b], self.counts[a:b], self.kpt_shape, self.names, self.orig_shape)
        if i < 0:
            i += len(self)
        if not 0 <= i < len(self):
            raise IndexError(i)
        if self._t is None:
            kp = self.keypoints
            self._t = (torch.from_numpy(self.rows[..., :6]), torch.from_numpy(kp) if kp is not None else None)
        c = int(self.counts[i])
        bt, kt = self._t
        return Result(Boxes(bt[i, :c]), Keypoints(kt[i, :c]) if kt is not None else None, self.names, self.orig_shape)

    def __iter__(self):
        return (self[i] for i in range(len(self)))

    @staticmethod
    def concat(blocks: list, like: "ResultBlock | None" = None) -> "ResultBlock":
        """Frames of several blocks in order, padded to the largest per-frame count (padding rows zeroed)."""
        ref = blocks[0] if blocks else like
        rowlen = ref.rows.shape[2]
        cap = max([int(b.counts.max()) for b in blocks if len(b)], default=0)
        cap = max(cap, 1)
        n = sum(len(b) for b in blocks)
        rows = np.zeros((n, cap, rowlen), dtype=np.float32)
        counts = np.zeros((n,), dtype=np.int32)
        at = 0
        for b in blocks:
            m, c = len(b), min(cap, b.rows.shape[1])
            rows[at:at + m, :c] = b.rows[:, :c]
            counts[at:at + m] = b.counts
            at += m
        rows[np.arange(cap)[None, :] >= counts[:, None]] = 0
        return ResultBlock(rows, counts, ref.kpt_shape, ref.names, ref.orig_shape)


def _kpad(c: int) -> int:
    """Channel count a conv should READ: widths in (32, 64) or not a multiple of 64 above that are rounded up to a
    multiple of 64 (zero channels in the buffer, zero weights), so the kernel runs 64-channel K blocks (128-byte rows,
    one TMA box per tap) instead of three to five 16/32-channel blocks."""
    return c if (c <= 32 or c % 64 == 0) else (c + 63) // 64 * 64


def _fold(sd, p, eps=1e-3):
    return ops.fold_bn(sd[f"{p}.conv.weight"].float(), sd[f"{p}.bn.weight"].float(), sd[f"{p}.bn.bias"].float(),
                       sd[f"{p}.bn.running_mean"].float(), sd[f"{p}.bn.running_var"].float(), eps)


class YoloEngine:
    """Drop-in for `ultralytics.YOLO(model_path)`: .predict(source, conf=, iou=, imgsz=, device=, classes=, max_det=),
    .to(device), .names.  `ckpt` is a dict {'model': state_dict (ultralytics key names), 'nc', 'kpt_shape'} or a path
    to a torch file holding one."""

    MAX_NMS = 30000  # ultralytics ops.non_max_suppression max_nms: candidates per image that enter NMS

    def __init__(self, ckpt, max_batch: int = 8, device: str = "cuda"):
        if not torch.cuda.is_available():
            raise L.PbError("YoloEngine needs a CUDA device (no CPU fallback)")
        L.lib()
        if not isinstance(ckpt, dict):
            ckpt = torch.load(ckpt, map_location="cpu", weights_only=False)
        self.sd = {k: v for k, v in ckpt["model"].items()}
        self.nc = int(ckpt["nc"])
        self.kpt_shape = tuple(ckpt["kpt_shape"]) if ckpt.get("kpt_shape") else None
        self.nk = self.kpt_shape[0] * self.kpt_shape[1] if self.kpt_shape else 0
        self.names = ckpt.get("names") or {i: ("person" if (i == 0 and self.nc == 80) else f"class{i}")
                                           for i in range(self.nc)}
        self.device = torch.device(device)
        self.B = max_batch
        self._progs = {}  # (Hn, Wn) -> built program state
        self._packed = {}
        self._tables = {}
        self._stage = None

    def to(self, device):
        return self

    # ------------------------------------------------------------------------------------------------------
    # weights
    # ------------------------------------------------------------------------------------------------------
    def _wb(self, prefix, cin_pad, cout_pad, bn=True):
        key = (prefix, cin_pad, cout_pad)
        if key not in self._packed:
            if bn:
                w, b = _fold(self.sd, prefix)
            else:
                w, b = self.sd[f"{prefix}.weight"].float(), self.sd[f"{prefix}.bias"].float()
            self._packed[key] = ops.pack_conv_weight(w, b, cin_pad, cout_pad, self.device)
        return self._packed[key]

    def _cout(self, prefix, bn=True):
        return self.sd[f"{prefix}.conv.weight" if bn else f"{prefix}.weight"].shape[0]

    # ------------------------------------------------------------------------------------------------------
    # program construction for one network input size
    # ------------------------------------------------------------------------------------------------------
    def _build(self, Hn, Wn):
        B, dev, sd = self.B, self.device, self.sd
        P = ops.Program()
        bufs = []

        def buf(h, w, c, dtype=torch.float16):
            t = torch.zeros((B, h, w, c), dtype=dtype, device=dev)
            bufs.append(t)
            return t

        SILU = L.ACT_SILU

        def conv(x, coff, cin, prefix, out, ooff, k, s, res=None, res_off=0, up=None):
            cout = self._cout(prefix)
            w, b = self._wb(prefix, cin, ops.pad16(cout))
            P.conv(ops.make_conv_desc(x, coff, cin, w, b, k, s, SILU, out, ooff, L.OUT_F16_NHWC, None, res, res_off,
                                      out2=None if up is None else (up, 0, L.OUT2_UP2)),
                   cin_real=self.sd[f"{prefix}.conv.weight"].shape[1], cout_real=cout)
            return ops.pad16(cout)

        def c2f(x, coff, cin, i, out, ooff, shortcut, up=None):
            """ultralytics C2f (App. A.2): cv1 -> [y0,y1] ; y_{j+2} = Bottleneck_j(y_{j+1}) ; cv2(cat(y))."""
            pre = f"model.{i}"
            c = self._cout(f"{pre}.cv1") // 2
            n = 0
            while f"{pre}.m.{n}.cv1.conv.weight" in sd:
                n += 1
            _, h, w_, _ = x.shape
            ccat = _kpad((2 + n) * c)
            cat = buf(h, w_, ccat)
            tmp = buf(h, w_, c)
            conv(x, coff, cin, f"{pre}.cv1", cat, 0, 1, 1)
            for j in range(n):
                conv(cat, (1 + j) * c, c, f"{pre}.m.{j}.cv1", tmp, 0, 3, 1)
                conv(tmp, 0, c, f"{pre}.m.{j}.cv2", cat, (2 + j) * c, 3, 1, res=cat if shortcut else None,
                     res_off=(1 + j) * c)
            conv(cat, 0, ccat, f"{pre}.cv2", out, ooff, 1, 1, up=up)

        # the two nn.Upsample(2, "nearest") of the neck (layers 10, 13) are a second, replicated store of the
        # producing 1x1 conv (PB_OUT2_UP2)
        c0, c1, c2, c3, c4 = (self._cout(f"model.{i}") for i in (0, 1, 3, 5, 7))
        for c in (c0, c1, c2, c3, c4):
            if c % 16:
                raise L.PbError(f"YoloEngine: channel width {c} is not a multiple of 16")
        H2, W2, H4, W4, H8, W8 = Hn // 2, Wn // 2, Hn // 4, Wn // 4, Hn // 8, Wn // 8
        H16, W16, H32, W32 = Hn // 16, Wn // 16, Hn // 32, Wn // 32
        # network input: 4-channel fp16 pixels with a one-pixel zero border (PB_IN_STEM4), written by the
        # pre-processing kernels; the border is never touched after this zero fill
        x0 = torch.zeros((B, Hn + 2, Wn + 2, 4), dtype=torch.float16, device=dev)
        bufs.append(x0)
        b0, b1, b2 = buf(H2, W2, c0), buf(H4, W4, c1), buf(H4, W4, c1)
        b3 = buf(H8, W8, c2)
        cat14 = buf(H8, W8, c3 + c2)  # [up(12) c3 | P3 c2]
        b5 = buf(H16, W16, c3)
        cat11 = buf(H16, W16, c4 + c3)  # [up(9) c4 | P4 c3]
        b7, b8 = buf(H32, W32, c4), buf(H32, W32, c4)
        sp = buf(H32, W32, 4 * (c4 // 2))
        cat20 = buf(H32, W32, c3 + c4)  # [conv19 c3 | P5 c4]
        cat17 = buf(H16, W16, c2 + c3)  # [conv16 c2 | h4 c3]
        o3, o4, o5 = buf(H8, W8, c2), buf(H16, W16, c3), buf(H32, W32, c4)

        w0, bias0 = _fold(sd, "model.0")
        if "stem" not in self._packed:
            self._packed["stem"] = ops.pack_stem_weight(w0, bias0, ops.pad16(c0), dev)
        P.conv(ops.make_stem_desc(x0, *self._packed["stem"], SILU, b0), cin_real=3, cout_real=c0)
        conv(b0, 0, c0, "model.1", b1, 0, 3, 2)
        c2f(b1, 0, c1, 2, b2, 0, True)
        conv(b2, 0, c1, "model.3", b3, 0, 3, 2)
        c2f(b3, 0, c2, 4, cat14, c3, True)  # P3
        conv(cat14, c3, c2, "model.5", b5, 0, 3, 2)
        c2f(b5, 0, c3, 6, cat11, c4, True)  # P4
        conv(cat11, c4, c3, "model.7", b7, 0, 3, 2)
        c2f(b7, 0, c4, 8, b8, 0, True)
        conv(b8, 0, c4, "model.9.cv1", sp, 0, 1, 1)  # SPPF
        P.sppf_pool(sp, c4 // 2)
        conv(sp, 0, 4 * (c4 // 2), "model.9.cv2", cat20, c3, 1, 1, up=cat11)  # P5 (+ layers 10-11)
        c2f(cat11, 0, c4 + c3, 12, cat17, c2, False, up=cat14)  # h4 (+ layers 13-14)
        c2f(cat14, 0, c3 + c2, 15, o3, 0, False)
        conv(o3, 0, c2, "model.16", cat17, 0, 3, 2)
        c2f(cat17, 0, c2 + c3, 18, o4, 0, False)
        conv(o4, 0, c3, "model.19", cat20, 0, 3, 2)
        c2f(cat20, 0, c3 + c4, 21, o5, 0, False)

        # heads: per level box / cls (/ kpt) branches -> one fp32 NHWC map (B,h,w,64+nc+nk)
        # head map layout: [box 0:64 | kpt 64:64+nk | cls ...], 32-byte aligned slices and rows so the epilogue's
        # fast path stores 8 floats per instruction
        kpt_off = 64
        cls_off = 64 + (self.nk + 7) // 8 * 8
        fC = (cls_off + self.nc + 7) // 8 * 8
        feats, levels = [], []
        branches = [("cv2", 64, 0), ("cv3", self.nc, cls_off)]
        if self.nk:
            branches.append(("cv4", self.nk, kpt_off))
        for l, (f, cf, st) in enumerate(((o3, c2, 8), (o4, c3, 16), (o5, c4, 32))):
            _, h, w_, _ = f.shape
            feat = buf(h, w_, fC, torch.float32)
            # the branches' first 3x3 convs all read `f`: run them as ONE conv (weights concatenated along cout) so the
            # level's feature map is fetched once; each branch then reads its channel slice of the merged tensor
            widths = [_kpad(ops.pad16(self._cout(f"model.22.{name}.{l}.0"))) for name, _, _ in branches]
            key = ("head0", l)
            if key not in self._packed:
                ws, bs = zip(*(ops.pack_conv_weight(*_fold(sd, f"model.22.{name}.{l}.0"), cf, wd, dev)
                               for (name, _, _), wd in zip(branches, widths)))
                self._packed[key] = (torch.cat(ws, 1).contiguous(), torch.cat(bs, 0).contiguous())
            wm, bm = self._packed[key]
            t1m = buf(h, w_, sum(widths))
            cin_real = sd[f"model.22.cv2.{l}.0.conv.weight"].shape[1]
            cout_real = sum(self._cout(f"model.22.{name}.{l}.0") for name, _, _ in branches)
            wsum = sum(widths)
            # A shallow-K level (cin <= 64) keeps its whole filter bank resident in shared memory only up to ~96 output
            # channels, and a 192-wide accumulator leaves room for one sub-tile per CTA tile (weights re-fetched from L2
            # for every 128 pixels: ncu shows the 64->192 @160^2 conv at 2x its tensor bound).  Two launches of half the
            # output channels each run with resident weights and two sub-tiles; the input is small (cin <= 64).
            nsplit = 2 if (cf <= 64 and wsum > 128 and (wsum // 2) % 16 == 0) else 1
            for part in range(nsplit):
                a, b_ = part * wsum // nsplit, (part + 1) * wsum // nsplit
                key = ("head0", l, part, nsplit)
                if key not in self._packed:
                    self._packed[key] = (wm[:, a:b_].contiguous(), bm[a:b_].contiguous())
                wp_, bp_ = self._packed[key]
                P.conv(ops.make_conv_desc(f, 0, cf, wp_, bp_, 3, 1, SILU, t1m, a),
                       cin_real=cin_real, cout_real=cout_real * (b_ - a) // wsum)
            for bi, (name, cout_real, off) in enumerate(branches):
                pre = f"model.22.{name}.{l}"
                cm = widths[bi]
                t2 = buf(h, w_, cm)
                conv(t1m, sum(widths[:bi]), cm, f"{pre}.1", t2, 0, 3, 1)
                w, b = self._wb(f"{pre}.2", cm, ops.pad16(cout_real), bn=False)
                # whole 8-float groups are stored (one 32-byte store each): the slice of every branch is padded to a
                # multiple of 8 channels in `feat`, and the padding channels have zero weights and bias
                store = min((cout_real + 7) // 8 * 8, ops.pad16(cout_real))
                P.conv(ops.make_conv_desc(t2, 0, cm, w, b, 1, 1, L.ACT_NONE, feat, off, L.OUT_F32_NHWC, store),
                       cin_real=self.sd[f"{pre}.2.weight"].shape[1], cout_real=cout_real)
            feats.append(feat)
            levels.append((feat, h, w_, st))
        lv = (L.YoloLevel * 3)()
        for l, (feat, h, w_, st) in enumerate(levels):
            lv[l].feat, lv[l].h, lv[l].w, lv[l].stride = feat.data_ptr(), h, w_, st
        rowlen = 6 + self.nk
        # candidate capacity = every anchor, capped at ultralytics' max_nms (so nothing the reference would keep is lost)
        cap = min(sum(h * w_ for _, h, w_, _ in levels), self.MAX_NMS)
        scratch_bytes = L.lib().pb_yolo_nms_scratch_bytes(B, cap)
        st = dict(prog=P, cap=cap,
                  nms_scratch=torch.empty((max(scratch_bytes, 16),), dtype=torch.uint8, device=dev), bufs=bufs, x0=x0, levels=lv, fC=fC, rowlen=rowlen, Hn=Hn, Wn=Wn, cls_off=cls_off,
                  kpt_off=kpt_off,
                  cand=torch.zeros((B, cap, rowlen), dtype=torch.float32, device=dev),
                  cand_anchor=torch.zeros((B, cap), dtype=torch.int32, device=dev),
                  cand_count=torch.zeros((B,), dtype=torch.int32, device=dev),
                  feats=feats)
        return st

    def _state(self, Hn, Wn):
        key = (Hn, Wn)
        if key not in self._progs:
            if Hn % 32 or Wn % 32:
                raise L.PbError(f"YoloEngine: network input {Hn}x{Wn} must be a multiple of 32")
            self._progs[key] = self._build(Hn, Wn)
        return self._progs[key]

    # ------------------------------------------------------------------------------------------------------
    # pre-processing front ends (all write st['x0'])
    # ------------------------------------------------------------------------------------------------------
    def _upload(self, frames) -> torch.Tensor:
        """list of HWC u8 arrays / (n,H,W,3) tensor (host or device) -> device u8 (n,H,W,3)."""
        if isinstance(frames, torch.Tensor):
            t = frames
        else:
            t = torch.from_numpy(np.stack([np.ascontiguousarray(f) for f in frames]))
        if t.dtype != torch.uint8 or t.dim() != 4 or t.shape[-1] != 3:
            raise L.PbError("frames must be uint8 (n,H,W,3)")
        if t.shape[0] > self.B:
            raise L.PbError(f"batch {t.shape[0]} exceeds engine max_batch {self.B}")
        if t.device.type != "cuda":
            n = t.shape[0]
            if self._stage is None or self._stage.shape[1:] != t.shape[1:]:
                self._stage = torch.empty((self.B,) + tuple(t.shape[1:]), dtype=torch.uint8, device=self.device)
            self._stage[:n].copy_(t, non_blocking=True)
            t = self._stage[:n]
        return t.contiguous()

    def _letterbox(self, frames_dev, imgsz, chan_map):
        n, Hs, Ws, _ = frames_dev.shape
        g = resample.letterbox_geometry(Hs, Ws, imgsz, 32, auto=True)
        st = self._state(g["Hn"], g["Wn"])
        key = ("lb", Hs, Ws, g["rh"], g["rw"])
        if key not in self._tables:
            xo, xc = resample.cv2_linear_tables(Ws, g["rw"])
            yo, yc = resample.cv2_linear_tables(Hs, g["rh"])
            self._tables[key] = tuple(torch.from_numpy(np.ascontiguousarray(a)).to(self.device) for a in (xo, xc, yo, yc))
        xo, xc, yo, yc = self._tables[key]
        L.check(L.lib().pb_letterbox_u8_f16(frames_dev.data_ptr(), n, Hs, Ws, st["x0"].data_ptr(), g["Hn"], g["Wn"],
                                            g["rh"], g["rw"], g["top"], g["left"], xo.data_ptr(), xc.data_ptr(),
                                            yo.data_ptr(), yc.data_ptr(), chan_map[0], chan_map[1], chan_map[2], 1,
                                            L.stream_ptr()))
        return st, (Hs, Ws)

    def _pil_square(self, frames_dev, size):
        """BGR frames -> RGB -> Pillow-exact bicubic resize to size x size -> network input (RGB order)."""
        n, Hs, Ws, _ = frames_dev.shape
        st = self._state(size, size)
        key = ("pil", Hs, Ws, size)
        if key not in self._tables:
            bh, kh, ksh = resample.pil_bicubic_tables(Ws, size)
            bv, kv, ksv = resample.pil_bicubic_tables(Hs, size)
            up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(self.device)
            self._tables[key] = dict(bh=up(bh), kh=up(kh), ksh=ksh, bv=up(bv), kv=up(kv), ksv=ksv,
                                     tmp=torch.empty((self.B, Hs, size, 3), dtype=torch.uint8, device=self.device))
        t = self._tables[key]
        # the vertical pass writes the normalised fp16 network input directly (no u8 round trip)
        L.check(L.lib().pb_pil_resize_u8(frames_dev.data_ptr(), n, Hs, Ws, t["tmp"].data_ptr(), None,
                                         size, size, t["bh"].data_ptr(), t["kh"].data_ptr(), t["ksh"],
                                         t["bv"].data_ptr(), t["kv"].data_ptr(), t["ksv"], 1, st["x0"].data_ptr(), 1,
                                         L.stream_ptr()))
        return st, (size, size)

    # ------------------------------------------------------------------------------------------------------
    # forward + decode + NMS + host epilogue
    # ------------------------------------------------------------------------------------------------------
    def _detect(self, st, n, conf, iou, classes, max_det):
        return self._detect_finish(self._detect_launch(st, n, conf, iou, classes, max_det))

    def _detect_launch(self, st, n, conf, iou, classes, max_det):
        """Enqueue forward + decode + NMS + the device->pinned-host copies on the current stream; no host sync."""
        lib = L.lib()
        st["prog"].run()
        kdim = self.kpt_shape[1] if self.kpt_shape else 0
        cls_arr, ncls = None, 0
        if classes is not None:
            ncls = len(classes)
            cls_arr = (C.c_int * max(ncls, 1))(*[int(c) for c in classes])
        # only the n images of this call are decoded / suppressed (slots >= n hold stale activations)
        L.check(lib.pb_yolo_decode(st["levels"], 3, n, st["fC"], self.nc, self.nk, kdim, st["cls_off"],
                                   st["kpt_off"], float(conf), cls_arr, ncls,
                                   st["cand"].data_ptr(), st["cand_anchor"].data_ptr(), st["cand_count"].data_ptr(),
                                   st["cap"], L.stream_ptr()))
        key = ("out", max_det)
        if key not in st:
            # device results + a small ring of pinned host copies: a caller may enqueue the next batch before it
            # has collected this one (FusedPass keeps one batch of look-ahead)
            st[key] = dict(out=torch.zeros((self.B, max_det, st["rowlen"]), dtype=torch.float32, device=self.device),
                           cnt=torch.zeros((self.B,), dtype=torch.int32, device=self.device),
                           host=[(torch.zeros((self.B, max_det, st["rowlen"]), dtype=torch.float32).pin_memory(),
                                  torch.zeros((2, self.B), dtype=torch.int32).pin_memory()) for _ in range(3)],
                           pending=[None] * 3, turn=0)
        ring = st[key]
        out, cnt = ring["out"], ring["cnt"]
        slot = ring["turn"]
        ring["turn"] = (slot + 1) % 3
        if ring["pending"][slot] is not None:  # an uncollected launch still owns this slot: resolve it first
            self._detect_resolve(ring["pending"][slot])
        out_h, cnt_h = ring["host"][slot]
        L.check(lib.pb_yolo_nms(st["cand"].data_ptr(), st["cand_anchor"].data_ptr(), st["cand_count"].data_ptr(),
                                n, st["cap"], st["rowlen"], float(iou), max_det, out.data_ptr(),
                                cnt.data_ptr(), st["nms_scratch"].data_ptr(), L.stream_ptr()))
        out_h.copy_(out, non_blocking=True)
        cnt_h[0].copy_(cnt, non_blocking=True)
        cnt_h[1].copy_(st["cand_count"], non_blocking=True)
        done = torch.cuda.Event()
        done.record()
        handle = dict(done=done, out_h=out_h, cnt_h=cnt_h, n=n, ring=ring, slot=slot, result=None, cap=st["cap"])
        ring["pending"][slot] = handle
        return handle

    def _detect_resolve(self, handle):
        if handle["result"] is None:
            handle["done"].synchronize()
            n, cnt_h = handle["n"], handle["cnt_h"]
            if int(cnt_h[1][:n].max()) > handle["cap"]:
                # only reachable when more than max_nms = 30000 anchors of one image pass `conf` (ultralytics would keep
                # the 30000 best-scoring ones; a threshold that lets 90 % of a 1280^2 grid through is a usage error)
                raise L.PbError(f"YoloEngine: {int(cnt_h[1][:n].max())} candidates exceed max_nms={handle['cap']}")
            handle["result"] = (handle["out_h"].numpy()[:n].copy(), cnt_h[0].numpy()[:n].copy())
            handle["ring"]["pending"][handle["slot"]] = None
        return handle["result"]

    def _detect_finish(self, handle):
        return self._detect_resolve(handle)

    def _results_block(self, rows, counts, n, net_hw, orig_hw) -> ResultBlock:
        """scale_boxes / scale_coords / clip / keypoint conf<0.5 -> 0 (ultralytics ops, SURVEY App. A.4 vi-vii),
        float32 arithmetic on the host, one vectorised pass over the whole (n, cap, 6+nk) block, cap = the largest
        per-image count (the padding rows beyond each image's own count are transformed too and never looked at)."""
        h1, w1 = net_hw
        h0, w0 = orig_hw
        gain = min(h1 / h0, w1 / w0)
        padb = (round((w1 - w0 * gain) / 2 - 0.1), round((h1 - h0 * gain) / 2 - 0.1))
        padk = ((w1 - w0 * gain) / 2, (h1 - h0 * gain) / 2)
        g32 = np.float32(gain)
        counts = np.asarray(counts[:n], dtype=np.int32)
        cap = max(int(counts.max()) if n else 0, 1)  # only the rows some image uses are transformed and kept
        r = rows[:n, :cap].astype(np.float32, copy=True)
        box = r[..., :6]
        box[..., [0, 2]] -= np.float32(padb[0])
        box[..., [1, 3]] -= np.float32(padb[1])
        box[..., :4] /= g32
        box[..., 0] = np.clip(box[..., 0], 0, w0)
        box[..., 2] = np.clip(box[..., 2], 0, w0)
        box[..., 1] = np.clip(box[..., 1], 0, h0)
        box[..., 3] = np.clip(box[..., 3], 0, h0)
        kall = None
        if self.kpt_shape:
            K, D = self.kpt_shape
            kall = r[..., 6:].reshape(n, r.shape[1], K, D)
            kall[..., 0] -= np.float32(padk[0])
            kall[..., 1] -= np.float32(padk[1])
            kall[..., 0] /= g32
            kall[..., 1] /= g32
            kall[..., 0] = np.clip(kall[..., 0], 0, w0)
            kall[..., 1] = np.clip(kall[..., 1], 0, h0)
            if D == 3:
                m = kall[..., 2] < 0.5
                kall[..., 0][m] = 0
                kall[..., 1][m] = 0
        return ResultBlock(r, counts, self.kpt_shape, self.names, (h0, w0))

    def _results(self, rows, counts, n, net_hw, orig_hw) -> list:
        return list(self._results_block(rows, counts, n, net_hw, orig_hw))

    @torch.no_grad()
    def predict(self, source, conf=0.25, iou=0.7, imgsz=640, device=None, classes=None, max_det=300, **kw):
        """ultralytics-compatible entry: `source` is a list of BGR ndarrays or of PIL RGB images (one batch)."""
        if len(source) == 0:
            return []
        if isinstance(source[0], np.ndarray):
            arrs, cmap = source, (2, 1, 0)  # BGR in -> network sees RGB (App. A.4 i,iii)
        else:
            arrs, cmap = [np.asarray(im) for im in source], (0, 1, 2)  # PIL RGB -> BGR -> flipped back
        if len({a.shape for a in arrs}) != 1:
            raise L.PbError("YoloEngine.predict: all images of a batch must share one shape")
        out = []
        for i in range(0, len(arrs), self.B):
            chunk = arrs[i:i + self.B]
            fr = self._upload(chunk)
            st, orig = self._letterbox(fr, imgsz, cmap)
            rows, counts = self._detect(st, len(chunk), conf, iou, classes, max_det)
            out += self._results(rows, counts, len(chunk), (st["Hn"], st["Wn"]), orig)
        return out

    @torch.no_grad()
    def predict_frames(self, frames, prep: str, conf, iou, imgsz, classes=None, max_det=300):
        """Fused fast path used by this repo's trackers: raw BGR video frames in, all pre-processing on device.
        prep='letterbox_q1': PlayerTracker path (processor BGR->RGB + ultralytics' own flip => the network sees the
            frame's B,G,R in its R,G,B slots; SURVEY App. E q1) + LetterBox.
        prep='pil_square' : PlayerKeypoints/Keypoints path (BGR->RGB, PIL resize to imgsz x imgsz).
        Returned coordinates are in the pre-processed image's pixel space, exactly like model.predict() on the
        processed sample (full frame for letterbox_q1, imgsz x imgsz for pil_square)."""
        fr = self._upload(frames)
        n = fr.shape[0]
        if prep == "letterbox_q1":
            st, orig = self._letterbox(fr, imgsz, (0, 1, 2))
        elif prep == "pil_square":
            st, orig = self._pil_square(fr, imgsz)
        else:
            raise L.PbError(f"unknown prep {prep!r}")
        rows, counts = self._detect(st, n, conf, iou, classes, max_det)
        return self._results_block(rows, counts, n, (st["Hn"], st["Wn"]), orig)

    @torch.no_grad()
    def predict_frames_async(self, frames, prep: str, conf, iou, imgsz, classes=None, max_det=300):
        """predict_frames split in two: enqueue all device work now, return a callable that waits for it and builds
        the Results (lets a caller overlap several trackers' device work with each other's host post-processing).
        One call in flight per engine."""
        fr = self._upload(frames)
        n = fr.shape[0]
        if prep == "letterbox_q1":
            st, orig = self._letterbox(fr, imgsz, (0, 1, 2))
        elif prep == "pil_square":
            st, orig = self._pil_square(fr, imgsz)
        else:
            raise L.PbError(f"unknown prep {prep!r}")
        handle = self._detect_launch(st, n, conf, iou, classes, max_det)

        def finish():
            rows, counts = self._detect_finish(handle)
            return self._results_block(rows, counts, n, (st["Hn"], st["Wn"]), orig)

        return finish
