"""TrackNet (ball heat-map U-Net) on the B200 conv kernels + the fused ball pipeline.

Replaces `self.tracknet` of the reference BallTracker (/root/reference/trackers/ball_tracker/ball_tracker.py:260-266,
called at :445-446) and, through `BallPipeline`, the surrounding CPU stages:
  iterable.py:167-199 (PIL resize + window assembly), ball_tracker.py:449-509,523 (temporal ensemble),
  predict.py:7-39,149-221 (threshold + findContours + bbox).
Network definition being replaced: /root/reference/trackers/ball_tracker/models.py:45-74.
"""
from __future__ import annotations

import numpy as np
import torch

from .. import _lib as L
from . import ops, resample

H_NET, W_NET = 288, 512

# (block name, n convs, cin, cout) in execution order — models.py:48-54
_BLOCKS = [
    ("down_block_1", 2, 27, 64), ("down_block_2", 2, 64, 128), ("down_block_3", 3, 128, 256),
    ("bottleneck", 3, 256, 512), ("up_block_1", 3, 768, 256), ("up_block_2", 2, 384, 128),
    ("up_block_3", 2, 192, 64),
]


class TrackNetEngine:
    """nn.Module-like: __call__(x (B,27,288,512) f32 cuda) -> (B,8,288,512) f32, .to(), .eval(), .load_state_dict()."""

    def __init__(self, state_dict: dict | None = None, max_batch: int = 8, device: str = "cuda",
                 height: int = H_NET, width: int = W_NET):
        if not torch.cuda.is_available():
            raise L.PbError("TrackNetEngine needs a CUDA device (no CPU fallback)")
        L.lib()
        assert height % 8 == 0 and width % 8 == 0
        self.device = torch.device(device)
        self.B, self.H, self.W = max_batch, height, width
        self._w = {}
        self.prog = None
        self._alloc()
        if state_dict is not None:
            self.load_state_dict(state_dict)

    # -- nn.Module-ish surface the reference touches -------------------------------------------------------
    def to(self, device):
        return self

    def eval(self):
        return self

    def load_state_dict(self, sd: dict):
        """Fold BN (eps=1e-5, torch default; models.py:9) and pack to the kernel layout, then (re)build the program."""
        self._w.clear()
        for name, n, cin, cout in _BLOCKS:
            for i in range(1, n + 1):
                p = f"{name}.conv_{i}"
                ci = cin if i == 1 else cout
                w, b = ops.fold_bn(sd[f"{p}.conv.weight"].float(), sd[f"{p}.bn.weight"].float(),
                                   sd[f"{p}.bn.bias"].float(), sd[f"{p}.bn.running_mean"].float(),
                                   sd[f"{p}.bn.running_var"].float(), 1e-5)
                self._w[p] = ops.pack_conv_weight(w, b, ops.pad16(ci) if ci != 27 else 32, cout, self.device)
        # predictor 1x1 (64 -> 8) + sigmoid: a 1x1 tensor-core conv (fp16 weights, N = 16) writing the fp32 NCHW planes
        # -- HBM-bound at ~4.8 TB/s, 158 us per 32 frames (a CUDA-core kernel with fp32 weights took 308 us, issue-bound).
        # The fused-epilogue variant of the conv kernel also exists but costs more (512 FMAs per pixel in the epilogue).
        self._w["predictor"] = ops.pack_conv_weight(sd["predictor.weight"].float().reshape(8, 64, 1, 1),
                                                    sd["predictor.bias"].float(), 64, 16, self.device)
        self._build()
        return self

    # -- buffers + program -----------------------------------------------------------------------------------
    def _alloc(self):
        B, H, W, dev = self.B, self.H, self.W, self.device
        h = lambda hh, ww, c: torch.zeros((B, hh, ww, c), dtype=torch.float16, device=dev)
        self.x = h(H, W, 32)
        self.t1 = h(H, W, 64)
        self.cat3 = h(H, W, 192)  # [up(u2) 128 | x1 64]
        self.p1 = h(H // 2, W // 2, 64)
        self.t2 = h(H // 2, W // 2, 128)
        self.cat2 = h(H // 2, W // 2, 384)  # [up(u1) 256 | x2 128]
        self.p2 = h(H // 4, W // 4, 128)
        self.t3a, self.t3b = h(H // 4, W // 4, 256), h(H // 4, W // 4, 256)
        self.cat1 = h(H // 4, W // 4, 768)  # [up(bottleneck) 512 | x3 256]
        self.p3 = h(H // 8, W // 8, 256)
        self.ba, self.bb = h(H // 8, W // 8, 512), h(H // 8, W // 8, 512)
        self.u1a, self.u1b = h(H // 4, W // 4, 256), h(H // 4, W // 4, 256)
        self.u2a = h(H // 2, W // 2, 128)
        self.u3a, self.u3b = h(H, W, 64), h(H, W, 64)
        # 7 carried windows + B new ones (ball_tracker.py:427-436, :523)
        self.pred = torch.zeros((7 + B, 8, H, W), dtype=torch.float32, device=dev)

    def _build(self):
        P = ops.Program()
        W_ = self._w
        R, UP, SIG = L.ACT_RELU, L.OUT_F16_NHWC_UP2, L.ACT_SIGMOID

        def conv(x, coff, cin, name, out, ooff, mode=L.OUT_F16_NHWC, act=R, k=3, store=None, pool=None):
            w, b = W_[name]
            P.conv(ops.make_conv_desc(x, coff, cin, w, b, k, 1, act, out, ooff, mode, store,
                                      out2=None if pool is None else (pool, 0, L.OUT2_POOL2)),
                   cin_real=27 if name == "down_block_1.conv_1" else cin)

        # MaxPool2d of the first two encoder blocks (models.py:60,62) is a second store of the producing conv
        # (PB_OUT2_POOL2).  The third one stays a launch: its 256-channel conv runs on the per-tap kernel, which has no
        # pooled store.
        conv(self.x, 0, 32, "down_block_1.conv_1", self.t1, 0)
        conv(self.t1, 0, 64, "down_block_1.conv_2", self.cat3, 128, pool=self.p1)
        conv(self.p1, 0, 64, "down_block_2.conv_1", self.t2, 0)
        conv(self.t2, 0, 128, "down_block_2.conv_2", self.cat2, 256, pool=self.p2)
        conv(self.p2, 0, 128, "down_block_3.conv_1", self.t3a, 0)
        conv(self.t3a, 0, 256, "down_block_3.conv_2", self.t3b, 0)
        conv(self.t3b, 0, 256, "down_block_3.conv_3", self.cat1, 512)
        P.maxpool2(self.cat1, 512, 256, self.p3, 0)
        conv(self.p3, 0, 256, "bottleneck.conv_1", self.ba, 0)
        conv(self.ba, 0, 512, "bottleneck.conv_2", self.bb, 0)
        conv(self.bb, 0, 512, "bottleneck.conv_3", self.cat1, 0, UP)  # nearest x2 fused into the store
        conv(self.cat1, 0, 768, "up_block_1.conv_1", self.u1a, 0)
        conv(self.u1a, 0, 256, "up_block_1.conv_2", self.u1b, 0)
        conv(self.u1b, 0, 256, "up_block_1.conv_3", self.cat2, 0, UP)
        conv(self.cat2, 0, 384, "up_block_2.conv_1", self.u2a, 0)
        conv(self.u2a, 0, 128, "up_block_2.conv_2", self.cat3, 0, UP)
        conv(self.cat3, 0, 192, "up_block_3.conv_1", self.u3a, 0)
        self._pred_new = self.pred[7:]
        conv(self.u3a, 0, 64, "up_block_3.conv_2", self.u3b, 0)
        conv(self.u3b, 0, 64, "predictor", self._pred_new, 0, L.OUT_F32_NCHW, SIG, k=1, store=8)
        self.prog = P

    # -- execution ---------------------------------------------------------------------------------------------
    def run_packed(self):
        """x (B,H,W,32 fp16, already packed) -> pred[7:7+B]."""
        if self.prog is None:
            raise L.PbError("TrackNetEngine: no weights loaded")
        self.prog.run()

    @torch.no_grad()
    def __call__(self, x: torch.Tensor) -> torch.Tensor:
        """Reference-compatible call (ball_tracker.py:445): NCHW fp32 in [0,1] -> (B,8,H,W) fp32 heat-maps."""
        nb = x.shape[0]
        if nb > self.B or tuple(x.shape[1:]) != (27, self.H, self.W):
            raise L.PbError(f"TrackNetEngine: expected (<= {self.B}, 27, {self.H}, {self.W}), got {tuple(x.shape)}")
        self.x[:nb, ..., :27] = x.to(self.device).permute(0, 2, 3, 1).to(torch.float16)
        self.run_packed()
        return self._pred_new[:nb].clone()


class BallPipeline:
    """Frames (BGR u8) -> per-frame ball bbox, entirely on device: PIL-exact resize, window packing, TrackNet,
    temporal ensemble + threshold, connected components.  Mirrors BallTracker.predict_frames' TrackNet stage
    (ball_tracker.py:373-523) including its head/tail ensemble rules (SURVEY App. C)."""

    def __init__(self, engine: TrackNetEngine, frame_hw: tuple[int, int], median_rgb: np.ndarray | torch.Tensor):
        self.eng = engine
        self.dev = engine.device
        self.Hs, self.Ws = frame_hw
        B = engine.B
        self.B = B
        H, W = engine.H, engine.W
        bh, kh, self.ksh = resample.pil_bicubic_tables(self.Ws, W)
        bv, kv, self.ksv = resample.pil_bicubic_tables(self.Hs, H)
        up = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(self.dev)
        self.bh, self.kh, self.bv, self.kv = up(bh), up(kh), up(bv), up(kv)
        self.ring = B + 8
        # resized RGB frames as normalised fp16 4-channel pixels (what the window-packing kernel gathers from)
        self.small = torch.zeros((self.ring, H, W, 4), dtype=torch.float16, device=self.dev)
        self.tmp = torch.zeros((B + 7, self.Hs, W, 3), dtype=torch.uint8, device=self.dev)
        self.stage = torch.zeros((B + 7, self.Hs, self.Ws, 3), dtype=torch.uint8, device=self.dev)
        self.mask = torch.zeros((B + 7, H, W), dtype=torch.uint8, device=self.dev)
        self.scratch = torch.zeros((B + 7, 5, H * W), dtype=torch.int32, device=self.dev)
        self.bbox = torch.zeros((B + 7, 4), dtype=torch.int32, device=self.dev)
        self._host_ring = [torch.zeros((B + 7, 4), dtype=torch.int32).pin_memory() for _ in range(3)]
        self._pending = [None] * 3
        self._turn = 0
        self.ens = None
        self.median_small = torch.zeros((1, H, W, 4), dtype=torch.float16, device=self.dev)
        self._median_src = None
        self.set_median(median_rgb)
        self.reset()

    def set_median(self, median_rgb):
        """(Re)apply the background: full-res RGB -> uint8 -> PIL resize (iterable.py:76-81), on device with the same
        kernel as the frames.  A no-op when called again with the very same array object/contents."""
        med = torch.as_tensor(median_rgb)
        if tuple(med.shape[:2]) != (self.Hs, self.Ws):
            raise L.PbError("median must have the frame resolution")
        med = med.to(torch.uint8)
        if self._median_src is not None and self._median_src.shape == med.shape and \
                torch.equal(self._median_src, med.cpu()):
            return
        self._median_src = med.cpu().clone()
        dev_med = med.to(self.dev).contiguous().view(1, self.Hs, self.Ws, 3)
        self._resize(dev_med, 1, self.median_small, swap_rb=0)

    def reset(self, base: int = 0):
        """base = absolute index of the first frame that will be pushed (= first window computed); > 0 for shards
        that start mid-video (the 7 windows before the shard are recomputed, SURVEY §8e)."""
        self.base = base
        self.n_frames_in = 0  # frames received
        self.n_windows = 0  # windows processed
        self.eng.pred.zero_()

    def _resize(self, src, n, dst_f16, swap_rb):
        """Pillow-exact resize of n frames; the vertical pass writes value/255 as fp16 4-channel pixels into dst_f16."""
        L.check(L.lib().pb_pil_resize_u8(src.data_ptr(), n, self.Hs, self.Ws, self.tmp.data_ptr(), None,
                                         self.eng.H, self.eng.W, self.bh.data_ptr(), self.kh.data_ptr(), self.ksh,
                                         self.bv.data_ptr(), self.kv.data_ptr(), self.ksv, swap_rb, dst_f16.data_ptr(),
                                         2, L.stream_ptr()))

    def push_frames(self, frames_bgr: torch.Tensor):
        """frames: (n,Hs,Ws,3) u8 BGR, host (pinned or not) or device; n <= B+7. Resized into the ring."""
        n = frames_bgr.shape[0]
        if n == 0:
            return
        if frames_bgr.device.type != "cuda":
            self.stage[:n].copy_(frames_bgr, non_blocking=True)
            frames_bgr = self.stage[:n]
        if self.n_frames_in + n > self.n_windows + self.ring:
            raise L.PbError("BallPipeline: frame ring overflow (process windows before pushing more frames)")
        frames_bgr = frames_bgr.contiguous()
        start = self.n_frames_in % self.ring
        first = min(n, self.ring - start)  # resize straight into the ring (two runs when it wraps)
        self._resize(frames_bgr[:first], first, self.small[start:start + first], swap_rb=1)
        if first < n:
            self._resize(frames_bgr[first:], n - first, self.small[: n - first], swap_rb=1)
        self.n_frames_in += n

    def windows_ready(self) -> int:
        return max(0, self.n_frames_in - 7) - self.n_windows

    def run_windows(self, nb: int, total_frames: int, want_ens: bool = False):
        """Process the next nb windows (nb <= B). Returns (first_frame, host int32 (nframes,4) bboxes) for the frames
        emitted: absolute frames [first_frame, first_frame+nframes)."""
        return self.run_windows_async(nb, total_frames, want_ens)()

    def run_windows_async(self, nb: int, total_frames: int, want_ens: bool = False):
        """Enqueue the device work for the next nb windows; returns a callable that waits and yields
        (first_frame, bboxes).  One call in flight."""
        eng = self.eng
        assert 0 < nb <= self.B and nb <= self.windows_ready()
        w0 = self.base + self.n_windows  # absolute window index
        total_windows = total_frames - 7
        if w0 + nb > total_windows:
            raise L.PbError("BallPipeline: more windows than total_frames allows")
        L.check(L.lib().pb_tracknet_pack_windows(self.small.data_ptr(), self.ring, self.n_windows % self.ring,
                                                 self.median_small.data_ptr(), nb, eng.H, eng.W, eng.x.data_ptr(),
                                                 L.stream_ptr()))
        eng.run_packed()
        nframes = nb + (7 if w0 + nb == total_windows else 0)
        ens_ptr = 0
        if want_ens:
            self.ens = torch.empty((nframes, eng.H, eng.W), dtype=torch.float32, device=self.dev)
            ens_ptr = self.ens.data_ptr()
        L.check(L.lib().pb_tracknet_ensemble(eng.pred.data_ptr(), 7 + nb, w0 - 7, total_windows, w0, nframes, eng.H,
                                             eng.W, 0.5, self.mask.data_ptr(), ens_ptr, L.stream_ptr()))
        L.check(L.lib().pb_ccl_bbox(self.mask.data_ptr(), nframes, eng.H, eng.W, self.scratch.data_ptr(),
                                    self.bbox.data_ptr(), L.stream_ptr()))
        slot = self._turn  # ring of pinned host copies: the caller may enqueue the next batch before collecting this one
        self._turn = (slot + 1) % len(self._host_ring)
        if self._pending[slot] is not None:
            self._pending[slot]()  # an uncollected launch still owns this slot: resolve it first
        host = self._host_ring[slot]
        host[:nframes].copy_(self.bbox[:nframes], non_blocking=True)
        # carry the last 7 windows for the next batch (ball_tracker.py:523)
        carry = eng.pred[nb:nb + 7].clone()
        eng.pred[:7].copy_(carry)
        self.n_windows += nb
        done = torch.cuda.Event()
        done.record()

        state = {"result": None}

        def finish():
            if state["result"] is None:
                done.synchronize()
                state["result"] = (w0, host[:nframes].numpy().copy())
                self._pending[slot] = None
            return state["result"]

        self._pending[slot] = finish
        return finish


def bbox_to_xyv(bbox: np.ndarray, img_scaler: tuple[float, float]):
    """predict.py:203-217 on host with Python float arithmetic (bit-identical to the reference's int() truncations)."""
    xs, ys, vs = [], [], []
    for x, y, w, h in bbox.tolist():
        cx, cy = int(x + w / 2), int(y + h / 2)
        cx, cy = int(cx * img_scaler[0]), int(cy * img_scaler[1])
        xs.append(cx), ys.append(cy), vs.append(0 if (cx == 0 and cy == 0) else 1)
    return xs, ys, vs
