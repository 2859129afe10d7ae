/*
 * padel_b200.h — C ABI of libpadel_b200.so: the B200 (sm_100a) per-frame inference engine that replaces the
 * model forwards of the four padel_analytics trackers.
 *
 * The reference (pure Python) has no FFI; its "plugin boundary" is the duck-typed model object each tracker holds:
 *   - YOLO trackers: self.model.predict(list_of_images, conf=, iou=, imgsz=, classes=, max_det=)
 *       trackers/players_tracker/players_tracker.py:303,351-359
 *       trackers/players_keypoints_tracker/players_keypoints_tracker.py:238,285-292
 *       trackers/keypoints_tracker/keypoints_tracker.py:169,238-245
 *   - Ball tracker: self.tracknet(x) + ensemble + heatmap->xy
 *       trackers/ball_tracker/ball_tracker.py:260-266,439-523 ; predict.py:7-39,149-221 ; iterable.py:167-199
 * Every entry point below takes plain device/host pointers, sizes and a cudaStream_t (as void*); no torch types.
 * The Python host side (padel_analytics_b200/engine/*.py) binds them with ctypes and mirrors the reference's
 * predict()/__call__ API above them.  See INTEGRATION.md for the reference-side stub a maintainer would add.
 *
 * Conventions
 *   - Activations are NHWC, IEEE fp16 ("half"), channel counts padded to multiples of 16 with zero channels.
 *   - All functions return 0 on success; on failure they return non-zero and pb_last_error() describes it.
 *   - All launches go to the stream passed in; nothing synchronises unless documented.
 */
#ifndef PADEL_B200_H
#define PADEL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PB_ACT_NONE 0
#define PB_ACT_RELU 1
#define PB_ACT_SILU 2
#define PB_ACT_SIGMOID 3

#define PB_OUT_F16_NHWC 0     /* half, channel slice [out_coff, out_coff+cout_pad) of an NHWC tensor           */
#define PB_OUT_F16_NHWC_UP2 1 /* same, each pixel replicated 2x2 into a (2Ho, 2Wo) tensor (nearest upsample)  */
#define PB_OUT_F32_NHWC 2     /* float, channels [out_coff, out_coff+cout_store) of an NHWC float tensor       */
#define PB_OUT_F32_NCHW 3     /* float, planar (N, cout_store, Ho, Wo)                                         */
#define PB_IN_NHWC 0
#define PB_IN_STEM4 1
#define PB_OUT_NONE 4         /* nothing stored by the conv itself (only valid with a fused head)              */
/* secondary output of a conv whose primary output is PB_OUT_F16_NHWC (out2_mode) */
#define PB_OUT2_NONE 0
#define PB_OUT2_UP2 1   /* also write every pixel 2x2-replicated into a slice of a (2Ho, 2Wo) tensor: the nearest
                           upsample of ultralytics layers 10 / 13 without a separate pass over the data            */
#define PB_OUT2_POOL2 2 /* also write the 2x2/stride-2 max-pool into a slice of a (Ho/2, Wo/2) tensor: TrackNet's
                           MaxPool2d after each encoder block (models.py:60,62,64); 3x3 stride-1 convs only       */

const char* pb_last_error(void);

int pb_version(void);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
long long pb_launch_count(void);

/* ---- fused conv + bias + activation (+ residual) : implicit GEMM on tcgen05 tensor cores ------------------
 * Replaces ultralytics Conv (Conv2d+BN+SiLU, BN folded) and TrackNet Conv2DBlock (models.py:5-17).          */
typedef struct pb_conv_desc {
  const void* in;  /* half NHWC (N,H,W,C); for in_layout == PB_IN_STEM4 see below */
  int N, H, W, C;  /* C = channel stride of the input tensor (multiple of 8)     */
  int c_in_off;    /* first input channel read                                   */
  int cin;         /* channels read (multiple of 16; zero-padded weights beyond the real count) */
  const void* weight; /* half [taps][cout_pad][cin], taps = ksize*ksize, tap = r*ksize+s       */
  const float* bias;  /* float [cout_pad] (folded BN shift or conv bias)                       */
  int cout_pad;       /* multiple of 16                                                        */
  int ksize;          /* 1 or 3 (padding = ksize/2)                                            */
  int stride;         /* 1 or 2 (stride 2 needs even H and W; with ksize 1 it reads every second pixel) */
  int act;            /* PB_ACT_*                                                              */
  const void* res;    /* optional half NHWC residual, or NULL; added after the activation (ultralytics Bottleneck:
                         x + cv2(cv1(x))) unless res_before_act is set                         */
  int res_C, res_coff;
  void* out;
  int out_C;      /* channel stride of the output tensor (elements)                            */
  int out_coff;   /* first output channel written                                              */
  int out_mode;   /* PB_OUT_*                                                                  */
  int cout_store; /* channels actually stored (<= cout_pad); f16 modes require a multiple of 8 */
  /* Optional fused 1x1 head applied to the activated outputs of this conv inside the epilogue (TrackNet predictor,
   * models.py:55,72-73): head_out[n][j][h][w] = sigmoid(sum_c head_weight[j][c] * y[c] + head_bias[j]), j < head_n <= 8.
   * Requires cout_pad <= 256 (one N tile).  With out_mode == PB_OUT_NONE the conv's own output is not stored.   */
  const float* head_weight; /* float [head_n][cout_pad] or NULL */
  const float* head_bias;   /* float [head_n]                   */
  int head_n;
  float* head_out;          /* float (N, head_n, Ho, Wo)        */
  /* PB_IN_NHWC (0): as documented above.  PB_IN_STEM4 (1): the 3-channel network input stored as 4-channel fp16
   * pixels with a one-pixel zero border, i.e. a (N, H+2, W+2, 4) tensor whose pixel (y,x) sits at [y+1][x+1]
   * (written by pb_letterbox_u8_f16 / pb_u8_to_f16 with out_layout = 1).  Only for the 3x3 stride-2 stem conv:
   * C = 4, cin = 16, weight = half [3 filter rows][cout_pad][16] with k = s*4 + c (s = filter column, c = channel;
   * k >= 12 and c == 3 are zero).  One dense TMA box of the tile's raw input pixels serves all three filter rows: the
   * 16-element row of output pixel ow (padded pixels 2ow .. 2ow+3) is read in place, 16 bytes after its neighbour's. */
  int in_layout;
  /* 1: out = act(conv + bias + res) -- the torchvision ResNet Bottleneck (relu(bn3(conv3) + identity), the court
   * regressor of keypoints_tracker.py:158-167); 0: out = act(conv + bias) + res.                                 */
  int res_before_act;
  /* optional secondary output (see PB_OUT2_*): half NHWC tensor, channel stride out2_C, first channel out2_coff */
  void* out2;
  int out2_C, out2_coff, out2_mode;
} pb_conv_desc;

/* One-shot launches (plan + run). The *_reference variant is a plain CUDA-core kernel used by tests to
 * cross-check the tensor-core kernel on the device; it is never used by the engines.                         */
int pb_conv2d(const pb_conv_desc* d, void* stream);
int pb_conv2d_reference(const pb_conv_desc* d, void* stream);

/* ---- programs: an ordered list of device ops over caller-owned buffers, replayed with one call ------------ */
typedef struct pb_program pb_program;
pb_program* pb_program_create(void);
void pb_program_destroy(pb_program* p);
int pb_program_add_conv(pb_program* p, const pb_conv_desc* d);
/* 2x2/s2 max-pool of a channel slice (TrackNet models.py:60,62,64) */
int pb_program_add_maxpool2(pb_program* p, const void* in, int N, int H, int W, int C, int c_off, int c,
                            void* out, int out_C, int out_coff);
/* SPPF pooling: slice0=[0,c) of buf is x'; writes maxpool5, maxpool5^2, maxpool5^3 into slices 1..3 */
int pb_program_add_sppf_pool(pb_program* p, void* buf, int N, int H, int W, int C, int c);
int pb_program_num_ops(const pb_program* p);
/* Kernel that op i launches: 0 conv_tc_kernel (per-tap boxes), 1 conv_halo_kernel (shared halo / stem), 2 maxpool2,
 * 4 sppf_pool (3 and 5 were kernels of earlier versions); -1 if i is out of range. */
int pb_program_op_kernel(const pb_program* p, int i);
int pb_program_run(pb_program* p, void* stream);
/* Run ops [first, last) only (per-layer timing / debugging). */
int pb_program_run_range(pb_program* p, int first, int last, void* stream);

/* ---- pre-processing --------------------------------------------------------------------------------------- */
/* cv2.resize(INTER_LINEAR) + copyMakeBorder(114) + channel pick + /255 -> half NHWC with 16 channels (3 real).
 * Bit-exact restatement of OpenCV's 11-bit fixed-point bilinear (ultralytics LetterBox; SURVEY App. B.1).
 * src: u8 (B,Hs,Ws,3). The resized area (rh,rw) is placed at (top,left) inside (Hn,Wn); everything else is 114.
 * xofs int32[rw], xcoef int32[rw][2], yofs int32[rh], ycoef int32[rh][2]: per-axis source index and 11-bit
 * coefficient pairs computed on the host exactly as cv::resize does. If rh==Hs and rw==Ws the copy is verbatim.
 * (c0,c1,c2): source channel feeding network channel 0,1,2.  out_layout 0: dst = half (B,Hn,Wn,16);
 * out_layout 1 (PB_IN_STEM4): dst = half (B,Hn+2,Wn+2,4), interior written, the zero border left untouched.      */
int pb_letterbox_u8_f16(const uint8_t* src, int B, int Hs, int Ws, void* dst, int Hn, int Wn, int rh, int rw,
                        int top, int left, const int32_t* xofs, const int32_t* xcoef, const int32_t* yofs,
                        const int32_t* ycoef, int c0, int c1, int c2, int out_layout, void* stream);
/* Pillow Image.resize (BICUBIC, reducing_gap=None) two-pass fixed-point resample, bit-exact (SURVEY App. B.2).
 * Coefficients are computed on the host exactly as Pillow does (precompute_coeffs) and passed in:
 *   bounds_*: int32 [out][2] = (xmin, xsize); kk_*: int32 [out][ksize] (22-bit fixed point).
 * src u8 (B,Hs,Ws,3) -> tmp u8 (B,Hs,Wo,3) -> dst u8 (B,Ho,Wo,3) (may be NULL). swap_rb!=0 swaps channels 0/2
 * (BGR->RGB). If dst_f16 != NULL the vertical pass also writes value/255 as the fp16 network input
 * (f16_layout 0: (B,Ho,Wo,16) NHWC; 1: PB_IN_STEM4 (B,Ho+2,Wo+2,4); 2: plain (B,Ho,Wo,4)), saving the u8 round
 * trip. Wo % 4 == 0.                                                                                            */
int pb_pil_resize_u8(const uint8_t* src, int B, int Hs, int Ws, uint8_t* tmp, uint8_t* dst, int Ho, int Wo,
                     const int32_t* bounds_h, const int32_t* kk_h, int ksize_h, const int32_t* bounds_v,
                     const int32_t* kk_v, int ksize_v, int swap_rb, void* dst_f16, int f16_layout, void* stream);
/* u8 (B,H,W,3) -> half NHWC (B,H,W,16): dst[...,k] = src[..., ck]/255 for k<3, 0 otherwise */
int pb_u8_to_f16_nhwc16(const uint8_t* src, int B, int H, int W, void* dst, int c0, int c1, int c2, int out_layout,
                        void* stream);
/* TrackNet window assembly (iterable.py:167-199): frames = ring of resized RGB frames as normalised fp16 4-channel
 * pixels (ring,H,W,4) (written by pb_pil_resize_u8 with f16_layout 2), median likewise (H,W,4) ->
 * x half NHWC (B,H,W,32): channels [med(3), f[first+b+0](3) ... f[first+b+7](3), 0 x5].                          */
int pb_tracknet_pack_windows(const void* frames, int ring, int first_slot, const void* median, int B, int H, int W,
                             void* x, void* stream);

/* ---- YOLOv8 head decode + NMS (ultralytics Detect/Pose decode, ops.non_max_suppression; SURVEY App. A.3-A.4) --- */
typedef struct pb_yolo_level {
  const float* feat; /* float NHWC (B, h, w, fC): [0,64) DFL logits, [cls_off,+nc) class logits, [kpt_off,+nk) kpts */
  int h, w, stride;
} pb_yolo_level;
/* cand: float (B, cap, 6+nk) rows = x1,y1,x2,y2,conf,cls,kpts(raw decoded, network px); cand_count: int (B) (may
 * exceed cap: rows beyond cap are dropped, the caller checks).  Candidates are the anchors whose best class score is
 * > conf and, when `classes` (HOST array of n_classes ids, the `classes=` list of predict()) is not NULL, whose best
 * class is in it.                                                                                                */
int pb_yolo_decode(const pb_yolo_level* levels, int nlevels, int B, int fC, int nc, int nk, int kdim, int cls_off,
                   int kpt_off, float conf, const int* classes, int n_classes, float* cand, int* cand_anchor,
                   int* cand_count, int cap, void* stream);
/* Per-image: sort by (conf desc, anchor asc), greedy NMS with IoU > iou suppression on class-offset boxes
 * (offset 7680*cls), keep first max_det. out: float (B, max_det, 6+nk); out_count int (B).
 * cap <= 4096: everything in shared memory.  Larger capacities (ultralytics keeps up to max_nms = 30000 candidates,
 * cap <= 32768 here) need `scratch` = device buffer of pb_yolo_nms_scratch_bytes(B, cap) bytes, used only by images
 * that actually hold more than 4096 candidates.                                                                  */
size_t pb_yolo_nms_scratch_bytes(int B, int cap);
int pb_yolo_nms(const float* cand, const int* cand_anchor, const int* cand_count, int B, int cap, int rowlen,
                float iou, int max_det, float* out, int* out_count, void* scratch, void* stream);

/* ---- ResNet50 court-keypoint regressor: the non-3x3/1x1 pieces (keypoints_tracker.py:158-167,276-312;
 *      keypoints_tracker/iterable.py:10-41).  The bottleneck stacks are pb_conv2d programs (res_before_act = 1). ---- */
/* ToTensor + Normalize: src u8 (npix,3) RGB -> dst half (npix,4) = ((x/255) - mean[c]) / std[c], channel 3 = 0.
 * mean3 / std3: HOST float[3].                                                                                  */
int pb_u8_normalize_f16(const uint8_t* src, long long npix, const float* mean3, const float* std3, void* dst,
                        void* stream);
/* conv1: 7x7 / stride 2 / pad 3, 3 -> 64, + bias (folded BN) + ReLU.  in half (N,H,W,4) (channel 3 ignored),
 * weight float [(r*7+s)*3+c][64], bias float [64], out half NHWC (N,H/2,W/2,64).                                 */
int pb_resnet_stem7x7(const void* in, int N, int H, int W, const float* weight, const float* bias, void* out,
                      void* stream);
/* MaxPool2d(3, stride 2, padding 1): half NHWC (N,H,W,C) -> (N,(H-1)/2+1,(W-1)/2+1,C), C % 8 == 0.             */
int pb_maxpool3x3s2(const void* in, int N, int H, int W, int C, void* out, void* stream);
/* AdaptiveAvgPool2d(1) + Linear(C -> n_out) + Sigmoid: in half (N,HW,C), weight float [n_out][C], bias float [n_out],
 * out float (N,n_out).                                                                                          */
int pb_avgpool_fc_sigmoid(const void* in, int N, int HW, int C, const float* weight, const float* bias, int n_out,
                          float* out, void* stream);

/* ---- ByteTrack on the host (players_tracker.py:311,367-369: sv.ByteTrack(frame_rate).update_with_detections) ----
 * The order-dependent stage after the players detector, in C++ (no CUDA): Kalman xyah filter, two-stage Hungarian
 * association on 1 - IoU (fused with the score in the first stage), unconfirmed-track handling, lost-track buffer,
 * duplicate pruning; ids count from 1.  One handle per video; frames must be fed in order.                        */
typedef struct pb_bytetrack pb_bytetrack;
pb_bytetrack* pb_bytetrack_create(double track_activation_threshold, int lost_track_buffer,
                                  double minimum_matching_threshold, double frame_rate);
void pb_bytetrack_destroy(pb_bytetrack* bt);
void pb_bytetrack_reset(pb_bytetrack* bt);
/* One frame: boxes float (n,4) xyxy, scores float (n) (HOST pointers) -> ids_out int (n): the track id attached to each
 * detection, -1 for detections without an active track (dropped by update_with_detections).                      */
int pb_bytetrack_update(pb_bytetrack* bt, const float* boxes, const float* scores, int n, int* ids_out);
/* the same for `frames` consecutive frames: counts int (frames), boxes / scores / ids_out concatenated in frame order */
int pb_bytetrack_update_many(pb_bytetrack* bt, const float* boxes, const float* scores, const int* counts, int frames,
                             int* ids_out);

/* ---- InpaintNet (ball_tracker/models.py:101-130, called at ball_tracker.py:573-576) ----------------------- */
/* coor float (N,L,2) normalised coordinates, mask float (N,L) inpaint mask -> out float (N,L,2) = sigmoid(net).
 * weights: float blob, the nine Conv1d layers in forward order (down_1, down_2, down_3, buttleneck.conv_1,
 * buttleneck.conv_2, up_1, up_2, up_3, predictor), each as weight [cout][cin][3] followed by bias [cout]. L <= 32. */
int pb_inpaintnet_forward(const float* coor, const float* mask, int N, int L, const float* weights, float* out,
                          void* stream);

/* ---- TrackNet background median (ball_tracker/iterable.py:58-81) ------------------------------------------- */
/* Per-byte temporal median of T frames: frames u8 (T, frame_bytes) contiguous on the device (frame_bytes % 4 == 0),
 * out u8 (frame_bytes) = np.median(frames, 0).astype(uint8), i.e. (s[(T-1)/2] + s[T/2]) >> 1 per byte position.
 * swap_rb != 0: the frames are 3-channel BGR pixels and the median is written in RGB order (the reference converts
 * every frame BGR->RGB before np.median, iterable.py:63).                                                        */
int pb_median_u8(const uint8_t* frames, int T, long long frame_bytes, uint8_t* out, int swap_rb, void* stream);

/* ---- TrackNet post-processing (ball_tracker.py:449-509 ; predict.py:7-39) ---------------------------------- */
/* Temporal ensemble + >thr. pred: float (S,8,H,W) raw heat-maps of consecutive windows; window index of pred[0]
 * is `first_window`; frames [frame0, frame0+nframes) are produced; total_windows = total_frames-7.
 * mask: u8 (nframes,H,W) (0/1). ens (optional, may be NULL): float (nframes,H,W).                               */
int pb_tracknet_ensemble(const float* pred, int S, int first_window, int total_windows, int frame0, int nframes,
                         int H, int W, float thr, uint8_t* mask, float* ens, void* stream);
/* 8-connected components of each mask; picks the component with max bbox area (ties: the one whose first pixel in
 * raster order comes last, = cv2.findContours order + predict_location's strict '>' scan).
 * bbox: int (nframes,4) = x,y,w,h (0,0,0,0 if empty). scratch: int32 (nframes, 5, H*W).                          */
int pb_ccl_bbox(const uint8_t* mask, int nframes, int H, int W, int* scratch, int* bbox, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PADEL_B200_H */
