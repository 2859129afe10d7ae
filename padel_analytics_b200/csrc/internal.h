// Internal helpers shared by the translation units of libpadel_b200.so (not part of the C ABI).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdlib>
#include <cstdio>
#include <string>

#include "../../include/padel_b200.h"

namespace pb {

void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }
int num_sms();  // streaming multiprocessors of the current device
// Raise a kernel's dynamic shared-memory limit to at least `bytes` on the CURRENT device (the attribute is per device
// and per function; remembered per (device, function) so the driver call happens once).  Returns a cudaError_t.
int ensure_dynamic_smem(const void* func, size_t bytes);

#ifdef __CUDACC__
// Launch `kernel` with programmatic dependent launch (the programmatic-stream-serialization attribute, see
// ptx.cuh::griddep_wait) and, for cluster > 1, as clusters of that many CTAs: only for kernels that call griddep_wait()
// before touching data another kernel may have written / may still be reading.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              int cluster, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (cluster > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = (unsigned)cluster;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[na].val.programmaticStreamSerializationAllowed = 1;
  ++na;
  cfg.attrs = attr;
  cfg.numAttrs = (unsigned)na;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
  return e == cudaSuccess ? cudaGetLastError() : e;
}
#endif

#define PB_CHECK(cond, ...)         \
  do {                              \
    if (!(cond)) {                  \
      pb::set_error(__VA_ARGS__);   \
      return 1;                     \
    }                               \
  } while (0)

#define PB_CUDA(expr)                                                                          \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      pb::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return 1;                                                                                \
    }                                                                                          \
  } while (0)

// ---- conv plan (built once per layer; holds TMA descriptors + launch geometry) -------------------------------
constexpr int kConvMaxStages = 12;
constexpr int kConvMaxAcc = 8;
// Warp roles of the conv kernels: w0 TMA-A, w1 UMMA issuer, w2-5 epilogue group 0, w6 TMA-B, then 4 warps per further
// epilogue group (w7-10, w11-14).  Epilogue groups take tiles round-robin; more groups = more warps to hide the
// dependent-issue latency of the activation math (ncu: the epilogue warps issue ~20% of the time each).  Three groups
// = 480 threads is the most that keeps 128 registers per thread (19 warps would be capped at 96).
constexpr int kConvThreads = 352;     // two groups
constexpr int kConvMaxThreads = 480;  // three groups
inline int conv_threads_for(int egroups) { return (7 + 4 * (egroups - 1)) * 32; }
// groups for a 1-CTA-per-SM launch: three, but at most one per accumulator stage (a group may only wait one phase ahead)
inline int conv_pick_egroups(int acc_stages) {
  const int want = acc_stages < 3 ? acc_stages : 3;
  return want < 1 ? 1 : want;
}
// Test / bring-up overrides of the kernel choice, never set by the product: tests/test_conv_gpu.py uses them to run the
// per-tap and the halo kernel, and the CTA-pair mode, on the same shapes.  Read at every plan build.
//   PADEL_B200_CONV_HALO: 0 = per-tap kernel only, 1 = halo kernel wherever it applies
//   PADEL_B200_CONV_PAIR: 0 = no CTA pairs, 1 = CTA pairs wherever they apply
// Returns the variable's value, or 2 when it is unset: the product rule.
inline int conv_override(const char* name) {
  const char* e = getenv(name);
  return e ? atoi(e) : 2;
}
constexpr int kConvMaxCout = 2048;  // ResNet50 layer4 (keypoints_tracker.py:158)

// Division by a launch-time constant as multiply-high + shift (dividend < 2^31): the per-tile coordinate decode of the
// persistent kernels would otherwise spend ~25 instructions per runtime `/` or `%` in every warp, every tile.
struct FastDiv {
  uint32_t d, mul, shr;
};
inline FastDiv make_fastdiv(int d) {
  FastDiv f{(uint32_t)d, 0u, 0u};
  if (d > 1) {
    int lg = 0;
    while ((1u << lg) < (uint32_t)d) ++lg;  // ceil(log2 d)
    const int p = 31 + lg;
    f.mul = (uint32_t)(((1ull << p) + (uint32_t)d - 1) / (uint32_t)d);
    f.shr = (uint32_t)(p - 32);
  }
  return f;
}
#ifdef __CUDACC__
__device__ __forceinline__ void fast_divmod(int& q, int& r, int n, const FastDiv& f) {
  q = f.d != 1u ? (int)(__umulhi((uint32_t)n, f.mul) >> f.shr) : n;
  r = n - q * (int)f.d;
}
#endif

struct ConvKParams {
  int N, Ho, Wo;
  int tiles_w, tiles_h, tiles_n, n_ntiles, total_tiles;
  FastDiv fd_w, fd_h, fd_nt;  // dividers by tiles_w, tiles_h, n_ntiles
  int tw_log2, th_log2;  // TW*TH*TN == 128
  int taps, kblocks, KB, BN, stages, cout_pad;
  int c_in_off;
  int tap_dc[9], tap_dw[9], tap_d2[9], tap_dh[9];
  const float* bias;
  int act;
  const __half* res;
  int res_C, res_coff;
  int res_first;  // 1: residual added before the activation (ResNet), 0: after (YOLO Bottleneck)
  void* out;
  int out_C, out_coff, out_mode, cout_store;
  void* out2;  // secondary output (PB_OUT2_*), fast epilogue only
  int out2_C, out2_coff, out2_mode;
  uint32_t idesc;
  uint32_t a_bytes, b_bytes, b_tx_bytes;
  int acc_stages, acc_cols;  // TMEM accumulator ring: acc_stages buffers, acc_cols columns apart
  int tmem_cols;             // TMEM columns allocated by the CTA (power of two; 512 unless two CTAs share an SM)
  int pair;                  // 1: CTA-pair mode (cluster of 2, cta_group::2 UMMAs issued by the even CTA)
  int egroups;               // epilogue warp groups (1 with 224 threads / two CTAs per SM, else 2 or 3)
  const float* head_w;
  const float* head_b;
  int head_n;
  float* head_out;
  int b_resident;  // halo variant: 1 = every weight box is fetched once per CTA and stays in shared memory
  int hs_S, hs_P, hs_G, a_stages, b_stages;  // halo variant: sub-tiles, halo pitch (px), taps per weight box, rings
  uint32_t halo_bytes;
  uint32_t hs_a_row_bytes;  // bytes of one halo row in shared memory (KB*2; 2*KB*2 for the stride-2 pixel-pair rows)
  int hs_ntaps, hs_sbo_rows, hs_x0, hs_y0, hs_tile_h;  // taps served from the halo, 8-row group stride (rows), box origin offsets
  int hs_tap_off[9];                                   // smem row offset of each tap's first pixel
  int hs_tap_desc[9];                                  // the same in 16-byte descriptor units (offset * row_bytes / 16)
  long long* dbg;  // optional timeline buffer (CTA 0, first 64 tiles): [role 0..2][64][4] clock64 stamps
};

struct ConvPlan {
  pb_conv_desc desc;
  ConvKParams kp;
  CUtensorMap tmap_a;
  CUtensorMap tmap_w;
  int grid;
  int threads;
  size_t smem_bytes;
  int variant;  // 0 = per-tap boxes (conv_tc_kernel), 1 = shared halo tile (conv_halo_kernel)
  int epi;      // PB_EPI_*: which epilogue instantiation of the kernel this layer runs
};

// epilogue classes (kernel template parameter kEpi)
#define PB_EPI_GENERIC 0
#define PB_EPI_SILU 1
#define PB_EPI_RELU 2
#define PB_EPI_SILU_RES 3  // SiLU, then + residual (ultralytics Bottleneck shortcut), fp16 NHWC
#define PB_EPI_F32 4       // no activation, fp32 NHWC slice (YOLO head outputs)
int conv_epi_class(const pb_conv_desc* d, const ConvKParams& kp);

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
// Tensor maps shared by the conv set-ups (conv_halo.cu); both return 0, or 1 with the error set.
// K-major weights [taps][cout_pad][cin], box (box_k x box_n x box_taps), swizzled to the box_k * 2-byte rows:
int conv_weight_tmap(CUtensorMap* map, EncodeTiledFn encode, const pb_conv_desc* d, int taps, int box_k, int box_n,
                     int box_taps);
// NHWC activations as the 5-D view (s*C, W/s, s, H/s, N) -- for stride 2 a row holds a horizontal pixel pair and dim 2
// is the image-row parity -- box (box_c, box_w, box_s, box_h, box_n), swizzled to the box_c * 2-byte rows:
int conv_act_tmap(CUtensorMap* map, EncodeTiledFn encode, const pb_conv_desc* d, int s, int box_c, int box_w,
                  int box_s, int box_h, int box_n);
int conv_halo_setup(const pb_conv_desc* d, ConvPlan* plan, EncodeTiledFn encode);  // -1: not applicable
int conv_stem_setup(const pb_conv_desc* d, ConvPlan* plan, EncodeTiledFn encode);
int conv_halo_s2_setup(const pb_conv_desc* d, ConvPlan* plan, EncodeTiledFn encode);  // -1: not applicable
int conv_halo_1x1_setup(const pb_conv_desc* d, ConvPlan* plan, EncodeTiledFn encode);  // -1: not applicable
int conv_halo_launch(const ConvPlan* plan, cudaStream_t stream);
int conv_plan_build(const pb_conv_desc* d, ConvPlan* plan);
int conv_plan_launch(const ConvPlan* plan, cudaStream_t stream);
int conv_reference_launch(const pb_conv_desc* d, cudaStream_t stream);

// aux kernels (aux_kernels.cu)
int launch_maxpool2(const void* in, int N, int H, int W, int C, int c_off, int c, void* out, int out_C,
                    int out_coff, cudaStream_t s);
int launch_sppf_pool(void* buf, int N, int H, int W, int C, int c, cudaStream_t s);

}  // namespace pb
