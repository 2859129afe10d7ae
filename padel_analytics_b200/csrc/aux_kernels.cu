// HBM-bound helper kernels on NHWC fp16 channel slices: 2x2 max-pool, SPPF pooling.
// All move 16-byte vectors (8 channels) per thread with consecutive threads on consecutive channel groups,
// so warps read/write contiguous NHWC runs.
#include "internal.h"
#include "ptx.cuh"

namespace pb {

__device__ __forceinline__ uint4 hmax8(uint4 a, uint4 b) {
  uint4 r;
  const __half2* x = reinterpret_cast<const __half2*>(&a);
  const __half2* y = reinterpret_cast<const __half2*>(&b);
  __half2* z = reinterpret_cast<__half2*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) z[i] = __hmax2(x[i], y[i]);
  return r;
}

// TrackNet nn.MaxPool2d((2,2), stride=(2,2)) — /root/reference/trackers/ball_tracker/models.py:60,62,64
__global__ void maxpool2_kernel(const __half* __restrict__ in, int N, int H, int W, int C, int c_off, int cg,
                                __half* __restrict__ out, int out_C, int out_coff) {
  const int Ho = H / 2, Wo = W / 2;
  const long total = (long)N * Ho * Wo * cg;
  griddep_launch_dependents();
  griddep_wait();
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int g = (int)(i % cg);
    long p = i / cg;
    const int ow = (int)(p % Wo);
    const int oh = (int)((p / Wo) % Ho);
    const int n = (int)(p / ((long)Wo * Ho));
    const __half* b = in + (((size_t)n * H + 2 * oh) * W + 2 * ow) * C + c_off + g * 8;
    const uint4 v00 = *reinterpret_cast<const uint4*>(b);
    const uint4 v01 = *reinterpret_cast<const uint4*>(b + C);
    const uint4 v10 = *reinterpret_cast<const uint4*>(b + (size_t)W * C);
    const uint4 v11 = *reinterpret_cast<const uint4*>(b + (size_t)W * C + C);
    *reinterpret_cast<uint4*>(out + (((size_t)n * Ho + oh) * Wo + ow) * out_C + out_coff + g * 8) =
        hmax8(hmax8(v00, v01), hmax8(v10, v11));
  }
}

// SPPF: y1 = mp5(x'), y2 = mp5(y1), y3 = mp5(y2) with MaxPool2d(5,1,2) (-inf padding).
// buf is the concat buffer (N,H,W,C=4c): slice 0 holds x', slices 1..3 are written.
// One CTA per (image, 8-channel group): the (H,W) plane of 16-byte vectors lives in shared memory and the three
// chained pools run as separable row/column passes (2x5 reads per pool instead of 169 reads per pixel).
__global__ void __launch_bounds__(256) sppf_pool_kernel(__half* __restrict__ buf, int N, int H, int W, int C,
                                                        int cg) {
  extern __shared__ uint4 sppf_smem[];
  uint4* cur = sppf_smem;           // H*W
  uint4* tmp = sppf_smem + H * W;   // H*W (row-pass result)
  const int g = blockIdx.x % cg;
  const int n = blockIdx.x / cg;
  const int c = cg * 8;
  const int HW = H * W;
  __half* base = buf + (size_t)n * HW * C + g * 8;
  griddep_launch_dependents();
  griddep_wait();
  for (int i = threadIdx.x; i < HW; i += blockDim.x) cur[i] = *reinterpret_cast<const uint4*>(base + (size_t)i * C);
  __syncthreads();
  for (int pass = 1; pass <= 3; ++pass) {
    for (int i = threadIdx.x; i < HW; i += blockDim.x) {  // horizontal max over [x-2, x+2]
      const int x = i % W, y = i / W;
      uint4 m = cur[i];
      for (int dx = -2; dx <= 2; ++dx) {
        const int xx = x + dx;
        if (dx != 0 && xx >= 0 && xx < W) m = hmax8(m, cur[y * W + xx]);
      }
      tmp[i] = m;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < HW; i += blockDim.x) {  // vertical max over [y-2, y+2]
      const int x = i % W, y = i / W;
      uint4 m = tmp[i];
      for (int dy = -2; dy <= 2; ++dy) {
        const int yy = y + dy;
        if (dy != 0 && yy >= 0 && yy < H) m = hmax8(m, tmp[yy * W + x]);
      }
      cur[i] = m;
      *reinterpret_cast<uint4*>(base + (size_t)i * C + pass * c) = m;
    }
    __syncthreads();
  }
}

static int grid_for(long total, int threads) {
  long b = (total + threads - 1) / threads;
  const long cap = (long)num_sms() * 16;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

int launch_maxpool2(const void* in, int N, int H, int W, int C, int c_off, int c, void* out, int out_C,
                    int out_coff, cudaStream_t s) {
  PB_CHECK(c % 8 == 0 && c_off % 8 == 0 && C % 8 == 0 && out_C % 8 == 0 && out_coff % 8 == 0,
           "maxpool2: channel slices must be multiples of 8");
  PB_CHECK(H % 2 == 0 && W % 2 == 0, "maxpool2: odd spatial size");
  const long total = (long)N * (H / 2) * (W / 2) * (c / 8);
  PB_CUDA(launch_pdl(maxpool2_kernel, dim3(grid_for(total, 256)), dim3(256), 0, s, 1,
                     reinterpret_cast<const __half*>(in), N, H, W, C, c_off, c / 8, reinterpret_cast<__half*>(out), out_C,
                     out_coff));
  count_launch();
  return 0;
}

int launch_sppf_pool(void* buf, int N, int H, int W, int C, int c, cudaStream_t s) {
  PB_CHECK(c % 8 == 0 && C >= 4 * c && C % 8 == 0, "sppf: bad channel layout");
  const size_t smem = (size_t)2 * H * W * sizeof(uint4);
  PB_CHECK(smem <= 200 * 1024, "sppf: %dx%d plane does not fit in shared memory", H, W);
  PB_CUDA((cudaError_t)ensure_dynamic_smem(reinterpret_cast<const void*>(sppf_pool_kernel), smem));
  PB_CUDA(launch_pdl(sppf_pool_kernel, dim3(N * (c / 8)), dim3(256), smem, s, 1, reinterpret_cast<__half*>(buf), N, H, W,
                     C, c / 8));
  count_launch();
  return 0;
}

}  // namespace pb
