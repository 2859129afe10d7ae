// Frame pre-processing on device, bit-exact with the CPU libraries the reference pipeline calls:
//   * OpenCV 8-bit INTER_LINEAR resize + 114 border  (ultralytics LetterBox [3P], used by
//     /root/reference/trackers/players_tracker/players_tracker.py:351-359)
//   * Pillow BICUBIC(antialias) two-pass fixed-point resample
//     (players_keypoints_tracker.py:260-266, keypoints_tracker.py:190-194, ball_tracker/iterable.py:188)
//   * u8 -> fp16 NHWC packing (ToTensor /255; TrackNet window assembly iterable.py:167-199)
// All coefficient tables come from the host (engine/resample.py); kernels do integer arithmetic only.
#include "internal.h"

namespace pb {

__device__ __forceinline__ uint4 pack_px16_first(float a, float b, float c) {
  uint4 v;
  __half2* h = reinterpret_cast<__half2*>(&v);
  h[0] = __floats2half2_rn(a, b);
  h[1] = __floats2half2_rn(c, 0.f);
  h[2] = __floats2half2_rn(0.f, 0.f);
  h[3] = h[2];
  return v;
}

__global__ void letterbox_kernel(const uint8_t* __restrict__ src, int B, int Hs, int Ws, __half* __restrict__ dst,
                                 int Hn, int Wn, int rh, int rw, int top, int left, const int* __restrict__ xofs,
                                 const int* __restrict__ xcoef, const int* __restrict__ yofs,
                                 const int* __restrict__ ycoef, int c0, int c1, int c2, int out_layout) {
  const long total = (long)B * Hn * Wn;
  const bool identity = (rh == Hs && rw == Ws);
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int x = (int)(i % Wn);
    const int y = (int)((i / Wn) % Hn);
    const int b = (int)(i / ((long)Wn * Hn));
    int px[3] = {114, 114, 114};
    const int ry = y - top, rx = x - left;
    if (ry >= 0 && ry < rh && rx >= 0 && rx < rw) {
      const uint8_t* img = src + (size_t)b * Hs * Ws * 3;
      if (identity) {
        const uint8_t* p = img + ((size_t)ry * Ws + rx) * 3;
        px[0] = p[0]; px[1] = p[1]; px[2] = p[2];
      } else {
        const int sx = xofs[rx], sy = yofs[ry];
        const int sx1 = min(sx + 1, Ws - 1), sy1 = min(sy + 1, Hs - 1);
        const int a0 = xcoef[2 * rx], a1 = xcoef[2 * rx + 1];
        const int b0 = ycoef[2 * ry], b1 = ycoef[2 * ry + 1];
        const uint8_t* p00 = img + ((size_t)sy * Ws + sx) * 3;
        const uint8_t* p01 = img + ((size_t)sy * Ws + sx1) * 3;
        const uint8_t* p10 = img + ((size_t)sy1 * Ws + sx) * 3;
        const uint8_t* p11 = img + ((size_t)sy1 * Ws + sx1) * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const int r0 = p00[c] * a0 + p01[c] * a1;  // horizontal pass, 11 fractional bits
          const int r1 = p10[c] * a0 + p11[c] * a1;
          // cv::VResizeLinear<uchar,int,short,FixedPtCast<int,uchar,22>> (scalar form)
          px[c] = (((b0 * (r0 >> 4)) >> 16) + ((b1 * (r1 >> 4)) >> 16) + 2) >> 2;
        }
      }
    }
    const float inv = 1.f / 255.f;
    if (out_layout == 0) {
      uint4* o = reinterpret_cast<uint4*>(dst + (size_t)i * 16);
      o[0] = pack_px16_first(px[c0] * inv, px[c1] * inv, px[c2] * inv);
      o[1] = make_uint4(0, 0, 0, 0);
    } else {  // PB_IN_STEM4: (B, Hn+2, Wn+2, 4), interior only
      const uint4 v = pack_px16_first(px[c0] * inv, px[c1] * inv, px[c2] * inv);
      *reinterpret_cast<uint2*>(dst + (((size_t)b * (Hn + 2) + (y + 1)) * (Wn + 2) + (x + 1)) * 4) =
          make_uint2(v.x, v.y);
    }
  }
}

// Pillow ImagingResampleHorizontal_8bpc / Vertical_8bpc: ss = 1<<21; ss += px*k; out = clip8(ss >> 22)
// Horizontal: one CTA per source row; the row is staged in shared memory with 16-byte loads, every thread then
// produces output pixels from shared memory (3 channels each).
__global__ void __launch_bounds__(256)
pil_horizontal_kernel(const uint8_t* __restrict__ src, int Ws, uint8_t* __restrict__ tmp, int Wo,
                      const int* __restrict__ bounds, const int* __restrict__ kk, int ksize, int swap_rb) {
  extern __shared__ __align__(16) uint8_t hrow[];  // [raw row: Ws*3 bytes, 16-aligned][packed row: Ws uint32]
  const size_t row = blockIdx.x;  // b*Hs + y
  const int rowbytes = Ws * 3;
  const int rawpad = (rowbytes + 15) & ~15;
  uint32_t* packed = reinterpret_cast<uint32_t*>(hrow + rawpad);
  const uint8_t* g = src + row * (size_t)rowbytes;
  if ((rowbytes & 15) == 0 && (reinterpret_cast<uintptr_t>(g) & 15) == 0) {
    for (int i = threadIdx.x; i < rowbytes / 16; i += blockDim.x)
      reinterpret_cast<uint4*>(hrow)[i] = __ldg(reinterpret_cast<const uint4*>(g) + i);
  } else {
    for (int i = threadIdx.x; i < rowbytes; i += blockDim.x) hrow[i] = g[i];
  }
  __syncthreads();
  // one 32-bit word per pixel (c0 | c1<<8 | c2<<16): a filter tap then costs one shared-memory load, not three
  for (int x = threadIdx.x; x < Ws; x += blockDim.x)
    packed[x] = (uint32_t)hrow[3 * x] | ((uint32_t)hrow[3 * x + 1] << 8) | ((uint32_t)hrow[3 * x + 2] << 16);
  __syncthreads();
  uint8_t* o = tmp + row * (size_t)Wo * 3;
  for (int xo = threadIdx.x; xo < Wo; xo += blockDim.x) {
    const int xmin = bounds[2 * xo], xs = bounds[2 * xo + 1];
    const int* k = kk + (size_t)xo * ksize;
    const uint32_t* p = packed + xmin;
    int s0 = 1 << 21, s1 = 1 << 21, s2 = 1 << 21;
    for (int x = 0; x < xs; ++x) {
      const int kv = __ldg(k + x);
      const uint32_t px = p[x];
      s0 += (int)(px & 0xFF) * kv;
      s1 += (int)((px >> 8) & 0xFF) * kv;
      s2 += (int)((px >> 16) & 0xFF) * kv;
    }
    const uint8_t v0 = (uint8_t)min(max(s0 >> 22, 0), 255);
    const uint8_t v1 = (uint8_t)min(max(s1 >> 22, 0), 255);
    const uint8_t v2 = (uint8_t)min(max(s2 >> 22, 0), 255);
    o[3 * xo + 0] = swap_rb ? v2 : v0;
    o[3 * xo + 1] = v1;
    o[3 * xo + 2] = swap_rb ? v0 : v2;
  }
}

// Horizontal, R source rows per CTA (the product path when Ws % 16 == 0): the same arithmetic, organised so that
// a thread computes output column xo for R rows with ONE read of its window bounds and filter taps, rows are packed to
// one 32-bit word per pixel straight from 16-byte global loads (48 bytes = 16 pixels per step, no byte-wise staging),
// and the R output rows -- contiguous in `tmp` -- leave through shared memory as 16-byte stores.  The one-row kernel
// above spends ~12 instructions per row and tap (it is instruction-bound: 175 us for 32 x 1080p -> 1280 columns,
// 5 x its HBM time); this one ~8, and the byte-wise stage / pack / scattered byte stores are gone.
template <int R>
__global__ void __launch_bounds__(256)
pil_horizontal_rows_kernel(const uint8_t* __restrict__ src, int Ws, long rows_total, uint8_t* __restrict__ tmp, int Wo,
                           const int* __restrict__ bounds, const int* __restrict__ kk, int ksize, int swap_rb) {
  extern __shared__ __align__(16) uint8_t hrow[];  // [R][Ws] uint32 pixels | [R][Wo*3] output bytes
  uint32_t* packed = reinterpret_cast<uint32_t*>(hrow);
  uint8_t* stage = hrow + (size_t)R * Ws * 4;
  const long row0 = (long)blockIdx.x * R;
  const int rows = (int)(rows_total - row0 < R ? rows_total - row0 : R);
  const int groups = Ws / 16;  // 16 pixels = 48 bytes = three 16-byte loads
  for (int i = threadIdx.x; i < rows * groups; i += blockDim.x) {
    const int r = i / groups, g = i - r * groups;
    const uint4* gp = reinterpret_cast<const uint4*>(src + (row0 + r) * (size_t)Ws * 3) + 3 * g;
    const uint4 a = __ldg(gp), b = __ldg(gp + 1), c = __ldg(gp + 2);
    const uint32_t w[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
    uint32_t px[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {  // 4 pixels per 3 words; the top byte of a packed pixel is never read
      px[4 * q + 0] = w[3 * q];
      px[4 * q + 1] = __byte_perm(w[3 * q], w[3 * q + 1], 0x0543);
      px[4 * q + 2] = __byte_perm(w[3 * q + 1], w[3 * q + 2], 0x0432);
      px[4 * q + 3] = w[3 * q + 2] >> 8;
    }
    uint4* pp = reinterpret_cast<uint4*>(packed + (size_t)r * Ws + 16 * g);
#pragma unroll
    for (int q = 0; q < 4; ++q) pp[q] = make_uint4(px[4 * q], px[4 * q + 1], px[4 * q + 2], px[4 * q + 3]);
  }
  __syncthreads();
  const int orow = Wo * 3;
  for (int xo = threadIdx.x; xo < Wo; xo += blockDim.x) {
    const int xmin = bounds[2 * xo], xs = bounds[2 * xo + 1];
    const int* k = kk + (size_t)xo * ksize;
    const uint32_t* p = packed + xmin;
    int s[R][3];
#pragma unroll
    for (int r = 0; r < R; ++r) s[r][0] = s[r][1] = s[r][2] = 1 << 21;
#pragma unroll 2
    for (int x = 0; x < xs; ++x) {
      const int kv = __ldg(k + x);
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const uint32_t v = p[(size_t)r * Ws + x];
        s[r][0] += (int)(v & 0xFF) * kv;
        s[r][1] += (int)((v >> 8) & 0xFF) * kv;
        s[r][2] += (int)((v >> 16) & 0xFF) * kv;
      }
    }
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const uint8_t v0 = (uint8_t)min(max(s[r][0] >> 22, 0), 255);
      const uint8_t v1 = (uint8_t)min(max(s[r][1] >> 22, 0), 255);
      const uint8_t v2 = (uint8_t)min(max(s[r][2] >> 22, 0), 255);
      uint8_t* o = stage + (size_t)r * orow + 3 * xo;
      o[0] = swap_rb ? v2 : v0;
      o[1] = v1;
      o[2] = swap_rb ? v0 : v2;
    }
  }
  __syncthreads();
  // rows row0 .. row0+rows-1 of `tmp` are one contiguous run of rows * Wo * 3 bytes (Wo % 4 == 0 -> 4-byte multiples;
  // 16-byte vectors when the run starts on a 16-byte boundary, i.e. (R * Wo * 3) % 16 == 0)
  uint8_t* o = tmp + (size_t)row0 * orow;
  const int nbytes = rows * orow;
  if ((reinterpret_cast<uintptr_t>(o) & 15) == 0 && (nbytes & 15) == 0) {
    for (int i = threadIdx.x; i < nbytes / 16; i += blockDim.x)
      reinterpret_cast<uint4*>(o)[i] = reinterpret_cast<const uint4*>(stage)[i];
  } else {
    for (int i = threadIdx.x; i < nbytes / 4; i += blockDim.x)
      reinterpret_cast<uint32_t*>(o)[i] = reinterpret_cast<const uint32_t*>(stage)[i];
  }
}

// Vertical: one thread per 4 output pixels (12 bytes = three 32-bit words per tap row).  Writes the uint8 result
// and/or the normalised fp16 network input directly (f16_layout 0: NHWC16, 1: PB_IN_STEM4 padded 4-channel).
__global__ void pil_vertical_kernel(const uint8_t* __restrict__ tmp, int B, int Hs, int Wo, uint8_t* __restrict__ dst,
                                    int Ho, const int* __restrict__ bounds, const int* __restrict__ kk, int ksize,
                                    __half* __restrict__ dst_f16, int f16_layout) {
  const int groups = Wo / 4;  // Wo % 4 == 0 (checked on the host)
  const long total = (long)B * Ho * groups;
  const int rowwords = Wo * 3 / 4;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int gidx = (int)(i % groups);
    const int yo = (int)((i / groups) % Ho);
    const int b = (int)(i / ((long)groups * Ho));
    const int ymin = bounds[2 * yo], ys = bounds[2 * yo + 1];
    const int* k = kk + (size_t)yo * ksize;
    const uint32_t* p = reinterpret_cast<const uint32_t*>(tmp) + ((size_t)b * Hs + ymin) * rowwords + gidx * 3;
    int s[12];
#pragma unroll
    for (int j = 0; j < 12; ++j) s[j] = 1 << 21;
    for (int y = 0; y < ys; ++y) {
      const int kv = __ldg(k + y);
      const uint32_t w0 = __ldg(p + (size_t)y * rowwords), w1 = __ldg(p + (size_t)y * rowwords + 1),
                     w2 = __ldg(p + (size_t)y * rowwords + 2);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        s[j] += (int)((w0 >> (8 * j)) & 0xFF) * kv;
        s[4 + j] += (int)((w1 >> (8 * j)) & 0xFF) * kv;
        s[8 + j] += (int)((w2 >> (8 * j)) & 0xFF) * kv;
      }
    }
    int v[12];
#pragma unroll
    for (int j = 0; j < 12; ++j) v[j] = min(max(s[j] >> 22, 0), 255);
    if (dst != nullptr) {
      uint32_t* o = reinterpret_cast<uint32_t*>(dst) + ((size_t)b * Ho + yo) * rowwords + gidx * 3;
      o[0] = v[0] | (v[1] << 8) | (v[2] << 16) | (v[3] << 24);
      o[1] = v[4] | (v[5] << 8) | (v[6] << 16) | (v[7] << 24);
      o[2] = v[8] | (v[9] << 8) | (v[10] << 16) | (v[11] << 24);
    }
    if (dst_f16 != nullptr) {
      const float inv = 1.f / 255.f;
      const int x0 = gidx * 4;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const uint4 pk = pack_px16_first(v[3 * q] * inv, v[3 * q + 1] * inv, v[3 * q + 2] * inv);
        if (f16_layout == 0) {
          uint4* o = reinterpret_cast<uint4*>(dst_f16 + (((size_t)b * Ho + yo) * Wo + x0 + q) * 16);
          o[0] = pk;
          o[1] = make_uint4(0, 0, 0, 0);
        } else if (f16_layout == 1) {
          *reinterpret_cast<uint2*>(dst_f16 + (((size_t)b * (Ho + 2) + yo + 1) * (Wo + 2) + x0 + q + 1) * 4) =
              make_uint2(pk.x, pk.y);
        } else {  // 2: plain 4-channel pixels (B,Ho,Wo,4)
          *reinterpret_cast<uint2*>(dst_f16 + (((size_t)b * Ho + yo) * Wo + x0 + q) * 4) = make_uint2(pk.x, pk.y);
        }
      }
    }
  }
}

__global__ void u8_to_f16_nhwc16_kernel(const uint8_t* __restrict__ src, long npix, __half* __restrict__ dst, int c0,
                                        int c1, int c2, int out_layout, int H, int W) {
  const float inv = 1.f / 255.f;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < npix; i += (long)gridDim.x * blockDim.x) {
    const uint8_t* p = src + i * 3;
    const uint4 v = pack_px16_first(p[c0] * inv, p[c1] * inv, p[c2] * inv);
    if (out_layout == 0) {
      uint4* o = reinterpret_cast<uint4*>(dst + i * 16);
      o[0] = v;
      o[1] = make_uint4(0, 0, 0, 0);
    } else {  // PB_IN_STEM4
      const int x = (int)(i % W);
      const long q = i / W;
      const int y = (int)(q % H);
      const long b = q / H;
      *reinterpret_cast<uint2*>(dst + ((b * (H + 2) + (y + 1)) * (W + 2) + (x + 1)) * 4) = make_uint2(v.x, v.y);
    }
  }
}

// x[b, h, w, :] = [median(3), frame[first+b+0](3), ..., frame[first+b+7](3), 0*5]   (32 channels, fp16)
// frames / median are already normalised fp16 4-channel pixels (written by the resize pass): one thread per pixel
// gathers nine 8-byte pixels and writes one 64-byte row.
__global__ void tracknet_pack_kernel(const uint2* __restrict__ frames, int ring, int first_slot,
                                     const uint2* __restrict__ median, int B, int HW, uint4* __restrict__ x) {
  const long total = (long)B * HW;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int pix = (int)(i % HW);
    const int b = (int)(i / HW);
    unsigned short h[32];
    {
      const uint2 m = __ldg(median + pix);
      h[0] = (unsigned short)(m.x & 0xFFFF);
      h[1] = (unsigned short)(m.x >> 16);
      h[2] = (unsigned short)(m.y & 0xFFFF);
    }
#pragma unroll
    for (int f = 0; f < 8; ++f) {
      const int slot = (first_slot + b + f) % ring;
      const uint2 p = __ldg(frames + (size_t)slot * HW + pix);
      h[3 + 3 * f] = (unsigned short)(p.x & 0xFFFF);
      h[4 + 3 * f] = (unsigned short)(p.x >> 16);
      h[5 + 3 * f] = (unsigned short)(p.y & 0xFFFF);
    }
#pragma unroll
    for (int j = 27; j < 32; ++j) h[j] = 0;
    uint4* o = x + i * 4;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      uint4 v;
      v.x = (uint32_t)h[8 * q + 0] | ((uint32_t)h[8 * q + 1] << 16);
      v.y = (uint32_t)h[8 * q + 2] | ((uint32_t)h[8 * q + 3] << 16);
      v.z = (uint32_t)h[8 * q + 4] | ((uint32_t)h[8 * q + 5] << 16);
      v.w = (uint32_t)h[8 * q + 6] | ((uint32_t)h[8 * q + 7] << 16);
      o[q] = v;
    }
  }
}

static int grid_for(long total, int threads) {
  long b = (total + threads - 1) / threads;
  const long cap = (long)num_sms() * 32;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

}  // namespace pb

using namespace pb;

extern "C" {

int pb_letterbox_u8_f16(const uint8_t* src, int B, int Hs, int Ws, void* dst, int Hn, int Wn, int rh, int rw,
                        int top, int left, const int32_t* xofs, const int32_t* xcoef, const int32_t* yofs,
                        const int32_t* ycoef, int c0, int c1, int c2, int out_layout, void* stream) {
  PB_CHECK(src && dst, "letterbox: null pointer");
  PB_CHECK(out_layout == 0 || out_layout == 1, "letterbox: bad out_layout");
  PB_CHECK((rh == Hs && rw == Ws) || (xofs && xcoef && yofs && ycoef), "letterbox: missing tables");
  PB_CHECK(top >= 0 && left >= 0 && top + rh <= Hn && left + rw <= Wn, "letterbox: bad geometry");
  const long total = (long)B * Hn * Wn;
  letterbox_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      src, B, Hs, Ws, reinterpret_cast<__half*>(dst), Hn, Wn, rh, rw, top, left, xofs, xcoef, yofs, ycoef, c0, c1,
      c2, out_layout);
  PB_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int pb_pil_resize_u8(const uint8_t* src, int B, int Hs, int Ws, uint8_t* tmp, uint8_t* dst, int Ho, int Wo,
                     const int32_t* bounds_h, const int32_t* kk_h, int ksize_h, const int32_t* bounds_v,
                     const int32_t* kk_v, int ksize_v, int swap_rb, void* dst_f16, int f16_layout, void* stream) {
  PB_CHECK(src && tmp && (dst || dst_f16) && bounds_h && kk_h && bounds_v && kk_v, "pil_resize: null pointer");
  PB_CHECK(Wo % 4 == 0, "pil_resize: output width %d must be a multiple of 4", Wo);
  PB_CHECK(f16_layout >= 0 && f16_layout <= 2, "pil_resize: bad f16_layout");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const size_t hsmem = (((size_t)Ws * 3 + 15) & ~(size_t)15) + (size_t)Ws * 4;
  // 4 (or 2) rows per CTA when the source rows are whole 48-byte groups (every video format in practice) and 16-byte
  // aligned; one row per CTA otherwise
  const long rows_total = (long)B * Hs;
  const size_t smem4 = (size_t)4 * Ws * 4 + (size_t)4 * Wo * 3;
  const size_t smem2 = (size_t)2 * Ws * 4 + (size_t)2 * Wo * 3;
  if (Ws % 16 == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0 && smem2 <= 200 * 1024) {
    if (smem4 <= 100 * 1024) {
      PB_CUDA((cudaError_t)ensure_dynamic_smem(reinterpret_cast<const void*>(&pil_horizontal_rows_kernel<4>), smem4));
      pil_horizontal_rows_kernel<4><<<(unsigned)((rows_total + 3) / 4), 256, smem4, s>>>(src, Ws, rows_total, tmp, Wo,
                                                                                         bounds_h, kk_h, ksize_h, swap_rb);
    } else {
      PB_CUDA((cudaError_t)ensure_dynamic_smem(reinterpret_cast<const void*>(&pil_horizontal_rows_kernel<2>), smem2));
      pil_horizontal_rows_kernel<2><<<(unsigned)((rows_total + 1) / 2), 256, smem2, s>>>(src, Ws, rows_total, tmp, Wo,
                                                                                         bounds_h, kk_h, ksize_h, swap_rb);
    }
  } else {
    PB_CHECK(hsmem <= 48 * 1024, "pil_resize: source rows of %d pixels do not fit the row buffer", Ws);
    pil_horizontal_kernel<<<B * Hs, 256, hsmem, s>>>(src, Ws, tmp, Wo, bounds_h, kk_h, ksize_h, swap_rb);
  }
  PB_CUDA(cudaGetLastError());
  const long t2 = (long)B * Ho * (Wo / 4);
  pil_vertical_kernel<<<grid_for(t2, 256), 256, 0, s>>>(tmp, B, Hs, Wo, dst, Ho, bounds_v, kk_v, ksize_v,
                                                         reinterpret_cast<__half*>(dst_f16), f16_layout);
  PB_CUDA(cudaGetLastError());
  count_launch(2);
  return 0;
}

int pb_u8_to_f16_nhwc16(const uint8_t* src, int B, int H, int W, void* dst, int c0, int c1, int c2, int out_layout,
                        void* stream) {
  PB_CHECK(src && dst, "u8_to_f16: null pointer");
  PB_CHECK(out_layout == 0 || out_layout == 1, "u8_to_f16: bad out_layout");
  const long npix = (long)B * H * W;
  u8_to_f16_nhwc16_kernel<<<grid_for(npix, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      src, npix, reinterpret_cast<__half*>(dst), c0, c1, c2, out_layout, H, W);
  PB_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int pb_tracknet_pack_windows(const void* frames, int ring, int first_slot, const void* median, int B, int H, int W,
                             void* x, void* stream) {
  PB_CHECK(frames && median && x, "tracknet_pack: null pointer");
  PB_CHECK(ring >= 8, "tracknet_pack: ring must hold at least 8 frames");
  const long total = (long)B * H * W;
  tracknet_pack_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const uint2*>(frames), ring, first_slot, reinterpret_cast<const uint2*>(median), B, H * W,
      reinterpret_cast<uint4*>(x));
  PB_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

}  // extern "C"
