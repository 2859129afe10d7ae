// Epilogue helpers shared by the conv kernels (per-tap conv_tc_kernel and halo conv_halo_kernel).
#pragma once
#include "internal.h"
#include "ptx.cuh"

namespace pb {

// bias + activation on 16 accumulator columns; `act` is CTA-uniform and each case is a straight unrolled loop so
// the 16 independent MUFU chains interleave
__device__ __forceinline__ void bias_act16(const uint32_t (&r)[16], const float* __restrict__ sbias, int act,
                                           float (&v)[16], const __half* __restrict__ res_first = nullptr) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float4 b = *reinterpret_cast<const float4*>(sbias + 4 * q);
    v[4 * q + 0] = __uint_as_float(r[4 * q + 0]) + b.x;
    v[4 * q + 1] = __uint_as_float(r[4 * q + 1]) + b.y;
    v[4 * q + 2] = __uint_as_float(r[4 * q + 2]) + b.z;
    v[4 * q + 3] = __uint_as_float(r[4 * q + 3]) + b.w;
  }
  if (res_first != nullptr) {  // ResNet: the identity joins before the activation
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] += __half2float(res_first[j]);
  }
  if (act == PB_ACT_SILU) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __fdividef(v[i], 1.f + __expf(-v[i]));
  } else if (act == PB_ACT_RELU) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.f);
  } else if (act == PB_ACT_SIGMOID) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __fdividef(1.f, 1.f + __expf(-v[i]));
  }
}

// 32-byte store (STG.256): one instruction and one full 32-byte sector per 16 fp16 channels
__device__ __forceinline__ void st_global_256(void* p, const uint4& a, const uint4& b) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(a.x), "r"(a.y), "r"(a.z),
               "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w)
               : "memory");
}

struct EpiPix {
  bool valid;
  int n, oh, ow;
  size_t pix;
};

// residual / fused head / store of 16 activated channels starting at output channel ch0 (c = column in the N tile)
__device__ __forceinline__ void epilogue_store16(const ConvKParams& kp, const EpiPix& px, int ch0, int c,
                                                 float (&v)[16], float (&hacc)[8]) {
  if (kp.res != nullptr && !kp.res_first) {
    const uint4* rp = reinterpret_cast<const uint4*>(kp.res + px.pix * kp.res_C + kp.res_coff + ch0);
#pragma unroll
    for (int g = 0; g < 2; ++g) {
      const uint4 rv = __ldg(rp + g);
      const __half2* h2 = reinterpret_cast<const __half2*>(&rv);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = __half22float2(h2[j]);
        v[8 * g + 2 * j] += f.x;
        v[8 * g + 2 * j + 1] += f.y;
      }
    }
  }
  if (kp.head_n > 0) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (j < kp.head_n) {
        const float4* w4 = reinterpret_cast<const float4*>(kp.head_w + (size_t)j * kp.BN + c);
        float s0 = 0.f, s1 = 0.f;
#pragma unroll
        for (int q = 0; q < 4; q += 2) {
          const float4 wa = __ldg(w4 + q), wb = __ldg(w4 + q + 1);
          s0 = fmaf(wa.x, v[4 * q], fmaf(wa.y, v[4 * q + 1], fmaf(wa.z, v[4 * q + 2], fmaf(wa.w, v[4 * q + 3], s0))));
          s1 = fmaf(wb.x, v[4 * q + 4], fmaf(wb.y, v[4 * q + 5], fmaf(wb.z, v[4 * q + 6], fmaf(wb.w, v[4 * q + 7], s1))));
        }
        hacc[j] += s0 + s1;
      }
    }
  }
  if (kp.out_mode == PB_OUT_F16_NHWC || kp.out_mode == PB_OUT_F16_NHWC_UP2) {
    uint4 pk[2];
    __half2* h2 = reinterpret_cast<__half2*>(pk);
#pragma unroll
    for (int j = 0; j < 8; ++j) h2[j] = __floats2half2_rn(v[2 * j], v[2 * j + 1]);
    __half* ob = reinterpret_cast<__half*>(kp.out);
    const bool two = (kp.cout_store - ch0 >= 16);  // cout_store is a multiple of 8
    const bool wide = two && (((kp.out_C | kp.out_coff) & 15) == 0);  // 32-byte aligned 16-channel run
    if (kp.out_mode == PB_OUT_F16_NHWC) {
      uint4* op = reinterpret_cast<uint4*>(ob + px.pix * kp.out_C + kp.out_coff + ch0);
      if (wide) {
        st_global_256(op, pk[0], pk[1]);
      } else {
        op[0] = pk[0];
        if (two) op[1] = pk[1];
      }
    } else {
      const int Wo2 = kp.Wo * 2;
#pragma unroll
      for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
          const size_t pix2 = ((size_t)px.n * (kp.Ho * 2) + (px.oh * 2 + dy)) * Wo2 + (px.ow * 2 + dx);
          uint4* op = reinterpret_cast<uint4*>(ob + pix2 * kp.out_C + kp.out_coff + ch0);
          if (wide) {
            st_global_256(op, pk[0], pk[1]);
          } else {
            op[0] = pk[0];
            if (two) op[1] = pk[1];
          }
        }
    }
  } else if (kp.out_mode == PB_OUT_F32_NHWC) {
    float* op = reinterpret_cast<float*>(kp.out) + px.pix * kp.out_C + kp.out_coff + ch0;
    if (((kp.out_C | kp.out_coff) & 3) == 0) {  // 16-byte aligned rows: vector stores for the full groups
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (ch0 + 4 * q + 4 <= kp.cout_store) {
          *reinterpret_cast<float4*>(op + 4 * q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        } else {
#pragma unroll
          for (int j = 4 * q; j < 4 * q + 4; ++j)
            if (ch0 + j < kp.cout_store) op[j] = v[j];
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (ch0 + j < kp.cout_store) op[j] = v[j];
    }
  } else if (kp.out_mode == PB_OUT_F32_NCHW) {
    float* ob = reinterpret_cast<float*>(kp.out);
    const size_t plane = (size_t)kp.Ho * kp.Wo;
    const size_t base = (size_t)px.n * kp.cout_store * plane + (size_t)px.oh * kp.Wo + px.ow;
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (ch0 + j < kp.cout_store) ob[base + (size_t)(ch0 + j) * plane] = v[j];
  }
}

// ------------------------------------------------------------------------------------------------------------
// Fast epilogue for the common case (fp16 NHWC slice out, 32-byte aligned 16-channel runs, no fused head):
// software-pipelined over 16-column chunks -- the tcgen05.ld (and the residual loads) of chunk i+1 are in flight
// while chunk i is activated, packed and stored -- and across the S sub-tiles of a halo tile.
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool epilogue_fast_ok(const ConvKParams& kp) {
  if (kp.head_n != 0 || (kp.res != nullptr && ((kp.res_C | kp.res_coff) & 7) != 0)) return false;
  if ((reinterpret_cast<uintptr_t>(kp.out) & 31) != 0) return false;  // 32-byte stores
  if (kp.out_mode == PB_OUT_F16_NHWC || kp.out_mode == PB_OUT_F16_NHWC_UP2)
    return ((kp.out_C | kp.out_coff) & 15) == 0 && (kp.cout_store & 15) == 0;
  if (kp.out_mode == PB_OUT_F32_NHWC) return ((kp.out_C | kp.out_coff) & 7) == 0;  // 32-byte aligned 8-float groups
  return false;
}

// SiLU on four values with ONE reciprocal: 1/da = db*dc*dd * r, ... with r = 1/(da*db*dc*dd), d = 1 + 2^(-v*log2 e).
// The fast epilogue of a wide SiLU layer is bound by the XU (MUFU) pipe -- ncu on the pose head conv 64->192 @160^2:
// sm__inst_executed_pipe_xu_realtime 75 %, every other pipe < 45 % (profiles/r02_ncu_yolo.md) -- and the plain form
// v / (1 + exp(-v)) costs two MUFU operations per value (EX2 + RCP); this one costs 1.25 plus a few FMULs on the
// idle FMA pipe, with the same few-ulp fp32 accuracy (no approximation of the function itself).
// The exponent is clamped to 2^30 so that the product of four stays finite (< 2^121); silu(v) for v < -20.8 is below
// 2e-8 in magnitude either way, i.e. an fp16 zero / smallest subnormal.
__device__ __forceinline__ void silu4(float& a, float& b, float& c, float& d) {
  constexpr float kNegLog2e = -1.4426950408889634f;
  const float da = 1.f + ex2_approx(fminf(a * kNegLog2e, 30.f));
  const float db = 1.f + ex2_approx(fminf(b * kNegLog2e, 30.f));
  const float dc = 1.f + ex2_approx(fminf(c * kNegLog2e, 30.f));
  const float dd = 1.f + ex2_approx(fminf(d * kNegLog2e, 30.f));
  const float pab = da * db, pcd = dc * dd;
  const float r = rcp_approx(pab * pcd);
  const float rab = pcd * r, rcd = pab * r;  // 1 / (da db), 1 / (dc dd)
  a *= db * rab;
  b *= da * rab;
  c *= dd * rcd;
  d *= dc * rcd;
}

// Where one thread's 16-channel chunk goes: byte pointer of the pixel (channel 0 of the N tile), byte strides of the
// 2x2 replication (UP2 only) and the number of channels of this chunk that exist (fp32 heads may end mid-chunk).
struct EpiOut {
  int mode;       // PB_OUT_F16_NHWC | PB_OUT_F16_NHWC_UP2 | PB_OUT_F32_NHWC   (CTA-uniform)
  size_t dx, dy;  // UP2: bytes to the pixel one to the right / one row down in the upsampled tensor
  int mode2;      // PB_OUT2_*: secondary output (CTA-uniform)
  size_t dx2, dy2;  // PB_OUT2_UP2: the same strides in the secondary tensor
  bool pool_writer;  // PB_OUT2_POOL2: this lane owns the top-left pixel of a 2x2 window
};

// bias + activation (+ residual) of one 16-column chunk of this thread's pixel
__device__ __forceinline__ void epi_add_res16(const uint4 (&rv)[2], float (&v)[16]) {
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    const __half2* h2 = reinterpret_cast<const __half2*>(&rv[g]);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = __half22float2(h2[j]);
      // __fadd_rn: never contracted with the activation's last multiply into an FMA -- the folded epilogue classes
      // would otherwise round differently from the run-time epilogue (which the CTA-pair kernels use), and a frame's
      // result must not depend on which of them its batch size selects (tests/test_full_size_gpu.py)
      v[8 * g + 2 * j] = __fadd_rn(v[8 * g + 2 * j], f.x);
      v[8 * g + 2 * j + 1] = __fadd_rn(v[8 * g + 2 * j + 1], f.y);
    }
  }
}

// has_res: 0 none, 1 residual after the activation, 2 residual before it (CTA-uniform)
__device__ __forceinline__ void epi_compute16(int act, int has_res, uint32_t (&r)[16],
                                              const float* __restrict__ sbias, const uint4 (&rv)[2], float (&v)[16]) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float4 b = *reinterpret_cast<const float4*>(sbias + 4 * q);
    v[4 * q + 0] = __uint_as_float(r[4 * q + 0]) + b.x;
    v[4 * q + 1] = __uint_as_float(r[4 * q + 1]) + b.y;
    v[4 * q + 2] = __uint_as_float(r[4 * q + 2]) + b.z;
    v[4 * q + 3] = __uint_as_float(r[4 * q + 3]) + b.w;
  }
  if (has_res == 2) epi_add_res16(rv, v);
  if (act == PB_ACT_SILU) {  // CTA-uniform
#pragma unroll
    for (int i = 0; i < 4; ++i) silu4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
  } else if (act == PB_ACT_RELU) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.f);
  } else if (act == PB_ACT_SIGMOID) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __fdividef(1.f, 1.f + __expf(-v[i]));
  }
  if (has_res == 1) epi_add_res16(rv, v);
}

__device__ __forceinline__ void epi_chunk(int act, int has_res, const EpiOut& eo, uint32_t (&r)[16],
                                          const float* __restrict__ sbias, char* op, const uint4 (&rv)[2], bool valid,
                                          int nvalid, char* op2 = nullptr, bool vec_tail = false) {
  float v[16];
  epi_compute16(act, has_res, r, sbias, rv, v);
  if (eo.mode == PB_OUT_F32_NHWC) {
    if (!valid) return;
    if (nvalid >= 16) {
      uint4 w[4];
#pragma unroll
      for (int q = 0; q < 4; ++q)
        w[q] = make_uint4(__float_as_uint(v[4 * q]), __float_as_uint(v[4 * q + 1]), __float_as_uint(v[4 * q + 2]),
                          __float_as_uint(v[4 * q + 3]));
      st_global_256(op, w[0], w[1]);
      st_global_256(op + 32, w[2], w[3]);
    } else {  // the N tile ends inside this chunk: one 32-byte store if at least 8 floats exist, scalars for the rest
      float* o = reinterpret_cast<float*>(op);
      int j0 = 0;
      if (vec_tail && nvalid >= 8) {
        st_global_256(op, make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3])),
                      make_uint4(__float_as_uint(v[4]), __float_as_uint(v[5]), __float_as_uint(v[6]), __float_as_uint(v[7])));
        j0 = 8;
      }
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (j >= j0 && j < nvalid) o[j] = v[j];
    }
    return;
  }
  uint4 pk[2];
  __half2* h2 = reinterpret_cast<__half2*>(pk);
#pragma unroll
  for (int j = 0; j < 8; ++j) h2[j] = __floats2half2_rn(v[2 * j], v[2 * j + 1]);
  if (eo.mode2 == PB_OUT2_POOL2) {
    // 2x2 max over the lanes holding (row, col), (row, col^1), (row^1, col), (row^1, col^1) of the 4 x 8 pixel patch of
    // this warp (lane = row_in_patch * 8 + col): two butterfly steps, executed by every lane (a window is entirely
    // valid or entirely invalid: H, W and the tile origins are even)
    uint4 mx[2] = {pk[0], pk[1]};
    __half2* m2 = reinterpret_cast<__half2*>(mx);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      uint32_t w = *reinterpret_cast<uint32_t*>(&m2[j]);
      uint32_t o = __shfl_xor_sync(0xffffffffu, w, 1);
      m2[j] = __hmax2(m2[j], *reinterpret_cast<__half2*>(&o));
      w = *reinterpret_cast<uint32_t*>(&m2[j]);
      o = __shfl_xor_sync(0xffffffffu, w, 8);
      m2[j] = __hmax2(m2[j], *reinterpret_cast<__half2*>(&o));
    }
    if (valid && eo.pool_writer) st_global_256(op2, mx[0], mx[1]);
  }
  if (!valid) return;
  st_global_256(op, pk[0], pk[1]);
  if (eo.mode2 == PB_OUT2_UP2) {
    st_global_256(op2, pk[0], pk[1]);
    st_global_256(op2 + eo.dx2, pk[0], pk[1]);
    st_global_256(op2 + eo.dy2, pk[0], pk[1]);
    st_global_256(op2 + eo.dy2 + eo.dx2, pk[0], pk[1]);
  }
  if (eo.mode == PB_OUT_F16_NHWC_UP2) {
    st_global_256(op + eo.dx, pk[0], pk[1]);
    st_global_256(op + eo.dy, pk[0], pk[1]);
    st_global_256(op + eo.dy + eo.dx, pk[0], pk[1]);
  }
}

// One thread's share of a tile: `S` sub-tiles (accumulator sets `sub_cols` TMEM columns apart, pixels `sub_out` /
// `sub_res` BYTES / halves apart in the output / residual tensors), `nch` 16-column chunks each (`cout_n` channels of
// this N tile exist).  valid_mask bit j = the thread's pixel of sub-tile j exists.  op0 / rp0 point at channel 0 of
// this N tile.  Software pipeline: the tcgen05.ld of chunk i+1 is in flight while chunk i is processed.
// kEpi (a kernel template parameter, chosen per plan by the host -- conv_epi_class): 0 = every case at run time;
// PB_EPI_SILU / PB_EPI_RELU = the plain case (that activation, no residual, fp16 NHWC store, no secondary output),
// PB_EPI_SILU_RES = SiLU then the shortcut add, PB_EPI_F32 = the linear fp32 head outputs, with everything folded at
// compile time.  The epilogue warps of the light layers are issue-latency-bound (two epilogue warps
// per SM sub-partition; profiles/r02_epilogue_stalls.md) and the run-time form spends 14 of its ~285 instructions per
// chunk on CTA-uniform branches.  One epilogue per kernel instantiation: a kernel holding several copies exceeds the
// 128-register budget and spills (measured; same note).
template <int kEpi>
__device__ __forceinline__ void epilogue_fast(const ConvKParams& kp, const EpiOut& eo_in, uint32_t t_addr0, int S,
                                              uint32_t sub_cols, int nch, int cout_n, const float* __restrict__ sbias,
                                              char* op0, const __half* rp0, size_t sub_out, size_t sub_res,
                                              uint32_t valid_mask, char* op20 = nullptr, size_t sub_out2 = 0) {
  uint32_t ra[16], rb[16];
  constexpr bool kSpec = kEpi != PB_EPI_GENERIC;
  EpiOut eo = eo_in;
  if (kSpec) {
    eo.mode = kEpi == PB_EPI_F32 ? PB_OUT_F32_NHWC : PB_OUT_F16_NHWC;
    eo.mode2 = PB_OUT2_NONE;
  }
  const int act = (kEpi == PB_EPI_SILU || kEpi == PB_EPI_SILU_RES) ? PB_ACT_SILU
                  : kEpi == PB_EPI_RELU                            ? PB_ACT_RELU
                  : kEpi == PB_EPI_F32                             ? PB_ACT_NONE
                                                                   : kp.act;
  const int has_res = kEpi == PB_EPI_SILU_RES ? 1 : kSpec ? 0 : (kp.res != nullptr ? (kp.res_first ? 2 : 1) : 0);
  const int cbytes = eo.mode == PB_OUT_F32_NHWC ? 64 : 32;  // bytes of one 16-channel chunk in the output
  int j = 0, c = 0;
  tmem_ld16(t_addr0, ra);
  // the shortcut operand is fetched one chunk ahead, like the accumulator: a global load issued and consumed inside
  // the same chunk would put its whole latency on the chunk's critical path
  constexpr bool kPrefetchRes = kEpi == PB_EPI_SILU_RES;  // (the run-time epilogue has no registers to spare for it)
  uint4 rva[2] = {}, rvb[2] = {};
  if (kPrefetchRes && (valid_mask & 1u)) {
    const uint4* rp = reinterpret_cast<const uint4*>(rp0);
    rva[0] = __ldg(rp);
    rva[1] = __ldg(rp + 1);
  }
#define PB_EPI_STAGE(cur, nxt, rvc, rvn)                                                                \
  {                                                                                                     \
    int jn = j, cn = c + 1;                                                                             \
    if (cn == nch) {                                                                                    \
      cn = 0;                                                                                           \
      ++jn;                                                                                             \
    }                                                                                                   \
    const bool more = jn < S;                                                                           \
    const bool valid = ((valid_mask >> j) & 1u) != 0;                                                   \
    if (kPrefetchRes) {                                                                                 \
      if (more && ((valid_mask >> jn) & 1u)) {                                                          \
        const uint4* rp = reinterpret_cast<const uint4*>(rp0 + (size_t)jn * sub_res + cn * 16);         \
        rvn[0] = __ldg(rp);                                                                             \
        rvn[1] = __ldg(rp + 1);                                                                         \
      }                                                                                                 \
    }                                                                                                   \
    uint4 rvl[2] = {};                                                                                  \
    if (!kPrefetchRes && has_res && valid) { /* consumed after the activation math of this chunk */     \
      const uint4* rp = reinterpret_cast<const uint4*>(rp0 + (size_t)j * sub_res + c * 16);             \
      rvl[0] = __ldg(rp);                                                                               \
      rvl[1] = __ldg(rp + 1);                                                                           \
    }                                                                                                   \
    tmem_ld_wait16(cur);                                                                                \
    if (more) tmem_ld16(t_addr0 + (uint32_t)jn * sub_cols + (uint32_t)(cn * 16), nxt);                  \
    epi_chunk(act, has_res, eo, cur, sbias + c * 16, op0 + (size_t)j * sub_out + (size_t)(c * cbytes), kPrefetchRes ? rvc : rvl, valid, \
              cout_n - c * 16, op20 + (size_t)j * sub_out2 + (size_t)(c * 32), kEpi == PB_EPI_F32);      \
    if (!more) break;                                                                                   \
    j = jn;                                                                                             \
    c = cn;                                                                                             \
  }
  for (;;) {
    PB_EPI_STAGE(ra, rb, rva, rvb)
    PB_EPI_STAGE(rb, ra, rvb, rva)
  }
#undef PB_EPI_STAGE
}

// Two alternative store paths were built and measured on B200 and then removed (profiles/r02_exp_epilogue.md): a
// shared-memory transposition so that every store instruction covers full 128-byte lines (slower on every layer), and
// a TMA bulk-store epilogue (cp.async.bulk.tensor from a swizzled smem tile: 34/34 correctness cases pass, no gain on
// any program, and merely compiling it in cost the product kernels 20 % through register pressure).

}  // namespace pb
