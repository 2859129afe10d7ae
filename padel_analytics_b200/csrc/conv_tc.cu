// Fused conv(k1|k3, s1|s2) + bias + activation (+ residual) as an implicit GEMM on Blackwell tensor cores.
//
//   D[M = 128 output pixels, N = BN out-channels] += A[M, K] * B[N, K]^T,   K = taps x input channels
//
// * A (activations, NHWC fp16) is fetched by TMA in tiled mode: one box = a (TN x TH x TW) patch of pixels x KB
//   channels, shifted by the filter tap; out-of-bounds coordinates are zero-filled by TMA, which implements the
//   conv zero padding for free.  Stride-2 convs read a 5-D view (N, H/2, 2, W/2, 2C) of the same tensor so every
//   tap is again a dense box.  The box lands in shared memory directly in the UMMA K-major swizzled layout
//   (one pixel = one KB*2-byte row; swizzle 32/64/128B == row size).
// * B (weights, fp16 [tap][cout][cin]) is fetched by TMA the same way.
// * warp 0 = TMA producer (activations), warp 6 = TMA producer (weights), warp 1 = tcgen05.mma issuer (whole warp on
//   warp-uniform values, elect.sync-predicated instructions), warps 2-5 / 7-10 / 11-14 = up to three epilogue groups
//   taking tiles round-robin (tcgen05.ld TMEM -> regs -> bias/act/residual -> global).  Up to 8 accumulator sets in
//   TMEM so the epilogues of tiles i-2..i overlap the MMAs of tile i+1.  Persistent CTAs (one per SM, or two for
//   light layers), static tile striding, tile coordinates via fast division.
//
// Replaces: ultralytics Conv/C2f/Bottleneck/Detect convs (3P, SURVEY App. A.2) and TrackNet Conv2DBlock
// (/root/reference/trackers/ball_tracker/models.py:5-17) with BN folded into weight/bias.
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "internal.h"
#include "ptx.cuh"
#include "conv_common.cuh"

namespace pb {

struct ConvSmemTail {
  uint64_t full[kConvMaxStages];
  uint64_t empty[kConvMaxStages];
  uint64_t tmem_full[kConvMaxAcc];
  uint64_t tmem_empty[kConvMaxAcc];
  uint32_t tmem_base;
  uint32_t pad_[3];
  float bias[kConvMaxCout];  // staged once per CTA
};

struct TileCoord {
  int nt, tw, th, tn;
};
__device__ __forceinline__ TileCoord decode_tile(const ConvKParams& kp, int tile) {
  TileCoord c;
  int t;
  fast_divmod(t, c.nt, tile, kp.fd_nt);
  fast_divmod(t, c.tw, t, kp.fd_w);
  fast_divmod(c.tn, c.th, t, kp.fd_h);
  return c;
}

template <int kEpi>
__global__ void __launch_bounds__(kConvMaxThreads, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_w,
               const __grid_constant__ ConvKParams kp) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // 1024B alignment is required by the 128B swizzle pattern; align explicitly (the launch adds 1 KB of slack).
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t stage_bytes = kp.a_bytes + kp.b_bytes;
  ConvSmemTail* tail = reinterpret_cast<ConvSmemTail*>(smem + (size_t)kp.stages * stage_bytes);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // bring-up timeline (libpadel_b200_debug.so only: kp.dbg is NULL in the product build): GPU-wide nanosecond stamps of
  // the first and the last CTA -- entry, after griddepcontrol.wait, exit -- to see how consecutive layers overlap
  const bool gdbg = kp.dbg != nullptr && threadIdx.x == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1);
  long long* gslot = kp.dbg + (3 * 64 + (blockIdx.x == 0 ? 0 : 1)) * 4;
  if (gdbg) gslot[0] = (long long)globaltimer_ns();
  const int k_iters = kp.taps * kp.kblocks;

  if (warp == 0 && lane == 0) tma_prefetch_desc(&tmap_a);
  if (warp == 6 && lane == 0) tma_prefetch_desc(&tmap_w);
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kp.stages; ++i) {
      mbar_init(&tail->full[i], 2);  // A producer + B producer (each arrives with its expected bytes)
      mbar_init(&tail->empty[i], 1);
    }
    for (int i = 0; i < kp.acc_stages; ++i) {
      mbar_init(&tail->tmem_full[i], 1);
      mbar_init(&tail->tmem_empty[i], 4);  // one arrive per epilogue warp
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    tmem_alloc(&tail->tmem_base, (uint32_t)kp.tmem_cols);
    tmem_relinquish();
  }
  for (int i = threadIdx.x; i < kp.cout_pad; i += blockDim.x) tail->bias[i] = kp.bias[i];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tail->tmem_base;
  // PDL: the prologue above touched constant data only; from here on activations are read and written.  The weight
  // producer (warp 6) reads constants only and starts fetching while the previous kernel is still running.
  griddep_launch_dependents();
  if (warp != 6) griddep_wait();
  if (gdbg) gslot[1] = (long long)globaltimer_ns();

  if (warp == 0) {
    // ============================== TMA producer: activations ==============================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const int TW = 1 << kp.tw_log2, TH = 1 << kp.th_log2;
      const int TN = 128 >> (kp.tw_log2 + kp.th_log2);
      int seq = -1;
      for (int tile = blockIdx.x; tile < kp.total_tiles; tile += gridDim.x) {
        const TileCoord tc = decode_tile(kp, tile);
        ++seq;
        const bool dbg = kp.dbg != nullptr && blockIdx.x == 0 && seq < 64;
        if (dbg) kp.dbg[(0 * 64 + seq) * 4 + 0] = clock64();
        for (int tap = 0; tap < kp.taps; ++tap) {
          const int cw = tc.tw * TW + kp.tap_dw[tap];
          const int ch = tc.th * TH + kp.tap_dh[tap];
          const int cc = kp.c_in_off + kp.tap_dc[tap];
          for (int kb = 0; kb < kp.kblocks; ++kb) {
            mbar_wait(&tail->empty[stage], phase ^ 1);
            mbar_arrive_expect_tx(&tail->full[stage], kp.a_bytes);
            tma_load_5d(smem + (size_t)stage * stage_bytes, &tmap_a, &tail->full[stage], cc + kb * kp.KB, cw,
                        kp.tap_d2[tap], ch, tc.tn * TN);
            if (++stage == kp.stages) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
        if (dbg) kp.dbg[(0 * 64 + seq) * 4 + 1] = clock64();
      }
    }
    __syncwarp();
  } else if (warp == 6) {
    // ============================== TMA producer: weights (issued in parallel with warp 0) =================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < kp.total_tiles; tile += gridDim.x) {
        int nt, tq;
        fast_divmod(tq, nt, tile, kp.fd_nt);
        for (int tap = 0; tap < kp.taps; ++tap) {
          for (int kb = 0; kb < kp.kblocks; ++kb) {
            mbar_wait(&tail->empty[stage], phase ^ 1);
            mbar_arrive_expect_tx(&tail->full[stage], kp.b_tx_bytes);
            tma_load_3d(smem + (size_t)stage * stage_bytes + kp.a_bytes, &tmap_w, &tail->full[stage], kb * kp.KB,
                        nt * kp.BN, tap);
            if (++stage == kp.stages) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ============================== UMMA issuer ==============================
    // All 32 lanes run the loop on warp-uniform values (descriptors stay in uniform registers); only the elected
    // lane's tcgen05 instructions take effect.
    {
      const uint32_t lead = elect_one();
      const uint32_t tm_base = __shfl_sync(0xffffffffu, tmem_base, 0);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      const uint32_t swz = (uint32_t)kp.KB * 2u;
      const int ksteps = kp.KB / 16;
      int seq = -1;
      for (int tile = blockIdx.x; tile < kp.total_tiles; tile += gridDim.x) {
        ++seq;
        const bool dbg = kp.dbg != nullptr && blockIdx.x == 0 && seq < 64 && lane == 0;
        if (dbg) kp.dbg[(1 * 64 + seq) * 4 + 0] = clock64();
        mbar_wait(&tail->tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        if (dbg) kp.dbg[(1 * 64 + seq) * 4 + 1] = clock64();
        const uint32_t d_tmem = tm_base + (uint32_t)(acc * kp.acc_cols);
        for (int it = 0; it < k_iters; ++it) {
          mbar_wait(&tail->full[stage], phase);
          tc_fence_after();
          if (dbg && it == 0) kp.dbg[(1 * 64 + seq) * 4 + 2] = clock64();
          const uint32_t a_addr = smem_u32(smem + (size_t)stage * stage_bytes);
          const uint32_t b_addr = a_addr + kp.a_bytes;
          const uint64_t adesc = umma_desc_kmajor(a_addr, swz);
          const uint64_t bdesc = umma_desc_kmajor(b_addr, swz);
#pragma unroll 4
          for (int k = 0; k < ksteps; ++k) {
            // advance 16 K-elements = 32 bytes inside the swizzle row: +2 in the (addr >> 4) field
            umma_f16_p(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), kp.idesc,
                       (uint32_t)((it | k) != 0), lead);
          }
          umma_commit_p(&tail->empty[stage], lead);  // frees the smem slot when these MMAs retire
          if (++stage == kp.stages) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit_p(&tail->tmem_full[acc], lead);  // accumulator ready for the epilogue
        if (dbg) kp.dbg[(1 * 64 + seq) * 4 + 3] = clock64();
        if (++acc == kp.acc_stages) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
    __syncwarp();
  } else {
    // ============ epilogue: up to three groups of 4 warps (2-5, 7-10, 11-14), tiles round-robin; one TMEM lane quarter per warp
    const int egroup = warp >= 7 ? 1 + ((warp - 7) >> 2) : 0;
    const int quarter = warp & 3;
    const int p = quarter * 32 + lane;  // row of the M=128 tile handled by this thread
    const int TWm = (1 << kp.tw_log2) - 1, THm = (1 << kp.th_log2) - 1;
    const int tw_i = p & TWm;
    const int th_i = (p >> kp.tw_log2) & THm;
    const int tn_i = p >> (kp.tw_log2 + kp.th_log2);
    const bool fast = kEpi != PB_EPI_GENERIC || epilogue_fast_ok(kp);  // the host picks a plain class only when it holds
    // per-CTA tile sequence number / accumulator stage / phase advance by counters (egroups <= acc_stages)
    int seq = egroup, acc = egroup;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x + egroup * gridDim.x; egroup < kp.egroups && tile < kp.total_tiles;
         tile += kp.egroups * gridDim.x, seq += kp.egroups) {
      const TileCoord tc = decode_tile(kp, tile);
      EpiPix px;
      px.ow = (tc.tw << kp.tw_log2) + tw_i;
      px.oh = (tc.th << kp.th_log2) + th_i;
      px.n = tc.tn * (128 >> (kp.tw_log2 + kp.th_log2)) + tn_i;
      px.valid = (px.ow < kp.Wo) && (px.oh < kp.Ho) && (px.n < kp.N);
      px.pix = ((size_t)px.n * kp.Ho + px.oh) * kp.Wo + px.ow;
      const bool dbg = kp.dbg != nullptr && blockIdx.x == 0 && seq < 64 && (threadIdx.x == 64 || (threadIdx.x >= 224 && ((threadIdx.x - 224) & 127) == 0));
      if (dbg) kp.dbg[(2 * 64 + seq) * 4 + 0] = clock64();
      mbar_wait(&tail->tmem_full[acc], acc_phase);
      tc_fence_after();
      if (dbg) kp.dbg[(2 * 64 + seq) * 4 + 1] = clock64();
      const uint32_t t_addr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * kp.acc_cols);
      float hacc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // fused 1x1 head partial sums
      const float* sb = tail->bias + tc.nt * kp.BN;
      if (fast) {
        int cn = kp.cout_store - tc.nt * kp.BN;  // channels of this N tile that exist
        cn = cn < kp.BN ? cn : kp.BN;
        if (cn > 0) {
          EpiOut eo;
          eo.mode = kp.out_mode;
          const size_t esz = eo.mode == PB_OUT_F32_NHWC ? 4 : 2;
          const size_t pxb = (size_t)kp.out_C * esz;
          size_t opix = px.pix;
          eo.dx = eo.dy = 0;
          if (eo.mode == PB_OUT_F16_NHWC_UP2) {
            opix = ((size_t)px.n * (2 * kp.Ho) + 2 * px.oh) * (2 * kp.Wo) + 2 * px.ow;
            eo.dx = pxb;
            eo.dy = (size_t)(2 * kp.Wo) * pxb;
          }
          char* obase = reinterpret_cast<char*>(kp.out) + opix * pxb + (size_t)(kp.out_coff + tc.nt * kp.BN) * esz;
          const __half* rbase = kp.res + px.pix * kp.res_C + kp.res_coff + tc.nt * kp.BN;
          eo.mode2 = kp.out2_mode;  // PB_OUT2_NONE | PB_OUT2_UP2 here (pool windows do not map onto this tiling)
          eo.dx2 = eo.dy2 = 0;
          eo.pool_writer = false;
          char* obase2 = nullptr;
          if (eo.mode2 == PB_OUT2_UP2) {
            const size_t pxb2 = (size_t)kp.out2_C * 2;
            const size_t pix2 = ((size_t)px.n * (2 * kp.Ho) + 2 * px.oh) * (2 * kp.Wo) + 2 * px.ow;
            eo.dx2 = pxb2;
            eo.dy2 = (size_t)(2 * kp.Wo) * pxb2;
            obase2 = reinterpret_cast<char*>(kp.out2) + pix2 * pxb2 + (size_t)(kp.out2_coff + tc.nt * kp.BN) * 2;
          }
            epilogue_fast<kEpi>(kp, eo, t_addr, 1, 0u, (cn + 15) >> 4, cn, sb, obase, rbase, 0, 0, px.valid ? 1u : 0u,
                                obase2, 0);
        }
      } else if constexpr (kEpi == PB_EPI_GENERIC) {
      for (int c = 0; c < kp.BN; c += 32) {
        // two 16-column TMEM loads in flight, one wait
        uint32_t r0[16], r1[16];
        const bool second = (c + 16 < kp.BN);
        tmem_ld16(t_addr + (uint32_t)c, r0);
        if (second) tmem_ld16(t_addr + (uint32_t)(c + 16), r1);
        tmem_ld_wait();
        const int ch0 = tc.nt * kp.BN + c;
        if (px.valid && ch0 < kp.cout_store) {
          float v[16];
          bias_act16(r0, sb + c, kp.act, v,
                     (kp.res && kp.res_first) ? kp.res + px.pix * kp.res_C + kp.res_coff + ch0 : nullptr);
          epilogue_store16(kp, px, ch0, c, v, hacc);
        }
        if (second && px.valid && ch0 + 16 < kp.cout_store) {
          float v[16];
          bias_act16(r1, sb + c + 16, kp.act, v,
                     (kp.res && kp.res_first) ? kp.res + px.pix * kp.res_C + kp.res_coff + ch0 + 16 : nullptr);
          epilogue_store16(kp, px, ch0 + 16, c + 16, v, hacc);
        }
      }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tail->tmem_empty[acc]);
      if (dbg) kp.dbg[(2 * 64 + seq) * 4 + 2] = clock64();
      if (kp.head_n > 0 && px.valid) {
        const size_t plane = (size_t)kp.Ho * kp.Wo;
        float* ho = kp.head_out + (size_t)px.n * kp.head_n * plane + (size_t)px.oh * kp.Wo + px.ow;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (j < kp.head_n) ho[(size_t)j * plane] = __fdividef(1.f, 1.f + __expf(-(hacc[j] + __ldg(kp.head_b + j))));
      }
      acc += kp.egroups;
      if (acc >= kp.acc_stages) {
        acc -= kp.acc_stages;
        acc_phase ^= 1u;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (gdbg) gslot[2] = (long long)globaltimer_ns();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)kp.tmem_cols);
  }
}

// ------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------
static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

#ifdef PB_DEBUG_BUILD  // libpadel_b200_debug.so only: clock64 role timelines of CTA 0 (scripts/exp_timeline*.py)
static long long* g_conv_dbg = nullptr;
extern "C" void pb_debug_conv_timeline(long long* buf) { g_conv_dbg = buf; }
#else
static long long* const g_conv_dbg = nullptr;
#endif

// Which epilogue instantiation a layer runs: a plain class when the vectorised epilogue applies (the conditions of
// epilogue_fast_ok) and the layer is activation-only -- no residual, fp16 NHWC store, no secondary output, no fused head.
// The debug library's role timelines (kp.dbg) are recorded by the run-time epilogue only.
int conv_epi_class(const pb_conv_desc* d, const ConvKParams& kp) {
  if (kp.dbg != nullptr) return PB_EPI_GENERIC;
  if (d->head_n != 0 || d->out2_mode != PB_OUT2_NONE || (reinterpret_cast<uintptr_t>(d->out) & 31) != 0)
    return PB_EPI_GENERIC;
  if (d->out_mode == PB_OUT_F32_NHWC) {  // 32-byte aligned 8-float groups
    return (!d->res && d->act == PB_ACT_NONE && ((d->out_C | d->out_coff) & 7) == 0 && d->ksize == 1) ? PB_EPI_F32
                                                                                                       : PB_EPI_GENERIC;
  }
  if (d->out_mode != PB_OUT_F16_NHWC || ((d->out_C | d->out_coff | d->cout_store) & 15) != 0) return PB_EPI_GENERIC;
  if (d->res) {
    const bool ok = !d->res_before_act && d->act == PB_ACT_SILU && ((d->res_C | d->res_coff) & 7) == 0;
    return ok ? PB_EPI_SILU_RES : PB_EPI_GENERIC;
  }
  return d->act == PB_ACT_SILU ? PB_EPI_SILU : (d->act == PB_ACT_RELU ? PB_EPI_RELU : PB_EPI_GENERIC);
}

static int conv_plan_build_impl(const pb_conv_desc* d, ConvPlan* plan) {
  PB_CHECK(d && plan, "conv: null argument");
  PB_CHECK(d->in_layout == PB_IN_NHWC || d->in_layout == PB_IN_STEM4, "conv: bad in_layout");
  const bool stem = d->in_layout == PB_IN_STEM4;
  PB_CHECK(d->ksize == 1 || d->ksize == 3, "conv: ksize %d unsupported", d->ksize);
  PB_CHECK(d->stride == 1 || d->stride == 2, "conv: stride %d unsupported", d->stride);
  PB_CHECK(d->cin > 0 && d->cin % 16 == 0, "conv: cin %d must be a positive multiple of 16", d->cin);
  PB_CHECK(d->cout_pad <= kConvMaxCout, "conv: cout_pad %d > %d", d->cout_pad, kConvMaxCout);
  PB_CHECK(d->cout_pad > 0 && d->cout_pad % 16 == 0, "conv: cout_pad %d must be a multiple of 16", d->cout_pad);
  PB_CHECK(stem || (d->C % 8 == 0 && d->c_in_off >= 0 && d->c_in_off + d->cin <= d->C),
           "conv: bad input channel slice");
  PB_CHECK(d->c_in_off % 8 == 0, "conv: c_in_off must be a multiple of 8");
  PB_CHECK((reinterpret_cast<uintptr_t>(d->in) & 15) == 0 && (reinterpret_cast<uintptr_t>(d->weight) & 15) == 0 &&
               (reinterpret_cast<uintptr_t>(d->bias) & 15) == 0 &&
               (d->out_mode == PB_OUT_NONE || (reinterpret_cast<uintptr_t>(d->out) & 15) == 0),
           "conv: pointers must be 16-byte aligned");
  PB_CHECK(d->stride == 1 || (d->H % 2 == 0 && d->W % 2 == 0), "conv: stride 2 needs even H and W");
  PB_CHECK(d->cout_store > 0 && d->cout_store <= d->cout_pad, "conv: bad cout_store");
  PB_CHECK(d->out_mode >= PB_OUT_F16_NHWC && d->out_mode <= PB_OUT_NONE, "conv: bad out_mode");
  PB_CHECK(d->out_mode != PB_OUT_NONE || d->head_n > 0, "conv: PB_OUT_NONE needs a fused head");
  if (d->head_n > 0) {
    PB_CHECK(d->head_n <= 8 && d->head_weight && d->head_bias && d->head_out, "conv: bad fused head");
    PB_CHECK(d->cout_pad <= 256 && d->cout_store == d->cout_pad, "conv: fused head needs a single full N tile");
    PB_CHECK((reinterpret_cast<uintptr_t>(d->head_weight) & 15) == 0, "conv: head_weight must be 16-byte aligned");
  }
  const bool f16out = d->out_mode == PB_OUT_F16_NHWC || d->out_mode == PB_OUT_F16_NHWC_UP2;
  if (f16out) {
    PB_CHECK(d->cout_store % 8 == 0 && d->out_coff % 8 == 0 && d->out_C % 8 == 0,
             "conv: f16 output needs cout_store/out_coff/out_C multiples of 8");
    PB_CHECK(d->out_coff + d->cout_store <= d->out_C, "conv: output slice exceeds out_C");
  }
  if (d->res) {
    PB_CHECK(d->res_C % 8 == 0 && d->res_coff % 8 == 0 && (reinterpret_cast<uintptr_t>(d->res) & 15) == 0,
             "conv: residual must be 16-byte aligned slices");
  }
  PB_CHECK(d->out2_mode >= PB_OUT2_NONE && d->out2_mode <= PB_OUT2_POOL2, "conv: bad out2_mode");
  if (d->out2_mode != PB_OUT2_NONE) {
    // the secondary store lives in the vectorised epilogue only: 32-byte channel groups on both outputs
    PB_CHECK(d->out_mode == PB_OUT_F16_NHWC && d->head_n == 0 && !stem, "conv: out2 needs a plain f16 NHWC primary output");
    PB_CHECK(d->out2 && (reinterpret_cast<uintptr_t>(d->out2) & 31) == 0 && (reinterpret_cast<uintptr_t>(d->out) & 31) == 0,
             "conv: out2 pointers must be 32-byte aligned");
    PB_CHECK(d->cout_store % 16 == 0 && d->out_C % 16 == 0 && d->out_coff % 16 == 0 && d->out2_C % 16 == 0 &&
                 d->out2_coff % 16 == 0 && d->out2_coff >= 0 && d->out2_coff + d->cout_store <= d->out2_C,
             "conv: out2 needs 16-channel aligned slices");
    if (d->out2_mode == PB_OUT2_POOL2)
      PB_CHECK(d->ksize == 3 && d->stride == 1 && d->H % 2 == 0 && d->W % 2 == 0,
               "conv: PB_OUT2_POOL2 needs a 3x3 stride-1 conv on even H, W");
  }
  EncodeTiledFn encode = get_encode_fn();
  PB_CHECK(encode != nullptr, "conv: cuTensorMapEncodeTiled not available (no CUDA driver?)");

  plan->desc = *d;
  ConvKParams& kp = plan->kp;
  memset(&kp, 0, sizeof(kp));
  kp.cout_pad = d->cout_pad;
  const int s = d->stride;
  kp.N = d->N;
  kp.Ho = d->H / s;
  kp.Wo = d->W / s;
  kp.taps = d->ksize * d->ksize;
  kp.KB = (d->cin % 64 == 0) ? 64 : (d->cin % 32 == 0 ? 32 : 16);
  kp.kblocks = d->cin / kp.KB;
  kp.c_in_off = d->c_in_off;
  kp.bias = d->bias;
  kp.act = d->act;
  kp.res = reinterpret_cast<const __half*>(d->res);
  kp.res_C = d->res_C;
  kp.res_coff = d->res_coff;
  kp.res_first = d->res_before_act ? 1 : 0;
  kp.out = d->out;
  kp.out_C = d->out_C;
  kp.out_coff = d->out_coff;
  kp.out_mode = d->out_mode;
  kp.cout_store = d->cout_store;
  kp.out2 = d->out2;
  kp.out2_C = d->out2_C;
  kp.out2_coff = d->out2_coff;
  kp.out2_mode = d->out2_mode;
  kp.head_w = d->head_weight;
  kp.head_b = d->head_bias;
  kp.head_n = d->head_n;
  kp.head_out = d->head_out;
  kp.dbg = g_conv_dbg;
  plan->variant = 0;
  plan->epi = conv_epi_class(d, kp);
  if (stem) return conv_stem_setup(d, plan, encode);
  {
    // halo variant: for cout <= 192 (the layers the per-tap kernel leaves L2/TMA-bound) unless overridden
    const int mode = conv_override("PADEL_B200_CONV_HALO");
    if (mode == 1 || (mode == 2 && d->cout_pad <= 192)) {
      const int rc = d->ksize == 1    ? conv_halo_1x1_setup(d, plan, encode)
                     : d->stride == 2 ? conv_halo_s2_setup(d, plan, encode)
                                      : conv_halo_setup(d, plan, encode);
      if (rc >= 0) return rc;
    }
  }
  PB_CHECK(d->out2_mode != PB_OUT2_POOL2, "conv: PB_OUT2_POOL2 is only implemented by the halo kernel (cout <= 192)");
  // N tile: largest multiple-of-16 divisor of cout_pad that is <= 256
  int nn = (d->cout_pad + 255) / 256;
  while (d->cout_pad % nn != 0 || (d->cout_pad / nn) % 16 != 0) ++nn;
  kp.n_ntiles = nn;
  kp.BN = d->cout_pad / nn;
  PB_CHECK(kp.BN >= 16 && kp.BN <= 256, "conv: cannot tile cout_pad %d", d->cout_pad);

  // pixel tile shape (TN x TH x TW = 128): minimise the number of tiles, prefer wide tiles
  long best_cost = -1;
  int best_tw = 0, best_th = 0;
  for (int twl = 7; twl >= 2; --twl) {
    for (int thl = 7 - twl; thl >= 0; --thl) {
      const int TW = 1 << twl, TH = 1 << thl, TN = 128 >> (twl + thl);
      const long cost = (long)((kp.Wo + TW - 1) / TW) * ((kp.Ho + TH - 1) / TH) * ((kp.N + TN - 1) / TN);
      if (best_cost < 0 || cost < best_cost) {
        best_cost = cost;
        best_tw = twl;
        best_th = thl;
      }
    }
  }
  kp.tw_log2 = best_tw;
  kp.th_log2 = best_th;
  const int TW = 1 << best_tw, TH = 1 << best_th, TN = 128 >> (best_tw + best_th);
  kp.tiles_w = (kp.Wo + TW - 1) / TW;
  kp.tiles_h = (kp.Ho + TH - 1) / TH;
  kp.tiles_n = (kp.N + TN - 1) / TN;
  kp.total_tiles = kp.tiles_w * kp.tiles_h * kp.tiles_n * kp.n_ntiles;

  for (int r = 0; r < d->ksize; ++r)
    for (int q = 0; q < d->ksize; ++q) {
      const int t = r * d->ksize + q;
      const int dy = r - d->ksize / 2, dx = q - d->ksize / 2;  // input offset relative to s*o
      if (s == 1) {
        kp.tap_dc[t] = 0;
        kp.tap_dw[t] = dx;
        kp.tap_d2[t] = 0;
        kp.tap_dh[t] = dy;
      } else {
        // input col = 2*ow + dx  ->  (w/2 coord, parity): dx=-1 -> (ow-1, 1); 0 -> (ow, 0); 1 -> (ow, 1)
        kp.tap_dw[t] = (dx < 0) ? -1 : 0;
        kp.tap_dc[t] = (dx != 0) ? d->C : 0;
        kp.tap_dh[t] = (dy < 0) ? -1 : 0;
        kp.tap_d2[t] = (dy != 0) ? 1 : 0;
      }
    }
  // TMEM accumulator ring: as many buffers as fit (<= 8) so short-K tiles are not bound by the
  // MMA -> epilogue -> MMA hand-shake latency
  kp.acc_cols = (kp.BN + 31) / 32 * 32;
  kp.acc_stages = 512 / kp.acc_cols;
  if (kp.acc_stages > kConvMaxAcc) kp.acc_stages = kConvMaxAcc;
  kp.idesc = umma_idesc_f16(kp.BN, 0);
  kp.a_bytes = 128u * kp.KB * 2u;
  kp.b_tx_bytes = (uint32_t)kp.BN * kp.KB * 2u;
  kp.b_bytes = (kp.b_tx_bytes + 1023u) & ~1023u;
  const uint32_t stage_bytes = kp.a_bytes + kp.b_bytes;
  // Two CTAs per SM for light layers (small stages, narrow N): each gets half the shared memory and 256 TMEM
  // columns, so one CTA's TMA / epilogue latency is covered by the other's work.
  const bool occ2 = (size_t)stage_bytes * 6 <= 96 * 1024 && kp.acc_cols * 2 <= 256 && kp.total_tiles > num_sms();
  const size_t budget = occ2 ? 96 * 1024 : 200 * 1024;
  int stages = (int)(budget / stage_bytes);
  if (stages > kConvMaxStages) stages = kConvMaxStages;
  PB_CHECK(stages >= 2, "conv: stage too large (%u bytes)", stage_bytes);
  kp.stages = stages;
  plan->smem_bytes = (size_t)stages * stage_bytes + sizeof(ConvSmemTail) + 1024;
  if (occ2) {
    if (kp.acc_stages * kp.acc_cols > 256) kp.acc_stages = 256 / kp.acc_cols;
    kp.tmem_cols = 256;
    kp.egroups = 1;
    plan->threads = 224;
    plan->grid = kp.total_tiles < 2 * num_sms() ? kp.total_tiles : 2 * num_sms();
  } else {
    if (plan->smem_bytes < 120 * 1024) plan->smem_bytes = 120 * 1024;  // force 1 CTA/SM (TMEM: 512 cols)
    kp.tmem_cols = 512;
    kp.egroups = conv_pick_egroups(kp.acc_stages);
    plan->threads = conv_threads_for(kp.egroups);
    plan->grid = kp.total_tiles < num_sms() ? kp.total_tiles : num_sms();
  }
  if (conv_act_tmap(&plan->tmap_a, encode, d, s, kp.KB, TW, 1, TH, TN)) return 1;
  return conv_weight_tmap(&plan->tmap_w, encode, d, kp.taps, kp.KB, kp.BN, 1);
}

int conv_plan_build(const pb_conv_desc* d, ConvPlan* plan) {
  const int rc = conv_plan_build_impl(d, plan);
  if (rc == 0) {
    plan->kp.fd_w = make_fastdiv(plan->kp.tiles_w);
    plan->kp.fd_h = make_fastdiv(plan->kp.tiles_h);
    plan->kp.fd_nt = make_fastdiv(plan->kp.n_ntiles);
  }
  return rc;
}

int conv_plan_launch(const ConvPlan* plan, cudaStream_t stream) {
  if (plan->variant == 1) return conv_halo_launch(plan, stream);
  typedef void (*TcKernelFn)(CUtensorMap, CUtensorMap, ConvKParams);
  const TcKernelFn fn = plan->epi == PB_EPI_SILU       ? conv_tc_kernel<PB_EPI_SILU>
                        : plan->epi == PB_EPI_RELU     ? conv_tc_kernel<PB_EPI_RELU>
                        : plan->epi == PB_EPI_SILU_RES ? conv_tc_kernel<PB_EPI_SILU_RES>
                        : plan->epi == PB_EPI_F32      ? conv_tc_kernel<PB_EPI_F32>
                                                       : conv_tc_kernel<PB_EPI_GENERIC>;
  PB_CUDA((cudaError_t)ensure_dynamic_smem(reinterpret_cast<const void*>(fn), 227 * 1024));
  PB_CUDA(launch_pdl(fn, dim3(plan->grid), dim3(plan->threads), plan->smem_bytes, stream, 1, plan->tmap_a, plan->tmap_w,
                     plan->kp));
  count_launch();
  return 0;
}

// ------------------------------------------------------------------------------------------------------------
// CUDA-core reference kernel (tests only): same descriptor, one thread per (pixel, out-channel)
// ------------------------------------------------------------------------------------------------------------
__global__ void conv_reference_kernel(pb_conv_desc d, int Ho, int Wo) {
  const long total = (long)d.N * Ho * Wo * d.cout_pad;
  for (long idx = blockIdx.x * (long)blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int co = (int)(idx % d.cout_pad);
    long pixl = idx / d.cout_pad;
    const int ow = (int)(pixl % Wo);
    const int oh = (int)((pixl / Wo) % Ho);
    const int n = (int)(pixl / ((long)Wo * Ho));
    if (co >= d.cout_store) continue;
    const __half* in = reinterpret_cast<const __half*>(d.in);
    const __half* w = reinterpret_cast<const __half*>(d.weight);
    float acc = 0.f;
    const int pad = d.ksize / 2;
    for (int r = 0; r < d.ksize; ++r)
      for (int q = 0; q < d.ksize; ++q) {
        const int ih = oh * d.stride + r - pad, iw = ow * d.stride + q - pad;
        if (ih < 0 || ih >= d.H || iw < 0 || iw >= d.W) continue;
        if (d.in_layout == PB_IN_STEM4) {  // padded 4-channel pixels; weight [r][cout][s*4 + c]
          const __half* ip = in + (((size_t)n * (d.H + 2) + ih + 1) * (d.W + 2) + iw + 1) * 4;
          const __half* wp = w + ((size_t)r * d.cout_pad + co) * 16 + q * 4;
          for (int c = 0; c < 3; ++c) acc += __half2float(ip[c]) * __half2float(wp[c]);
          continue;
        }
        const __half* ip = in + (((size_t)n * d.H + ih) * d.W + iw) * d.C + d.c_in_off;
        const __half* wp = w + ((size_t)(r * d.ksize + q) * d.cout_pad + co) * d.cin;
        for (int c = 0; c < d.cin; ++c) acc += __half2float(ip[c]) * __half2float(wp[c]);
      }
    float v = acc + d.bias[co];
    const size_t pix = ((size_t)n * Ho + oh) * Wo + ow;
    const float resv = d.res ? __half2float(reinterpret_cast<const __half*>(d.res)[pix * d.res_C + d.res_coff + co]) : 0.f;
    if (d.res_before_act) v += resv;
    if (d.act == PB_ACT_RELU) v = fmaxf(v, 0.f);
    else if (d.act == PB_ACT_SILU) v = v / (1.f + expf(-v));
    else if (d.act == PB_ACT_SIGMOID) v = 1.f / (1.f + expf(-v));
    if (!d.res_before_act) v += resv;
    if (d.out_mode == PB_OUT_F16_NHWC) {
      reinterpret_cast<__half*>(d.out)[pix * d.out_C + d.out_coff + co] = __float2half_rn(v);
    } else if (d.out_mode == PB_OUT_F16_NHWC_UP2) {
      for (int dy = 0; dy < 2; ++dy)
        for (int dx = 0; dx < 2; ++dx) {
          const size_t pix2 = ((size_t)n * (Ho * 2) + (oh * 2 + dy)) * (Wo * 2) + (ow * 2 + dx);
          reinterpret_cast<__half*>(d.out)[pix2 * d.out_C + d.out_coff + co] = __float2half_rn(v);
        }
    } else if (d.out_mode == PB_OUT_F32_NHWC) {
      reinterpret_cast<float*>(d.out)[pix * d.out_C + d.out_coff + co] = v;
    } else if (d.out_mode == PB_OUT_F32_NCHW) {
      reinterpret_cast<float*>(d.out)[(((size_t)n * d.cout_store + co) * Ho + oh) * Wo + ow] = v;
    }
    if (d.head_n > 0)  // tests only: head_out pre-zeroed by the caller, receives the pre-sigmoid sums (no bias)
      for (int j = 0; j < d.head_n; ++j)
        atomicAdd(d.head_out + (((size_t)n * d.head_n + j) * Ho + oh) * Wo + ow, d.head_weight[j * d.cout_pad + co] * v);
  }
}

int conv_reference_launch(const pb_conv_desc* d, cudaStream_t stream) {
  PB_CHECK(d != nullptr, "conv_reference: null desc");
  const int Ho = d->H / d->stride, Wo = d->W / d->stride;
  const long total = (long)d->N * Ho * Wo * d->cout_pad;
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 32) blocks = 148 * 32;
  conv_reference_kernel<<<blocks, 256, 0, stream>>>(*d, Ho, Wo);
  PB_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

}  // namespace pb
