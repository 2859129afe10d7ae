// 3x3 / stride-1 conv + bias + activation as an implicit GEMM whose nine filter taps are all served from ONE
// shared-memory halo tile per 64(32/16)-channel block.
//
// Why: with one TMA box per tap (conv_tc_kernel) every K-block of a small-N layer moves 16 KB of activations for
// four UMMAs and the kernel is bound by L2->SM / TMA delivery (measured 0.35-0.43 PFLOP/s on TrackNet's N=64
// layers).  Here the CTA tile is 16 rows x (8*S) columns of output pixels = S sub-tiles of M=128; its
// (16+2) x (8*S+2) pixel halo is fetched by a single TMA box, and tap (r,s) of sub-tile j is just a different
// UMMA descriptor over the same bytes:
//     start = halo + ((r*P + 8*j + s) * row_bytes),   SBO (8-row group stride) = P * row_bytes,   P = 8*S + 2
// (one 8-row group = 8 horizontally adjacent pixels, consecutive groups = consecutive image rows).  This relies on
// tcgen05 applying the 128/64/32-byte swizzle XOR on absolute shared-memory address bits, which
// scripts/exp_umma_shift.py verified on B200 (descriptor base_offset = 0 is exact for any row shift / any SBO).
// Weights are fetched per (channel block, tap group) by a second producer warp and shared by the S sub-tile MMAs.
//
// Replaces the same reference layers as conv_tc.cu (TrackNet Conv2DBlock models.py:5-17; ultralytics 3x3 convs).
#include <cstdlib>
#include <mutex>
#include <vector>

#include "conv_common.cuh"
#include "internal.h"
#include "ptx.cuh"

namespace pb {

constexpr int kHaloMaxA = 4;
constexpr int kHaloMaxB = 12;

struct HaloSmemTail {
  uint64_t a_full[kHaloMaxA];
  uint64_t a_empty[kHaloMaxA];
  uint64_t b_full[kHaloMaxB];
  uint64_t b_empty[kHaloMaxB];
  uint64_t tmem_full[kConvMaxAcc];
  uint64_t tmem_empty[kConvMaxAcc];
  uint32_t tmem_base;
  uint32_t pad_[3];
  float bias[kConvMaxCout];
};

struct HaloTile {
  int tw, th, n;
};
// pair mode: a "tile" is two vertically adjacent 16-row tiles, one per CTA of the pair (crank = 0 / 1)
__device__ __forceinline__ HaloTile halo_decode(const ConvKParams& kp, int tile, uint32_t crank) {
  HaloTile t;
  int q, th;
  fast_divmod(q, t.tw, tile, kp.fd_w);
  fast_divmod(t.n, th, q, kp.fd_h);
  t.th = kp.pair ? th * 2 + (int)crank : th;
  return t;
}

// row_bytes 128 / 64 / 32: the swizzled K-major layouts.  row_bytes 16: the un-swizzled K-major layout -- 8-row core
// matrices of 16-byte rows at a 16-byte pitch, 8-row groups `sbo_bytes` apart, the second 16-byte half of a K = 16 row
// `lbo_bytes` further (16: the row that follows -- overlapping rows, used by the stem's raw-pixel operand; the roles of
// LBO and SBO in this layout were confirmed on hardware: swapping them fails tests/test_conv_gpu.py::test_stem_*).
__device__ __forceinline__ uint64_t umma_desc_sbo(uint32_t saddr, uint32_t row_bytes, uint32_t sbo_bytes,
                                                  uint32_t lbo_bytes = 16) {
  const uint64_t layout = row_bytes == 128 ? 2ull : (row_bytes == 64 ? 4ull : (row_bytes == 32 ? 6ull : 0ull));
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
         (1ull << 46) | (layout << 61);
}

// kPair is a compile-time switch: a kernel that contains cta_group::2 instructions can only be launched as a
// cluster of two, so the single-CTA and the CTA-pair variants are separate instantiations.
// kS (sub-tiles) and kSteps (16-element k-steps per channel block) are compile-time so the UMMA issue
// loop is straight-line code with immediate descriptor offsets.
template <bool kPair, int kS, int kSteps, int kEpi>
__global__ void __launch_bounds__(kConvMaxThreads, 1)
conv_halo_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_w,
                 const __grid_constant__ ConvKParams kp) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* a_base = smem;
  uint8_t* b_base = smem + (size_t)kp.a_stages * kp.a_bytes;
  HaloSmemTail* tail = reinterpret_cast<HaloSmemTail*>(b_base + (size_t)kp.b_stages * kp.b_bytes);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // bring-up timeline (libpadel_b200_debug.so only: kp.dbg is NULL in the product build): GPU-wide nanosecond stamps of
  // the first and the last CTA -- entry, after griddepcontrol.wait, exit -- to see how consecutive layers overlap
  const bool gdbg = kp.dbg != nullptr && threadIdx.x == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1);
  long long* gslot = kp.dbg + (3 * 64 + (blockIdx.x == 0 ? 0 : 1)) * 4;
  if (gdbg) gslot[0] = (long long)globaltimer_ns();
  constexpr int S = kS;
  const int G = kp.hs_G;
  const uint32_t row_bytes = (uint32_t)kp.KB * 2u;       // weight rows (and activation rows unless stride 2)
  const uint32_t a_row_bytes = kp.hs_a_row_bytes;        // activation (halo) rows
  const int tap_groups = kp.hs_ntaps / G;
  // CTA-pair mode (cluster of 2, cta_group::2): both CTAs load their own halo and half of the weights, the even
  // CTA issues M=256 UMMAs over both, so every SM reads only half of B from its shared memory.
  constexpr int pair = kPair ? 1 : 0;
  const uint32_t crank = pair ? cluster_ctarank() : 0u;
  const int cta0 = pair ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int cstride = pair ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  if (warp == 0 && lane == 0) tma_prefetch_desc(&tmap_a);
  if (warp == 6 && lane == 0) tma_prefetch_desc(&tmap_w);
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kp.a_stages; ++i) {
      mbar_init(&tail->a_full[i], 1);
      mbar_init(&tail->a_empty[i], 1);
    }
    for (int i = 0; i < kp.b_stages; ++i) {
      mbar_init(&tail->b_full[i], 1);
      mbar_init(&tail->b_empty[i], 1);
    }
    for (int i = 0; i < kp.acc_stages; ++i) {
      mbar_init(&tail->tmem_full[i], 1);
      mbar_init(&tail->tmem_empty[i], pair ? 8 : 4);  // one arrive per epilogue warp (of both CTAs in pair mode)
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    if (pair) {
      tmem_alloc2(&tail->tmem_base, (uint32_t)kp.tmem_cols);
      tmem_relinquish2();
    } else {
      tmem_alloc(&tail->tmem_base, (uint32_t)kp.tmem_cols);
      tmem_relinquish();
    }
  }
  for (int i = threadIdx.x; i < kp.cout_pad; i += blockDim.x) tail->bias[i] = kp.bias[i];
  tc_fence_before();
  __syncthreads();
  if (pair) cluster_sync_all();  // the peer's barriers must be initialised before anything arrives on them
  tc_fence_after();
  const uint32_t tmem_base = tail->tmem_base;
  // PDL: the prologue above touched constant data only; from here on activations are read and written.  The weight
  // producer (warp 6) reads constants only and starts fetching while the previous kernel is still running.
  griddep_launch_dependents();
  if (warp != 6) griddep_wait();
  if (gdbg) gslot[1] = (long long)globaltimer_ns();

  if (warp == 0) {
    // ===================== halo producer: one TMA box per (tile, channel block) =====================
    if (lane == 0) {
      int st = 0;
      uint32_t ph = 0;
      int seq = -1;
      for (int tile = cta0; tile < kp.total_tiles; tile += cstride) {
        const HaloTile t = halo_decode(kp, tile, crank);
        ++seq;
        const bool dbg = kp.dbg != nullptr && blockIdx.x == 0 && seq < 64;
        if (dbg) kp.dbg[(0 * 64 + seq) * 4 + 0] = clock64();
        for (int cb = 0; cb < kp.kblocks; ++cb) {
          mbar_wait(&tail->a_empty[st], ph ^ 1);
          if (dbg && cb == 0) kp.dbg[(0 * 64 + seq) * 4 + 1] = clock64();
          if (pair) {
            if (crank == 0) mbar_arrive_expect_tx(&tail->a_full[st], 2u * kp.halo_bytes);  // both CTAs' halos
            tma_load_5d_2sm(a_base + (size_t)st * kp.a_bytes, &tmap_a, &tail->a_full[st], kp.c_in_off + cb * kp.KB,
                            t.tw * 8 * S + kp.hs_x0, 0, t.th * 16 + kp.hs_y0, t.n);
          } else {
            mbar_arrive_expect_tx(&tail->a_full[st], kp.halo_bytes);
            tma_load_5d(a_base + (size_t)st * kp.a_bytes, &tmap_a, &tail->a_full[st], kp.c_in_off + cb * kp.KB,
                        t.tw * 8 * S + kp.hs_x0, 0, t.th * 16 + kp.hs_y0, t.n);
          }
          if (++st == kp.a_stages) {
            st = 0;
            ph ^= 1;
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 6) {
    // ===================== weight producer: one TMA box per (channel block, tap group) =====================
    // Resident mode (kp.b_resident: the whole filter bank fits next to the halo ring): every box is fetched ONCE per
    // CTA and reused by all its tiles -- without it a small-channel layer re-reads its weights from L2 for every
    // tile, as many bytes as the activations themselves.
    if (lane == 0) {
      int st = 0;
      uint32_t ph = 0;
      for (int tile = cta0; tile < kp.total_tiles; tile += cstride) {
        for (int cb = 0; cb < kp.kblocks; ++cb) {
          for (int tg = 0; tg < tap_groups; ++tg) {
            if (!kp.b_resident) mbar_wait(&tail->b_empty[st], ph ^ 1);
            if (pair) {  // each CTA fetches its half of the output channels
              if (crank == 0) mbar_arrive_expect_tx(&tail->b_full[st], 2u * kp.b_tx_bytes);
              tma_load_3d_2sm(b_base + (size_t)st * kp.b_bytes, &tmap_w, &tail->b_full[st], cb * kp.KB,
                              (int)crank * (kp.BN / 2), tg * G);
            } else {
              mbar_arrive_expect_tx(&tail->b_full[st], kp.b_tx_bytes);
              tma_load_3d(b_base + (size_t)st * kp.b_bytes, &tmap_w, &tail->b_full[st], cb * kp.KB, 0, tg * G);
            }
            if (++st == kp.b_stages) {
              st = 0;
              ph ^= 1;
            }
          }
        }
        if (kp.b_resident) break;
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== UMMA issuer (pair mode: the even CTA only) =====================
    // All 32 lanes run the loops on warp-uniform values; only the elected lane's tcgen05 instructions take effect.
    if (crank == 0) {
      const uint32_t lead = elect_one();
      const uint32_t tm_base = __shfl_sync(0xffffffffu, tmem_base, 0);
      int ast = 0, bst = 0, acc = 0;
      uint32_t aph = 0, bph = 0, acc_ph = 0;
      const uint32_t sbo = (uint32_t)kp.hs_sbo_rows * a_row_bytes;
      const uint32_t tap_b_units = ((uint32_t)(pair ? kp.BN / 2 : kp.BN) * row_bytes) >> 4;  // 16-byte units
      const uint64_t sub_units = (uint64_t)((8u * a_row_bytes) >> 4);                          // next sub-tile: +8 pixels
      const uint32_t acc_cols = (uint32_t)kp.acc_cols;
      const uint32_t idesc = kp.idesc;
      int seq = -1;
      for (int tile = cta0; tile < kp.total_tiles; tile += cstride) {
        ++seq;
        const bool dbg = kp.dbg != nullptr && blockIdx.x == 0 && seq < 64;
        if (dbg && lane == 0) kp.dbg[(1 * 64 + seq) * 4 + 0] = clock64();
        mbar_wait(&tail->tmem_empty[acc], acc_ph ^ 1);
        tc_fence_after();
        if (dbg && lane == 0) kp.dbg[(1 * 64 + seq) * 4 + 1] = clock64();
        const uint32_t d0 = tm_base + (uint32_t)(acc * S * kp.acc_cols);
        long long bwait = 0;
        for (int cb = 0; cb < kp.kblocks; ++cb) {
          const long long ta = dbg ? clock64() : 0;
          mbar_wait(&tail->a_full[ast], aph);
          tc_fence_after();
          if (dbg) bwait += clock64() - ta;
          // Descriptor arithmetic is hoisted: per (channel block, weight stage) one base descriptor each; taps,
          // sub-tiles and k-steps only add precomputed 16-byte-unit offsets to the low word.
          const uint64_t a_desc0 = umma_desc_sbo(smem_u32(a_base + (size_t)ast * kp.a_bytes), a_row_bytes, sbo);
          for (int tg = 0; tg < tap_groups; ++tg) {
            const long long tb = dbg ? clock64() : 0;
            mbar_wait(&tail->b_full[bst], kp.b_resident ? 0u : bph);  // resident: filled once, phase 0 stays complete
            tc_fence_after();
            if (dbg) bwait += clock64() - tb;
            const uint64_t b_desc0 = umma_desc_kmajor(smem_u32(b_base + (size_t)bst * kp.b_bytes), row_bytes);
            for (int ti = 0; ti < G; ++ti) {
              const int tap = tg * G + ti;
              const uint64_t bd = b_desc0 + (uint64_t)((uint32_t)ti * tap_b_units);
              const uint64_t ad = a_desc0 + (uint64_t)(uint32_t)kp.hs_tap_desc[tap];
              const uint32_t first = (uint32_t)((cb | tap) != 0);
#pragma unroll
              for (int j = 0; j < kS; ++j) {
#pragma unroll
                for (int k = 0; k < kSteps; ++k) {
                  const uint32_t accf = k == 0 ? first : 1u;
                  if (kPair)
                    umma_f16_2sm_p(d0 + (uint32_t)j * acc_cols, ad + (uint64_t)j * sub_units + (uint64_t)(2 * k),
                                   bd + (uint64_t)(2 * k), idesc, accf, lead);
                  else
                    umma_f16_p(d0 + (uint32_t)j * acc_cols, ad + (uint64_t)j * sub_units + (uint64_t)(2 * k),
                               bd + (uint64_t)(2 * k), idesc, accf, lead);
                }
              }
            }
            if (!kp.b_resident) {
              if (pair) umma_commit_2sm_p(&tail->b_empty[bst], lead); else umma_commit_p(&tail->b_empty[bst], lead);
            }
            if (++bst == kp.b_stages) {
              bst = 0;
              bph ^= 1;
            }
          }
          if (pair) umma_commit_2sm_p(&tail->a_empty[ast], lead); else umma_commit_p(&tail->a_empty[ast], lead);
          if (++ast == kp.a_stages) {
            ast = 0;
            aph ^= 1;
          }
        }
        if (pair) umma_commit_2sm_p(&tail->tmem_full[acc], lead); else umma_commit_p(&tail->tmem_full[acc], lead);
        if (dbg && lane == 0) {
          kp.dbg[(1 * 64 + seq) * 4 + 2] = bwait;  // cycles this tile spent waiting for operands (a_full + b_full)
          kp.dbg[(1 * 64 + seq) * 4 + 3] = clock64();
        }
        if (++acc == kp.acc_stages) {
          acc = 0;
          acc_ph ^= 1;
        }
      }
    }
    __syncwarp();
  } else {
    // ===== epilogue: up to three groups of 4 warps (2-5, 7-10, 11-14), tiles round-robin; S sub-tiles of 16 rows x 8 columns each
    const int egroup = warp >= 7 ? 1 + ((warp - 7) >> 2) : 0;
    const int quarter = warp & 3;
    const int m = quarter * 32 + lane;
    const int row = m >> 3, col = m & 7;
    const bool fast = kEpi != PB_EPI_GENERIC || epilogue_fast_ok(kp);  // the host picks a plain class only when it holds
    int seq = egroup, acc = egroup;  // sequence number / accumulator stage / phase by counters (egroups <= acc_stages)
    uint32_t acc_ph = 0;
    for (int tile = cta0 + egroup * cstride; egroup < kp.egroups && tile < kp.total_tiles;
         tile += kp.egroups * cstride, seq += kp.egroups) {
      const HaloTile t = halo_decode(kp, tile, crank);
      const bool dbg = kp.dbg != nullptr && blockIdx.x == 0 && seq < 64 && (threadIdx.x == 64 || (threadIdx.x >= 224 && ((threadIdx.x - 224) & 127) == 0));
      if (dbg) kp.dbg[(2 * 64 + seq) * 4 + 0] = clock64();
      mbar_wait(&tail->tmem_full[acc], acc_ph);
      tc_fence_after();
      if (dbg) kp.dbg[(2 * 64 + seq) * 4 + 1] = clock64();
      if (fast) {
        const int oh = t.th * 16 + row, ow0 = t.tw * 8 * S + col;
        uint32_t vm = 0;
#pragma unroll
        for (int j = 0; j < S; ++j) vm |= (uint32_t)((ow0 + 8 * j < kp.Wo) && (oh < kp.Ho)) << j;
        const size_t pix0 = ((size_t)t.n * kp.Ho + oh) * kp.Wo + ow0;
        EpiOut eo;
        eo.mode = kp.out_mode;
        const size_t esz = eo.mode == PB_OUT_F32_NHWC ? 4 : 2;
        const size_t pxb = (size_t)kp.out_C * esz;  // bytes per output pixel
        size_t opix = pix0, sub_out = 8 * pxb;
        eo.dx = eo.dy = 0;
        if (eo.mode == PB_OUT_F16_NHWC_UP2) {
          opix = ((size_t)t.n * (2 * kp.Ho) + 2 * oh) * (2 * kp.Wo) + 2 * ow0;
          eo.dx = pxb;
          eo.dy = (size_t)(2 * kp.Wo) * pxb;
          sub_out = 16 * pxb;
        }
        eo.mode2 = kp.out2_mode;
        eo.dx2 = eo.dy2 = 0;
        eo.pool_writer = ((row | col) & 1) == 0;
        char* obase2 = nullptr;
        size_t sub_out2 = 0;
        if (eo.mode2 != PB_OUT2_NONE) {
          const size_t pxb2 = (size_t)kp.out2_C * 2;
          size_t pix2;
          if (eo.mode2 == PB_OUT2_UP2) {
            pix2 = ((size_t)t.n * (2 * kp.Ho) + 2 * oh) * (2 * kp.Wo) + 2 * ow0;
            eo.dx2 = pxb2;
            eo.dy2 = (size_t)(2 * kp.Wo) * pxb2;
            sub_out2 = 16 * pxb2;
          } else {  // POOL2 (Ho, Wo even): the pooled pixel of the window whose top-left corner this lane holds
            pix2 = ((size_t)t.n * (kp.Ho >> 1) + (oh >> 1)) * (kp.Wo >> 1) + (ow0 >> 1);
            sub_out2 = 4 * pxb2;
          }
          obase2 = reinterpret_cast<char*>(kp.out2) + pix2 * pxb2 + (size_t)kp.out2_coff * 2;
        }
        const uint32_t t0 = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * S * kp.acc_cols);
        char* obase = reinterpret_cast<char*>(kp.out) + opix * pxb + (size_t)kp.out_coff * esz;
          epilogue_fast<kEpi>(kp, eo, t0, S, (uint32_t)kp.acc_cols, (kp.cout_store + 15) >> 4, kp.cout_store, tail->bias,
                        obase, kp.res + pix0 * kp.res_C + kp.res_coff, sub_out, (size_t)8 * kp.res_C, vm, obase2,
                        sub_out2);
      } else if constexpr (kEpi == PB_EPI_GENERIC)
      for (int j = 0; j < S; ++j) {
        EpiPix px;
        px.n = t.n;
        px.oh = t.th * 16 + row;
        px.ow = t.tw * 8 * S + 8 * j + col;
        px.valid = (px.ow < kp.Wo) && (px.oh < kp.Ho);
        px.pix = ((size_t)px.n * kp.Ho + px.oh) * kp.Wo + px.ow;
        const uint32_t t_addr =
            tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)((acc * S + j) * kp.acc_cols);
        float hacc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int c = 0; c < kp.BN; c += 32) {
          uint32_t r0[16], r1[16];
          const bool second = (c + 16 < kp.BN);
          tmem_ld16(t_addr + (uint32_t)c, r0);
          if (second) tmem_ld16(t_addr + (uint32_t)(c + 16), r1);
          tmem_ld_wait();
          if (px.valid && c < kp.cout_store) {
            float v[16];
            bias_act16(r0, tail->bias + c, kp.act, v,
                       (kp.res && kp.res_first) ? kp.res + px.pix * kp.res_C + kp.res_coff + c : nullptr);
            epilogue_store16(kp, px, c, c, v, hacc);
          }
          if (second && px.valid && c + 16 < kp.cout_store) {
            float v[16];
            bias_act16(r1, tail->bias + c + 16, kp.act, v,
                       (kp.res && kp.res_first) ? kp.res + px.pix * kp.res_C + kp.res_coff + c + 16 : nullptr);
            epilogue_store16(kp, px, c + 16, c + 16, v, hacc);
          }
        }
        if (kp.head_n > 0 && px.valid) {
          const size_t plane = (size_t)kp.Ho * kp.Wo;
          float* ho = kp.head_out + (size_t)px.n * kp.head_n * plane + (size_t)px.oh * kp.Wo + px.ow;
#pragma unroll
          for (int q = 0; q < 8; ++q)
            if (q < kp.head_n) ho[(size_t)q * plane] = __fdividef(1.f, 1.f + __expf(-(hacc[q] + __ldg(kp.head_b + q))));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (pair) mbar_arrive_cluster(&tail->tmem_empty[acc], 0);  // the leader's MMA thread waits for both CTAs
        else mbar_arrive(&tail->tmem_empty[acc]);
      }
      if (dbg) kp.dbg[(2 * 64 + seq) * 4 + 2] = clock64();
      acc += kp.egroups;
      if (acc >= kp.acc_stages) {
        acc -= kp.acc_stages;
        acc_ph ^= 1u;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (gdbg) gslot[2] = (long long)globaltimer_ns();
  if (pair) cluster_sync_all();
  if (warp == 2) {
    tc_fence_after();
    if (pair) tmem_dealloc2(tmem_base, (uint32_t)kp.tmem_cols);
    else tmem_dealloc(tmem_base, (uint32_t)kp.tmem_cols);
  }
}

// ------------------------------------------------------------------------------------------------------------
// host: geometry + tensor maps for the halo variant. Returns 0 and sets plan->variant = 1 when applicable,
// returns -1 (no error) when the layer should use the per-tap kernel.
// ------------------------------------------------------------------------------------------------------------
constexpr size_t kHaloBudget = 196 * 1024;  // halo + weight rings of a CTA that has the SM to itself
constexpr size_t kHalfSm = 108 * 1024;      // the whole footprint of one of two CTAs per SM

// TMA swizzle of K-major rows of 128 / 64 / 32 bytes: the swizzle span is the row
static CUtensorMapSwizzle swizzle_for(uint32_t row_bytes) {
  return row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
         : row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                           : CU_TENSOR_MAP_SWIZZLE_32B;
}

int conv_weight_tmap(CUtensorMap* map, EncodeTiledFn encode, const pb_conv_desc* d, int taps, int box_k, int box_n,
                     int box_taps) {
  const cuuint64_t dims[3] = {(cuuint64_t)d->cin, (cuuint64_t)d->cout_pad, (cuuint64_t)taps};
  const cuuint64_t strides[2] = {(cuuint64_t)d->cin * 2, (cuuint64_t)d->cin * d->cout_pad * 2};
  const cuuint32_t box[3] = {(cuuint32_t)box_k, (cuuint32_t)box_n, (cuuint32_t)box_taps};
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(d->weight), dims, strides, box,
                            estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for((uint32_t)box_k * 2u),
                            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PB_CHECK(r == CUDA_SUCCESS, "conv: cuTensorMapEncodeTiled(W) failed with %d (cin %d, cout_pad %d, %d taps)", (int)r,
           d->cin, d->cout_pad, taps);
  return 0;
}

int conv_act_tmap(CUtensorMap* map, EncodeTiledFn encode, const pb_conv_desc* d, int s, int box_c, int box_w,
                  int box_s, int box_h, int box_n) {
  const cuuint64_t C = (cuuint64_t)d->C, W = (cuuint64_t)d->W, H = (cuuint64_t)d->H, S = (cuuint64_t)s;
  const cuuint64_t dims[5] = {S * C, W / S, S, H / S, (cuuint64_t)d->N};
  const cuuint64_t strides[4] = {S * C * 2, W * C * 2, S * W * C * 2, H * W * C * 2};
  const cuuint32_t box[5] = {(cuuint32_t)box_c, (cuuint32_t)box_w, (cuuint32_t)box_s, (cuuint32_t)box_h,
                             (cuuint32_t)box_n};
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, const_cast<void*>(d->in), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for((uint32_t)box_c * 2u),
                            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PB_CHECK(r == CUDA_SUCCESS, "conv: cuTensorMapEncodeTiled(A) failed with %d (N=%d H=%d W=%d C=%d s=%d)", (int)r, d->N,
           d->H, d->W, d->C, s);
  return 0;
}

// Halo ring next to a resident filter bank of res_total bytes (b_stages = kblocks fixed slots): whatever shared memory is
// left goes to halo buffers, 2 .. kHaloMaxA.  A light tile (set_cols = S * acc_cols TMEM columns per accumulator set)
// whose bank and two halo buffers fit in half an SM is sized for half an SM, so two CTAs can share one
// (halo_finish_config).
static int halo_resident_a_stages(const ConvKParams& kp, size_t res_total, int set_cols) {
  const bool small = (size_t)2 * kp.a_bytes + res_total + sizeof(HaloSmemTail) + 1024 <= kHalfSm && set_cols * 2 <= 256;
  const size_t budget = small ? kHalfSm - sizeof(HaloSmemTail) - 1024 : kHaloBudget;
  int as = (int)((budget - res_total) / kp.a_bytes);
  if (as > kHaloMaxA) as = kHaloMaxA;
  if (as > 2 * kp.kblocks + 1) as = 2 * kp.kblocks + 1;
  return as < 2 ? 2 : as;
}

// Tiles, accumulator ring and launch configuration, shared by the halo and stem set-ups once they have set BN, hs_S,
// pair and the rings.  A tile is 16 output rows (32 for a CTA pair: 16 per CTA) x 8S columns of one image, S
// accumulator sets of acc_cols TMEM columns.  Two CTAs per SM when the CTA fits in half an SM's shared memory and 256
// TMEM columns and there are more tiles than SMs (light n-scale YOLO layers), else one CTA per SM with up to three
// epilogue groups.
static void halo_finish_config(ConvPlan* plan) {
  ConvKParams& kp = plan->kp;
  const int S = kp.hs_S;
  kp.acc_cols = (kp.BN + 31) / 32 * 32;
  kp.acc_stages = 512 / (S * kp.acc_cols);
  if (kp.acc_stages > kConvMaxAcc) kp.acc_stages = kConvMaxAcc;
  kp.idesc = kp.pair ? umma_idesc_f16_m256(kp.BN) : umma_idesc_f16(kp.BN, 0);
  kp.tiles_w = (kp.Wo + 8 * S - 1) / (8 * S);
  kp.tiles_h = kp.pair ? (kp.Ho + 31) / 32 : (kp.Ho + 15) / 16;
  kp.tiles_n = kp.N;
  kp.total_tiles = kp.tiles_w * kp.tiles_h * kp.tiles_n;

  const size_t need = (size_t)kp.a_stages * kp.a_bytes + (size_t)kp.b_stages * kp.b_bytes + sizeof(HaloSmemTail) + 1024;
  const int set_cols = S * kp.acc_cols;
  const bool occ2 = !kp.pair && need <= 110 * 1024 && set_cols * 2 <= 256 && kp.total_tiles > num_sms();
  plan->smem_bytes = need;
  if (occ2) {
    if (kp.acc_stages * set_cols > 256) kp.acc_stages = 256 / set_cols;
    kp.tmem_cols = 256;
    kp.egroups = 1;
    plan->threads = 224;
    plan->grid = kp.total_tiles < 2 * num_sms() ? kp.total_tiles : 2 * num_sms();
  } else {
    if (plan->smem_bytes < 120 * 1024) plan->smem_bytes = 120 * 1024;
    kp.tmem_cols = 512;
    kp.egroups = kp.pair ? 2 : conv_pick_egroups(kp.acc_stages);
    plan->threads = conv_threads_for(kp.egroups);
    plan->grid = kp.total_tiles < num_sms() ? kp.total_tiles : num_sms();
    if (kp.pair) {  // total_tiles counts pair tiles: two CTAs each
      const int pairs = kp.total_tiles < num_sms() / 2 ? kp.total_tiles : num_sms() / 2;
      plan->grid = 2 * pairs;
    }
  }
  plan->variant = 1;
}

// Stem (PB_IN_STEM4): 3x3 stride-2 conv over the padded 4-channel input, K = 16 per filter row (12 real), 3 UMMAs per
// sub-tile.  The tile's input region -- 34 rows x (16 S + 2) pixels of 8 bytes, every byte once -- is one dense TMA box,
// and the UMMA descriptor reads the im2col rows out of it: output pixel ow's K = 16 row (pixels 2ow .. 2ow+3) starts 16
// bytes after its neighbour's, so in the un-swizzled K-major layout (16-byte rows at a 16-byte pitch, second half of a
// row LBO = 16 bytes on) the overlapping rows ARE the canonical core matrix; the next output row is two image rows
// further (SBO), filter row r one image row (descriptor offset).
int conv_stem_setup(const pb_conv_desc* d, ConvPlan* plan, EncodeTiledFn encode) {
  PB_CHECK(d->ksize == 3 && d->stride == 2 && d->C == 4 && d->cin == 16 && d->c_in_off == 0,
           "conv(stem): needs ksize 3, stride 2, C = 4, cin = 16");
  PB_CHECK(d->cout_pad <= 128, "conv(stem): cout_pad %d > 128", d->cout_pad);
  ConvKParams& kp = plan->kp;
  const int BN = d->cout_pad;
  const int acc_cols = (BN + 31) / 32 * 32;
  int S = 4;
  while (S > 1 && (S * acc_cols * 2 > 512)) S >>= 1;
  const uint32_t pairs = (uint32_t)(8 * S) + 1;  // pixel pairs (16 bytes) per image row of the region
  const uint32_t pitch = pairs * 16u;
  kp.KB = 16;
  kp.kblocks = 1;
  kp.taps = 3;
  kp.hs_S = S;
  kp.hs_P = 8 * S;
  kp.hs_G = 3;
  kp.hs_ntaps = 3;
  kp.hs_sbo_rows = (int)(2u * pitch / 16u);  // x hs_a_row_bytes = 2 image rows
  kp.hs_x0 = 0;
  kp.hs_y0 = 0;
  for (int r = 0; r < 3; ++r) {
    kp.hs_tap_off[r] = r * 8 * S;
    kp.hs_tap_desc[r] = (int)(((uint32_t)r * pitch) >> 4);
  }
  kp.BN = BN;
  kp.n_ntiles = 1;
  kp.halo_bytes = 17u * 2u * pitch;  // 17 row pairs (2 * 16 + 1 rows are read, the 34th is never addressed)
  kp.hs_a_row_bytes = 16u;
  kp.a_bytes = (kp.halo_bytes + 1023u) & ~1023u;
  kp.b_tx_bytes = 3u * (uint32_t)BN * 32u;
  kp.b_bytes = (kp.b_tx_bytes + 1023u) & ~1023u;
  kp.a_stages = 4;
  kp.b_stages = 1;  // the three filter rows are one small box: resident
  kp.b_resident = 1;
  halo_finish_config(plan);
  {
    // dense view (pixel pair, image-row parity, image-row pair) of the padded (N, H+2, W+2, 4) tensor: element
    // (k, p, q, y, n) = base + n*Hp*Wp*8 + (2*y + q)*Wp*8 + p*16 + 2*k; the producer's coordinates (0, ow0, 0, oh0, n)
    // address pixel pair ow0 = pixel 2*ow0 and image row 2*oh0 of the padded tensor, i.e. the tile's top-left tap
    const cuuint64_t Wp = (cuuint64_t)d->W + 2, Hp = (cuuint64_t)d->H + 2;
    const cuuint64_t dims[5] = {8, Wp / 2, 2, Hp / 2, (cuuint64_t)d->N};
    const cuuint64_t strides[4] = {16, Wp * 8, 2 * Wp * 8, Hp * Wp * 8};
    const cuuint32_t box[5] = {8, pairs, 2, 17, 1};
    const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    const CUresult r = encode(&plan->tmap_a, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, const_cast<void*>(d->in), dims,
                              strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    PB_CHECK(r == CUDA_SUCCESS, "conv(stem): cuTensorMapEncodeTiled(A) failed with %d", (int)r);
  }
  return conv_weight_tmap(&plan->tmap_w, encode, d, 3, 16, BN, 3);
}

int conv_halo_setup(const pb_conv_desc* d, ConvPlan* plan, EncodeTiledFn encode) {
  if (d->ksize != 3 || d->stride != 1 || d->cout_pad > 256) return -1;
  ConvKParams& kp = plan->kp;  // common fields (epilogue, KB, kblocks, ...) already filled by the caller
  const int BN = d->cout_pad;
  const uint32_t row_bytes = (uint32_t)kp.KB * 2u;
  const int acc_cols = (BN + 31) / 32 * 32;
  // Choose S (sub-tiles per CTA tile: fewer halo + weight bytes per pixel) first, then G (taps per weight box:
  // fewer TMA operations) as large as shared memory allows.
  const uint32_t tap_bytes = (uint32_t)BN * row_bytes;
  // Resident filter bank: all nine taps of every channel block (one box per block) stay in shared memory for the
  // whole kernel when they fit next to two halo buffers; otherwise weight boxes are streamed through a ring.
  const uint32_t res_box = (9u * tap_bytes + 1023u) & ~1023u;
  const size_t res_total = (size_t)kp.kblocks * res_box;
  bool resident = kp.kblocks <= kHaloMaxB && res_total <= 120 * 1024;
  int bestS = 0, best_cols = 0, G = 1;
  for (int pass = resident ? 0 : 1; pass < 2 && bestS == 0; ++pass) {
    resident = resident && pass == 0;
    for (int S = 4; S >= 1; S >>= 1) {
      if (S * acc_cols * 2 > 512) continue;  // keep >= 2 accumulator sets in TMEM
      const uint32_t halo = 18u * (uint32_t)(8 * S + 2) * row_bytes;
      const uint32_t a_alloc = (halo + 1023u) & ~1023u;
      int g_fit = 0;
      if (resident) {
        if ((size_t)2 * a_alloc + res_total <= kHaloBudget) g_fit = 9;
      } else {
        for (int g = 9; g >= 1; g = (g == 9 ? 3 : (g == 3 ? 1 : 0))) {
          const uint32_t ba = ((uint32_t)g * tap_bytes + 1023u) & ~1023u;
          const int min_b = g == 9 ? 2 : (g == 3 ? 3 : 4);
          if ((size_t)2 * a_alloc + (size_t)min_b * ba <= kHaloBudget) {
            g_fit = g;
            break;
          }
        }
      }
      if (!g_fit) continue;
      const int cols = (d->W + 8 * S - 1) / (8 * S) * 8 * S;  // padded width actually computed
      // resident: prefer the largest S that fits (less halo overlap); streaming: the least padding
      if (bestS == 0 || (!resident && cols < best_cols)) {
        bestS = S;
        best_cols = cols;
        G = g_fit;
      }
    }
  }
  const uint32_t b_alloc = ((uint32_t)G * tap_bytes + 1023u) & ~1023u;
  if (bestS == 0) return -1;
  const int S = bestS, P = 8 * S + 2;
  // CTA-pair mode (cta_group::2): one M=256 UMMA per instruction slot, each CTA of the pair fetching half of the
  // weights.  Measured on TrackNet at batch 32 (profiles/r01_layers.txt): the deep-K narrow layers gain (192->64:
  // 935 -> 757 us = 1.38 PFLOP/s, above the ~1.27 PFLOP/s a single CTA can issue at N = 64; 384->128: 768 -> 676 us;
  // 128->128: 269 -> 231 us), shallow-K layers (cin <= 64) and the 2x2-replicating stores lose a few percent.
  // Rule: cin >= 128, plain fp16 store, enough tiles to fill the machine with pairs (unless overridden).
  {
    const int pm = conv_override("PADEL_B200_CONV_PAIR");
    const bool can = BN % 32 == 0 && BN >= 32 && kp.Ho >= 32;
    const long pair_tiles = (long)((d->W + 8 * S - 1) / (8 * S)) * ((kp.Ho + 31) / 32) * kp.N;
    const bool want = d->cin >= 128 && d->out_mode == PB_OUT_F16_NHWC && pair_tiles >= 2L * (num_sms() / 2);
    kp.pair = (can && (pm == 1 || (pm == 2 && want))) ? 1 : 0;
    if (kp.pair && resident) {  // forced pair mode: stream the weights (each CTA holds half of them)
      resident = false;
      if (G == 9 && (size_t)2 * (((18u * (uint32_t)(8 * bestS + 2) * row_bytes) + 1023u) & ~1023u) + (size_t)2 * b_alloc > kHaloBudget)
        return -1;
    }
  }
  kp.b_resident = resident ? 1 : 0;
  kp.hs_S = S;
  kp.hs_P = P;
  kp.hs_G = G;
  kp.hs_ntaps = 9;
  kp.hs_sbo_rows = P;
  kp.hs_x0 = -1;
  kp.hs_y0 = -1;
  for (int r = 0; r < 3; ++r)
    for (int q = 0; q < 3; ++q) {
      kp.hs_tap_off[r * 3 + q] = r * P + q;
      kp.hs_tap_desc[r * 3 + q] = (int)(((uint32_t)(r * P + q) * row_bytes) >> 4);
    }
  kp.BN = BN;
  kp.n_ntiles = 1;
  kp.halo_bytes = 18u * (uint32_t)P * row_bytes;
  kp.hs_a_row_bytes = row_bytes;
  kp.a_bytes = (kp.halo_bytes + 1023u) & ~1023u;
  kp.b_tx_bytes = (uint32_t)G * tap_bytes / (kp.pair ? 2u : 1u);  // per CTA
  kp.b_bytes = b_alloc;
  kp.a_stages = 2;
  if (resident) {
    kp.b_stages = kp.kblocks;
    kp.a_stages = halo_resident_a_stages(kp, res_total, S * acc_cols);
  } else {
    // light layers: size the rings for half an SM so that two CTAs can be co-resident (see halo_finish_config)
    const int min_b_small = G == 9 ? 2 : (G == 3 ? 3 : 4);
    const bool small =
        (size_t)2 * kp.a_bytes + (size_t)min_b_small * b_alloc + sizeof(HaloSmemTail) + 1024 <= kHalfSm &&
        S * acc_cols * 2 <= 256;
    const size_t budget2 = small ? kHalfSm - sizeof(HaloSmemTail) - 1024 : kHaloBudget;
    size_t rest = budget2 - (size_t)2 * kp.a_bytes;
    if (kp.kblocks > 2 && rest > (size_t)kp.a_bytes + 4 * (size_t)b_alloc) {  // a third halo buffer when K is deep
      kp.a_stages = 3;
      rest -= kp.a_bytes;
    }
    int bs = (int)(rest / b_alloc);
    if (bs > kHaloMaxB) bs = kHaloMaxB;
    if (bs > 9 * kp.kblocks / G * 2) bs = 9 * kp.kblocks / G * 2;
    if (bs < 2) bs = 2;
    kp.b_stages = bs;
  }
  halo_finish_config(plan);
  if (conv_act_tmap(&plan->tmap_a, encode, d, 1, kp.KB, P, 1, 18, 1)) return 1;
  return conv_weight_tmap(&plan->tmap_w, encode, d, 9, kp.KB, kp.pair ? BN / 2 : BN, G);
}

// 1x1 / stride-1 layers through the same kernel (one tap, no halo): a CTA tile is 16 rows x 8S columns (up to 512
// pixels, S accumulator sets) instead of the per-tap kernel's 128, and the whole filter bank (cin x cout, one box per
// channel block) is fetched ONCE per CTA and stays in shared memory -- the per-tap kernel re-reads it from L2 for every
// 128-pixel tile, as many bytes as the activations when cin ~ cout, and pays its fixed per-tile costs four times as
// often.  Measured on the pose program (batch 32, profiles/r02_layers_final.txt): cin 32 -> 32 @320^2 152 -> 93 us; every
// layer with cin >= 64 is 0-15 % SLOWER than on the per-tap kernel (whose flattened 128-pixel tiles waste nothing at the
// image edges and whose K loop is deeper).  Rule therefore: cin <= 32.
int conv_halo_1x1_setup(const pb_conv_desc* d, ConvPlan* plan, EncodeTiledFn encode) {
  if (d->ksize != 1 || d->stride != 1 || d->cout_pad > 256 || d->head_n != 0 || d->cin > 32) return -1;
  // fp32 outputs (YOLO head maps, the TrackNet predictor) keep the per-tap kernel and its fp32 epilogue class
  if (d->out_mode != PB_OUT_F16_NHWC && d->out_mode != PB_OUT_F16_NHWC_UP2) return -1;
  ConvKParams& kp = plan->kp;  // common fields already filled by the caller
  const int BN = d->cout_pad;
  const uint32_t row_bytes = (uint32_t)kp.KB * 2u;
  const int acc_cols = (BN + 31) / 32 * 32;
  const uint32_t tap_bytes = (uint32_t)BN * row_bytes;
  const uint32_t res_box = (tap_bytes + 1023u) & ~1023u;
  const size_t res_total = (size_t)kp.kblocks * res_box;
  if (kp.kblocks > kHaloMaxB || res_total > 120 * 1024) return -1;
  int S = 0;
  for (int s = 4; s >= 1; s >>= 1) {
    if (s * acc_cols * 2 > 512) continue;  // keep >= 2 accumulator sets in TMEM
    const uint32_t a_alloc = (16u * (uint32_t)(8 * s) * row_bytes + 1023u) & ~1023u;
    if ((size_t)2 * a_alloc + res_total > kHaloBudget) continue;
    if (s > 1 && d->W <= 8 * (s / 2)) continue;  // a narrower tile already covers the row
    S = s;
    break;
  }
  if (S == 0) return -1;
  const int P = 8 * S;
  kp.pair = 0;
  kp.b_resident = 1;
  kp.hs_S = S;
  kp.hs_P = P;
  kp.hs_G = 1;
  kp.hs_ntaps = 1;
  kp.hs_sbo_rows = P;
  kp.hs_x0 = 0;
  kp.hs_y0 = 0;
  kp.hs_tap_off[0] = 0;
  kp.hs_tap_desc[0] = 0;
  kp.BN = BN;
  kp.n_ntiles = 1;
  kp.halo_bytes = 16u * (uint32_t)P * row_bytes;
  kp.hs_a_row_bytes = row_bytes;
  kp.a_bytes = (kp.halo_bytes + 1023u) & ~1023u;
  kp.b_tx_bytes = tap_bytes;
  kp.b_bytes = res_box;
  kp.b_stages = kp.kblocks;
  kp.a_stages = halo_resident_a_stages(kp, res_total, S * acc_cols);
  halo_finish_config(plan);
  if (conv_act_tmap(&plan->tmap_a, encode, d, 1, kp.KB, P, 1, 16, 1)) return 1;
  return conv_weight_tmap(&plan->tmap_w, encode, d, 1, kp.KB, BN, 1);
}

// 3x3 / stride-2 conv over a whole C = 16 / 32 channel tensor.  The input is read through the pixel-pair view
// (2C, W/2, 2, H/2, N) -- element (k, w2, ph, h2, n) = channel k % C of pixel (2*h2 + ph, 2*w2 + k / C) -- so one TMA
// box (2C, 8S+1, 2, 17, 1) holds everything a 16 x 8S output tile needs, as rows of one PIXEL PAIR (4C bytes):
//   smem row = ((h2i * 2 + ph) * P + w2i),  P = 8S + 1,  box origin (w2, h2) = (ow0 - 1, oh0 - 1).
// Tap (r, s) of output (ohi, owi) reads input (2*oh + r - 1, 2*ow + s - 1):
//   r = 0 -> (h2i, ph) = (ohi, 1)      r = 1 -> (ohi + 1, 0)      r = 2 -> (ohi + 1, 1)
//   s = 0 -> (w2i, half) = (owi, 1)    s = 1 -> (owi + 1, 0)      s = 2 -> (owi + 1, 1)
// i.e. again only a descriptor start offset (row offset * 4C + half * 2C bytes) with SBO = 2P rows, and K = C per tap
// (the 32-byte k-step advance inside the swizzle row is the usual one).  Versus nine per-tap boxes of 2C-byte rows
// this issues one TMA per tile with rows twice as long (TMA delivery of 32-byte rows is what bounds the per-tap path).
int conv_halo_s2_setup(const pb_conv_desc* d, ConvPlan* plan, EncodeTiledFn encode) {
  if (d->ksize != 3 || d->stride != 2 || d->cout_pad > 256 || d->c_in_off != 0 || d->C != d->cin ||
      (d->cin != 16 && d->cin != 32))
    return -1;
  ConvKParams& kp = plan->kp;  // common fields already filled by the caller (KB = cin, kblocks = 1)
  const int BN = d->cout_pad;
  const uint32_t row_bytes = (uint32_t)d->cin * 2u;  // weight rows
  const uint32_t a_row = 2u * row_bytes;             // pixel-pair rows
  const int acc_cols = (BN + 31) / 32 * 32;
  const uint32_t tap_bytes = (uint32_t)BN * row_bytes;
  const uint32_t b_alloc = (9u * tap_bytes + 1023u) & ~1023u;  // all nine taps in one weight box
  int S = 0;
  for (int s = 4; s >= 1; s >>= 1) {
    if (s * acc_cols * 2 > 512) continue;
    const uint32_t halo = 34u * (uint32_t)(8 * s + 1) * a_row;
    if ((size_t)2 * ((halo + 1023u) & ~1023u) + (size_t)2 * b_alloc <= kHaloBudget) {
      S = s;
      break;
    }
  }
  if (S == 0) return -1;
  const int P = 8 * S + 1;
  kp.pair = 0;
  kp.KB = d->cin;
  kp.kblocks = 1;
  kp.hs_S = S;
  kp.hs_P = P;
  kp.hs_G = 9;
  kp.hs_ntaps = 9;
  kp.hs_sbo_rows = 2 * P;
  kp.hs_x0 = -1;
  kp.hs_y0 = -1;
  kp.hs_a_row_bytes = a_row;
  for (int r = 0; r < 3; ++r)
    for (int q = 0; q < 3; ++q) {
      const int row = ((r == 0 ? 0 : 1) * 2 + (r == 1 ? 0 : 1)) * P + (q == 0 ? 0 : 1);
      const int half = q == 1 ? 0 : 1;
      kp.hs_tap_off[r * 3 + q] = row;
      kp.hs_tap_desc[r * 3 + q] = (int)(((uint32_t)row * a_row + (uint32_t)half * row_bytes) >> 4);
    }
  kp.BN = BN;
  kp.n_ntiles = 1;
  kp.halo_bytes = 34u * (uint32_t)P * a_row;
  kp.a_bytes = (kp.halo_bytes + 1023u) & ~1023u;
  kp.b_tx_bytes = 9u * tap_bytes;
  kp.b_bytes = b_alloc;
  kp.a_stages = 2;
  kp.b_stages = 1;  // all nine taps are one box: resident
  kp.b_resident = 1;
  halo_finish_config(plan);
  if (conv_act_tmap(&plan->tmap_a, encode, d, 2, 2 * d->cin, P, 2, 17, 1)) return 1;
  return conv_weight_tmap(&plan->tmap_w, encode, d, 9, d->cin, BN, 9);
}

typedef void (*HaloKernelFn)(CUtensorMap, CUtensorMap, ConvKParams);

template <bool kPair, int kEpi>
static HaloKernelFn halo_kernel_for(int S, int steps) {
#define PB_HALO_CASE(s_, k_) \
  if (S == s_ && steps == k_) return conv_halo_kernel<kPair, s_, k_, kEpi>;
  PB_HALO_CASE(1, 1) PB_HALO_CASE(1, 2) PB_HALO_CASE(1, 4)
  PB_HALO_CASE(2, 1) PB_HALO_CASE(2, 2) PB_HALO_CASE(2, 4)
  PB_HALO_CASE(4, 1) PB_HALO_CASE(4, 2) PB_HALO_CASE(4, 4)
#undef PB_HALO_CASE
  return nullptr;
}

// CTA-pair layers are deep (cin >= 128) and tensor-bound: the run-time epilogue only
static HaloKernelFn halo_kernel_pick(const ConvPlan* plan) {
  const ConvKParams& kp = plan->kp;
  const int S = kp.hs_S, steps = kp.KB / 16;
  if (kp.pair) return halo_kernel_for<true, PB_EPI_GENERIC>(S, steps);
  if (plan->epi == PB_EPI_SILU) return halo_kernel_for<false, PB_EPI_SILU>(S, steps);
  if (plan->epi == PB_EPI_RELU) return halo_kernel_for<false, PB_EPI_RELU>(S, steps);
  if (plan->epi == PB_EPI_SILU_RES) return halo_kernel_for<false, PB_EPI_SILU_RES>(S, steps);
  return halo_kernel_for<false, PB_EPI_GENERIC>(S, steps);
}

int conv_halo_launch(const ConvPlan* plan, cudaStream_t stream) {
  const ConvKParams& kp = plan->kp;
  HaloKernelFn fn = halo_kernel_pick(plan);
  PB_CHECK(fn != nullptr, "conv(halo): no kernel instantiation for S=%d, k-steps=%d", kp.hs_S, kp.KB / 16);
  PB_CUDA((cudaError_t)ensure_dynamic_smem(reinterpret_cast<const void*>(fn), 227 * 1024));
  cudaError_t le = launch_pdl(fn, dim3(plan->grid), dim3(plan->threads), plan->smem_bytes, stream, kp.pair ? 2 : 1,
                              plan->tmap_a, plan->tmap_w, plan->kp);
  PB_CHECK(le == cudaSuccess,
           "conv(halo): launch failed: %s (pair %d, grid %d, threads %d, smem %zu, tiles %d, S %d, BN %d, KB %d)",
           cudaGetErrorString(le), kp.pair, plan->grid, plan->threads, plan->smem_bytes, kp.total_tiles, kp.hs_S, kp.BN,
           kp.KB);
  count_launch();
  return 0;
}

}  // namespace pb
