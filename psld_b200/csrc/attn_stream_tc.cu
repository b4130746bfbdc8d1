// Key-streaming tcgen05 attention for the NCSN++ AttnBlockpp (reference layerspp.py:82-91) over
// HW = 512, 640, ... (any multiple of 128 from 512: 32x32 maps and larger) tokens of C = 64, 128, 192
// or 256 channels.  attn_tc.cu keeps all keys of a query tile in one TMEM accumulator, which caps it at
// 256 tokens; here the keys stream through in tiles of KT with an online softmax (flash attention):
//
// One CTA = one sample x 128 queries; warp 0 = TMA producer, warp 1 = MMA issuer, warps 2..5 = 128
// softmax / epilogue threads (one query row each).  For key tile j:
//   S_j[128 x KT] = Q K_j^T    A = Q (resident in shared memory for the whole key loop), B = K tiles
//                              (64 channels x KT keys) from the ring; S is double-buffered in TMEM, so
//                              the softmax of tile j overlaps the MMA of tile j+1
//   P_j = exp2(S_j*c - m)      written by the row-owner threads over the P region in the 128B-swizzled
//                              K-major UMMA layout (bf16; kX3: hi | lo split).  m = running row max in
//                              log2 units, l = running row sum (of the rounded P in the bf16 tier)
//   lazy rescale               m moves only when the tile max exceeds it by more than kRescale (P <=
//                              2^kRescale otherwise); then O and l are multiplied by exp2(m_old - m_new).
//                              O and l always share the same m, so O / l is exact either way
//   O[128 x C] += P_j V_j      per 64-channel group: B = V tile (KT keys x 64 channels) as an MN-major
//                              operand, accumulator in TMEM
// After the last tile O / l is written over Q (bf16, kX3: split).  kProj: Y = Onorm W3^T (the NIN_3
// projection, W3 tiles through the ring) accumulates over the O columns and tc_epilogue_tile finishes
// the tile (bias, residual, scale, store, GroupNorm statistics); otherwise O / l is stored directly.
// q|k|v arrive packed along the channel axis of one [N, HW, 3C] tensor, addressed with one 3-D map.
//
// Budget (per CTA, one CTA per SM):
//   TMEM 512 columns: O [0, C) (C <= 256, later Y), S buffers at 256 and 256 + KT
//   shared memory, bf16 (KT = 128): Q 4 x 16 KB + P 2 x 16 KB + ring 4 x 16 KB (K / V / W3 tiles of
//     128 rows x 64 channels)                                                      = 160 KB + barriers
//   kX3 (KT = 64, every tile has a lo twin): Q 4 x 32 KB + P 1 x 32 KB + ring 4 x 16 KB (64 rows x 64
//     channels, hi | lo)                                                           = 224 KB + barriers
//   W3 tiles are KT output rows; the epilogue staging tiles alias the ring once every MMA is done.

#include <cuda.h>

#include <new>

#include "common.cuh"
#include "tc_common.cuh"
#include "conv_tc_common.cuh"

namespace psld {

template <bool kX3>
struct AsCfg {
  static constexpr int kTile = 128 * 64 * 2;                 // 128 rows x 64 bf16 (128 B rows, SW128)
  static constexpr int kMul = kX3 ? 2 : 1;
  static constexpr int kKT = kX3 ? 64 : 128;                 // keys per tile
  static constexpr int kQLo = 4 * kTile;                     // lo tiles of the Q region
  static constexpr int kQ = kQLo * kMul;
  static constexpr int kPLo = (kKT / 64) * kTile;            // lo tiles of the P region
  static constexpr int kP = kPLo * kMul;
  static constexpr int kSlotLo = kKT * 128;                  // lo half of a ring slot
  static constexpr int kSlot = kSlotLo * kMul;
  static constexpr int kRing = 4;
  static constexpr int kThreads = 192;
  static constexpr int kSmem = kQ + kP + kRing * kSlot + 256;
  static_assert(kSmem <= 227 * 1024, "shared-memory budget");
};
constexpr float kRescale = 8.0f;                             // lazy-rescale threshold (log2 units)

struct AttnStreamParams {
  __nv_bfloat16* out;
  int HW, C;
  float scale_log2;  // C^-0.5 * log2(e)
  ConvTcParams ep;   // kProj: epilogue of the fused NIN_3 projection
};

struct AttnStreamState {
  CUtensorMap tq, tkv, tw;
  bool proj, x3;
  AttnStreamParams p;
  dim3 grid;
};

__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]),
        "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]),
        "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]),
        "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]),
        "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

template <bool kProj, bool kX3>
__global__ void __launch_bounds__(AsCfg<kX3>::kThreads, 1)
attn_stream_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
                      const __grid_constant__ CUtensorMap tmW, const AttnStreamParams p) {
  using Cfg = AsCfg<kX3>;
  constexpr int KT = Cfg::kKT;
  constexpr uint32_t kTile = Cfg::kTile;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = smem_u32(smem_raw);
  if (base & 1023u) __trap();                        // SW128 atoms need 1024-byte alignment
  const uint32_t qs = base;                          // Q, later the normalised O
  const uint32_t ps = qs + Cfg::kQ;                  // P of the current key tile
  const uint32_t ring = ps + Cfg::kP;
  const uint32_t bar_base = ring + Cfg::kRing * Cfg::kSlot;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::kRing + s); };
  const uint32_t q_full = bar_base + 8u * (2 * Cfg::kRing);
  auto s_full = [&](int b) { return q_full + 8u + 8u * b; };
  const uint32_t p_ready = q_full + 24u;
  const uint32_t pv_done = q_full + 32u;
  const uint32_t o_ready = q_full + 40u;
  const uint32_t y_full = q_full + 48u;
  const uint32_t tmem_slot = q_full + 56u;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = blockIdx.y, q0 = blockIdx.x * 128;
  const int nck = p.C / 64;                          // 64-channel chunks
  const int nt = p.HW / KT;                          // key tiles
  const int w_rows = p.C < KT ? p.C : KT;            // output rows of a NIN_3 weight tile
  const int nwt = (p.C + w_rows - 1) / w_rows;       // C = 192, KT = 128: the second tile's rows past C
                                                     // are TMA zero fill
  const int lo_c = 3 * p.C;                          // kX3: lo half of a q|k|v row

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQ) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmKV) : "memory");
    if (kProj) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmW) : "memory");
    for (int s = 0; s < Cfg::kRing; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(q_full, 1);
    mbar_init(s_full(0), 1);
    mbar_init(s_full(1), 1);
    mbar_init(p_ready, 128);
    mbar_init(pv_done, 1);
    mbar_init(o_ready, 128);
    mbar_init(y_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(tmem_slot), "n"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  // dependents may start only once every CTA of this grid holds its TMEM: a dependent CTA that took
  // TMEM on this SM first would wait on this grid while this CTA waits for all 512 columns
  pdl_trigger_early();
  pdl_wait();
  const uint32_t tmem = *tmem_slot_ptr;              // O / Y at [0, C), S buffers at 256 + b * KT

  if (warp == 0) {
    // ===================== TMA producer (same order as the MMA issuer consumes) =====================
    if (lane == 0) {
      const uint32_t mul = kX3 ? 2u : 1u;
      mbar_arrive_expect_tx(q_full, (uint32_t)nck * kTile * mul);
      for (int c = 0; c < nck; ++c) {
        tma_load_3d(qs + (uint32_t)c * kTile, &tmQ, q_full, c * 64, q0, n);
        if (kX3) tma_load_3d(qs + Cfg::kQLo + (uint32_t)c * kTile, &tmQ, q_full, lo_c + c * 64, q0, n);
      }
      int slot = 0;
      uint32_t phase = 0;
      auto kv_tile = [&](int col, int key0) {
        mbar_wait(empty_bar(slot), phase ^ 1);
        mbar_arrive_expect_tx(full_bar(slot), (uint32_t)Cfg::kSlot);
        const uint32_t st = ring + (uint32_t)slot * Cfg::kSlot;
        tma_load_3d(st, &tmKV, full_bar(slot), col, key0, n);
        if (kX3) tma_load_3d(st + Cfg::kSlotLo, &tmKV, full_bar(slot), lo_c + col, key0, n);
        if (++slot == Cfg::kRing) { slot = 0; phase ^= 1; }
      };
      auto k_tiles = [&](int j) { for (int c = 0; c < nck; ++c) kv_tile(p.C + c * 64, j * KT); };
      k_tiles(0);
      if (nt > 1) k_tiles(1);
      for (int j = 0; j < nt; ++j) {
        for (int g = 0; g < nck; ++g) kv_tile(2 * p.C + g * 64, j * KT);
        if (j + 2 < nt) k_tiles(j + 2);
      }
      if (kProj) {   // NIN_3 weight tiles: (input-channel chunk, w_rows-row output tile)
        for (int c = 0; c < nck; ++c)
          for (int t = 0; t < nwt; ++t) {
            mbar_wait(empty_bar(slot), phase ^ 1);
            mbar_arrive_expect_tx(full_bar(slot), (uint32_t)w_rows * 128u * mul);
            const uint32_t st = ring + (uint32_t)slot * Cfg::kSlot;
            tma_load_2d(st, &tmW, full_bar(slot), c * 64, t * w_rows);
            if (kX3) tma_load_2d(st + Cfg::kSlotLo, &tmW, full_bar(slot), c * 64, p.C + t * w_rows);
            if (++slot == Cfg::kRing) { slot = 0; phase ^= 1; }
          }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      int slot = 0;
      uint32_t phase = 0;
      auto wait_slot = [&]() {
        mbar_wait(full_bar(slot), phase);
        tc_fence_after();
        return ring + (uint32_t)slot * Cfg::kSlot;
      };
      auto free_slot = [&]() {
        tc_commit(empty_bar(slot));
        if (++slot == Cfg::kRing) { slot = 0; phase ^= 1; }
      };
      // one (A tile, B tile) product group of 4 k-steps (64 channels); kX3: hi*hi + hi*lo + lo*hi
      auto kgroup = [&](uint32_t d, uint32_t a_hi, uint32_t b_hi, uint32_t a_lo, uint32_t b_lo, uint32_t idesc,
                        bool first) {
        const uint64_t ad = make_sw128_desc(a_hi), bd = make_sw128_desc(b_hi);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          tc_mma_bf16(d, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, (!first || k > 0) ? 1u : 0u);
        if (kX3) {
          const uint64_t al = make_sw128_desc(a_lo), bl = make_sw128_desc(b_lo);
#pragma unroll
          for (int k = 0; k < 4; ++k) tc_mma_bf16(d, ad + (uint64_t)(2 * k), bl + (uint64_t)(2 * k), idesc, 1u);
#pragma unroll
          for (int k = 0; k < 4; ++k) tc_mma_bf16(d, al + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, 1u);
        }
      };
      // S_j = Q K_j^T : M = 128, N = KT, both operands K-major
      const uint32_t idesc_s = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(KT >> 3) << 17) |
                               ((uint32_t)(128 >> 4) << 24);
      auto issue_s = [&](int j) {
        const uint32_t d = tmem + 256u + (uint32_t)(j & 1) * KT;
        for (int c = 0; c < nck; ++c) {
          const uint32_t st = wait_slot();
          kgroup(d, qs + (uint32_t)c * kTile, st, qs + Cfg::kQLo + (uint32_t)c * kTile, st + Cfg::kSlotLo, idesc_s,
                 c == 0);
          free_slot();
        }
        tc_commit(s_full(j & 1));
      };
      // O[:, g*64 ..] += P_j V_{g,j} : M = 128, N = 64, A = P (K-major over keys), B = V MN-major
      const uint32_t idesc_o = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) |
                               ((uint32_t)(64 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
      mbar_wait(q_full, 0);
      tc_fence_after();
      issue_s(0);
      if (nt > 1) issue_s(1);
      for (int j = 0; j < nt; ++j) {
        mbar_wait(p_ready, (uint32_t)(j & 1));   // P_j written, O rescaled, S_j read
        tc_fence_after();
        for (int g = 0; g < nck; ++g) {
          const uint32_t st = wait_slot();
          const uint32_t d = tmem + (uint32_t)g * 64u;
#pragma unroll
          for (int ks = 0; ks < KT / 16; ++ks) {
            const uint32_t pa = ps + (uint32_t)(ks >> 2) * kTile;
            const uint64_t adesc = make_sw128_desc(pa) + (uint64_t)(2 * (ks & 3));
            const uint64_t bdesc = make_sw128_desc(st + (uint32_t)ks * 2048u);   // 16 keys x 128 B
            tc_mma_bf16(d, adesc, bdesc, idesc_o, (j > 0 || ks > 0) ? 1u : 0u);
            if (kX3) {
              const uint64_t adesc_lo = make_sw128_desc(pa + Cfg::kPLo) + (uint64_t)(2 * (ks & 3));
              const uint64_t bdesc_lo = make_sw128_desc(st + Cfg::kSlotLo + (uint32_t)ks * 2048u);
              tc_mma_bf16(d, adesc, bdesc_lo, idesc_o, 1u);
              tc_mma_bf16(d, adesc_lo, bdesc, idesc_o, 1u);
            }
          }
          free_slot();
        }
        tc_commit(pv_done);
        if (j + 2 < nt) issue_s(j + 2);
      }
      if (kProj) {
        // Y[:, t*w_rows ..] += Onorm_c W3_{c,t}^T over the O columns (read into shared memory by then)
        const uint32_t idesc_y = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(w_rows >> 3) << 17) |
                                 ((uint32_t)(128 >> 4) << 24);
        mbar_wait(o_ready, 0);
        tc_fence_after();
        for (int c = 0; c < nck; ++c)
          for (int t = 0; t < nwt; ++t) {
            const uint32_t st = wait_slot();
            kgroup(tmem + (uint32_t)(t * w_rows), qs + (uint32_t)c * kTile, st, qs + Cfg::kQLo + (uint32_t)c * kTile,
                   st + Cfg::kSlotLo, idesc_y, c == 0);
            free_slot();
          }
        tc_commit(y_full);
      }
    }
  } else {
    // ===================== softmax + epilogue: 128 threads, one query row each =====================
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
    const float c = p.scale_log2;
    float m = 0.f, l = 0.f;                          // running max (log2 units, scaled) and sum
    for (int j = 0; j < nt; ++j) {
      const int b = j & 1;
      mbar_wait(s_full(b), (uint32_t)((j >> 1) & 1));
      tc_fence_after();
      const uint32_t sa = tmem + lane_addr + 256u + (uint32_t)b * KT;
      float mx = -INFINITY;
#pragma unroll 1
      for (int ch = 0; ch < KT; ch += 32) {
        uint32_t r[32];
        tmem_ld32(sa + (uint32_t)ch, r);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 32; ++i) mx = fmaxf(mx, __uint_as_float(r[i]));
      }
      const float mxs = mx * c;
      float alpha = 1.f;
      bool grow = false;
      if (j == 0) {
        m = mxs;
      } else if (mxs > m + kRescale) {
        alpha = exp2f(m - mxs);
        m = mxs;
        grow = true;
      }
      if (j > 0) {
        // PV_{j-1} is complete: the P region is free and O is final for tiles < j
        mbar_wait(pv_done, (uint32_t)((j - 1) & 1));
        tc_fence_after();
        if (__any_sync(0xffffffffu, grow)) {
          const uint32_t oa = tmem + lane_addr;
#pragma unroll 1
          for (int ch = 0; ch < p.C; ch += 32) {
            uint32_t r[32];
            tmem_ld32(oa + (uint32_t)ch, r);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) r[i] = __float_as_uint(__uint_as_float(r[i]) * alpha);
            tmem_st32(oa + (uint32_t)ch, r);
          }
          tmem_st_wait();
        }
        l *= alpha;
      }
#pragma unroll 1
      for (int ch = 0; ch < KT; ch += 32) {
        uint32_t r[32];
        tmem_ld32(sa + (uint32_t)ch, r);
        tmem_ld_wait();
        const uint32_t tile = ps + (uint32_t)(ch >> 6) * kTile + (uint32_t)row * 128u;
        const int cbase = (ch & 63) >> 3;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint32_t w[4], wl[4];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const float e0 = exp2f(fmaf(__uint_as_float(r[q * 8 + 2 * t]), c, -m));
            const float e1 = exp2f(fmaf(__uint_as_float(r[q * 8 + 2 * t + 1]), c, -m));
            if (kX3) {
              split_bf2(e0, e1, w[t], wl[t]);
              l += e0 + e1;
            } else {
              __nv_bfloat162 h = __floats2bfloat162_rn(e0, e1);
              // the sum of the ROUNDED values, so that P / l is a true softmax of P
              const float2 f = __bfloat1622float2(h);
              l += f.x + f.y;
              w[t] = *reinterpret_cast<uint32_t*>(&h);
            }
          }
          const uint32_t dst = tile + (uint32_t)(((cbase + q) ^ (row & 7)) << 4);
          sts128(dst, w[0], w[1], w[2], w[3]);
          if (kX3) sts128(dst + Cfg::kPLo, wl[0], wl[1], wl[2], wl[3]);
        }
      }
      // generic-proxy smem writes -> visible to the tensor core; S_j and O reads / stores are complete
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      tc_fence_before();
      mbar_arrive(p_ready);
    }
    mbar_wait(pv_done, (uint32_t)((nt - 1) & 1));
    tc_fence_after();
    const float inv = 1.0f / l;
    if (kProj) {
      // normalised O -> (split) bf16 over Q (tile = ch / 64); every S MMA completed before pv_done
#pragma unroll 1
      for (int ch = 0; ch < p.C; ch += 32) {
        uint32_t r[32];
        tmem_ld32(tmem + lane_addr + (uint32_t)ch, r);
        tmem_ld_wait();
        const uint32_t tile = qs + (uint32_t)(ch >> 6) * kTile + (uint32_t)row * 128u;
        const int cbase = (ch & 63) >> 3;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint32_t w[4], wl[4];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const float o0 = __uint_as_float(r[q * 8 + 2 * t]) * inv;
            const float o1 = __uint_as_float(r[q * 8 + 2 * t + 1]) * inv;
            if (kX3) split_bf2(o0, o1, w[t], wl[t]);
            else w[t] = f2_to_bf2(o0, o1);
          }
          const uint32_t dst = tile + (uint32_t)(((cbase + q) ^ (row & 7)) << 4);
          sts128(dst, w[0], w[1], w[2], w[3]);
          if (kX3) sts128(dst + Cfg::kQLo, wl[0], wl[1], wl[2], wl[3]);
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      tc_fence_before();
      mbar_arrive(o_ready);
      mbar_wait(y_full, 0);
      tc_fence_after();
      const int m_tile = n * (p.HW >> 7) + (int)blockIdx.x;
      const int ew = warp - 2;
      // staging tiles + additive vectors alias the ring: every TMA load has been consumed by now
#pragma unroll 1
      for (int half = 0; half < 2; ++half)
        tc_epilogue_tile<true, kX3 ? 32 : 64, !kX3, kX3>(p.ep, tmem, 0, m_tile, 0, p.ep.block_n, quarter, half, lane,
                                                         ring + (uint32_t)ew * 4096u,
                                                         ring + 8u * 4096u + (uint32_t)ew * 256u, []() {}, []() {});
    } else {
      __nv_bfloat16* orow = p.out + ((int64_t)n * p.HW + q0 + row) * (p.C * (kX3 ? 2 : 1));
#pragma unroll 1
      for (int ch = 0; ch < p.C; ch += 32) {
        uint32_t r[32];
        tmem_ld32(tmem + lane_addr + (uint32_t)ch, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          uint32_t w[4], wl[4];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const float o0 = __uint_as_float(r[j + 2 * t]) * inv;
            const float o1 = __uint_as_float(r[j + 2 * t + 1]) * inv;
            if (kX3) split_bf2(o0, o1, w[t], wl[t]);
            else w[t] = f2_to_bf2(o0, o1);
          }
          *reinterpret_cast<uint4*>(orow + ch + j) = make_uint4(w[0], w[1], w[2], w[3]);
          if (kX3) *reinterpret_cast<uint4*>(orow + p.C + ch + j) = make_uint4(wl[0], wl[1], wl[2], wl[3]);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(512) : "memory");
  }
}

// ---------------------------------------------------------------- host side
int prepare_attn_stream_tc(psld_op& op) {
  const int N = op.i[PSLD_ATTN_N], HW = op.i[PSLD_ATTN_HW], C = op.i[PSLD_ATTN_C];
  auto unsupported = [&](const char* why) {
    set_error("attn_tc: not eligible (%s): N=%d HW=%d C=%d", why, N, HW, C);
    return PSLD_EUNSUPPORTED;
  };
  const int adt = op.i[PSLD_ATTN_DTYPE];
  if (adt != PSLD_BF16 && adt != PSLD_BF16S) return unsupported("dtype must be bf16 or split bf16");
  const bool x3 = adt == PSLD_BF16S;
  const int cm = x3 ? 2 : 1;
  if (C % 64 || C < 64 || C > 256) return unsupported("C must be 64..256, multiple of 64");
  if (HW % 128 || HW < 512) return unsupported("HW must be 64, 128, 256 or a multiple of 128 from 512");
  if (N <= 0) return unsupported("N must be positive");
  if (!op.in[0] || !op.out[0]) { set_error("attn_tc: null pointer"); return PSLD_EINVAL; }
  AttnStreamState* st = new (std::nothrow) AttnStreamState();
  if (!st) { set_error("attn_tc: out of host memory"); return PSLD_ECUDA; }
  const int kt = x3 ? AsCfg<true>::kKT : AsCfg<false>::kKT;
  st->x3 = x3;
  int rc = encode_qkv_map(&st->tq, op.in[0], N, HW, cm * 3 * C, 128);
  if (rc == PSLD_OK) rc = encode_qkv_map(&st->tkv, op.in[0], N, HW, cm * 3 * C, kt);
  if (rc != PSLD_OK) { delete st; return rc; }
  st->p.out = (__nv_bfloat16*)op.out[0];
  st->p.HW = HW; st->p.C = C;
  st->p.scale_log2 = op.f[0] * 1.4426950408889634f;
  st->grid = dim3((unsigned)(HW / 128), (unsigned)N);
  // optional fused output projection (in[1] = W3 bf16 [C out, C in], in[2] = bias, in[3] = residual)
  st->proj = op.i[PSLD_ATTN_PROJ] != 0;
  if (st->proj) {
    if (!op.in[1] || !op.in[3]) { delete st; return unsupported("fused projection needs weight and residual"); }
    rc = encode_w_map(&st->tw, op.in[1], cm * C, C, C < kt ? C : kt);
    if (rc != PSLD_OK) { delete st; return rc; }
    ConvTcParams& e = st->p.ep;
    e = ConvTcParams{};
    e.bias = (const float*)op.in[2];
    e.temb = nullptr;
    e.res = (const __nv_bfloat16*)op.in[3];
    e.y = (__nv_bfloat16*)op.out[0];
    e.y_nchw = nullptr;
    e.mg_stats = (double*)op.out[1];
    e.cout_valid = C;
    e.scale = op.f[1];
    e.HW = HW; e.Cout = C; e.H = 0; e.W = 0;
    e.block_n = C; e.n_tiles_n = 1;
    e.M = (int64_t)N * HW;
  } else {
    st->tw = st->tq;       // unused
  }
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(attn_stream_tc_kernel<false, false>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, AsCfg<false>::kSmem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(attn_stream_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               AsCfg<false>::kSmem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(attn_stream_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               AsCfg<true>::kSmem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(attn_stream_tc_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               AsCfg<true>::kSmem);
    if (e != cudaSuccess) {
      set_error("attn_tc: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
      delete st;
      return PSLD_ECUDA;
    }
    attr_set = true;
  }
  op.aux = st;
  return PSLD_OK;
}

int release_attn_stream_tc(psld_op& op) {
  if (op.aux) {
    delete (AttnStreamState*)op.aux;
    op.aux = nullptr;
  }
  return PSLD_OK;
}

int run_attn_stream_tc(const psld_op& op, cudaStream_t s) {
  const AttnStreamState* st = (const AttnStreamState*)op.aux;
  PSLD_CHECK_ARG(st != nullptr, "attn_tc: op not prepared (call psld_op_prepare)");
#define ATTN_LAUNCH(PROJ, X3)                                                                          \
  PSLD_CHECK_CUDA(launch_pdl(attn_stream_tc_kernel<PROJ, X3>, st->grid, dim3(AsCfg<X3>::kThreads),     \
                             AsCfg<X3>::kSmem, s, 1, st->tq, st->tkv, st->tw, st->p))
  if (st->proj) { if (st->x3) ATTN_LAUNCH(true, true); else ATTN_LAUNCH(true, false); }
  else { if (st->x3) ATTN_LAUNCH(false, true); else ATTN_LAUNCH(false, false); }
#undef ATTN_LAUNCH
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}

}  // namespace psld
