// tcgen05 single-head attention block for the NCSN++ AttnBlockpp (reference layerspp.py:82-91):
//   w = softmax_keys( einsum(q, k) * C^-0.5 ) ;  h = einsum(w, v) ;  out = (NIN_3(h) + x) * scale
// over HW = 64/128/256 tokens of C = 64..256 channels per sample (16x16 and 8x8 maps).
//
// One CTA = one sample x 128 queries.  All HW keys fit in one accumulator, so there is no
// online-softmax rescaling:
//   S[128 x HW]  = Q K^T      tcgen05.mma, A = Q chunk (resident), B = K tile (64 channels x 128 keys,
//                             streamed by TMA through a 3-slot ring of 16 KB tiles), accumulator in TMEM
//   P            = exp2(S*c - max*c) -> bf16, written by the 128 softmax threads (one row each)
//                  straight into shared memory in the 128B-swizzled K-major UMMA layout, over Q
//   O[128 x C]   = P V        per (64-channel group, 128-key half): A = P, B = V tile as an MN-major
//                             operand (V is [keys, channels] in memory = contiguous along N); O reuses
//                             the TMEM columns of S
//   Y[128 x C]   = Onorm W3^T  (fused projection) A = O / rowsum written over P, B = NIN_3 weight
//                             tiles; Y reuses the same TMEM columns; conv epilogue finishes the tile
// q|k|v arrive packed along the channel axis of one [N, HW, 3C] tensor (the fused NIN_0/1/2 GEMM),
// addressed with ONE 3-D tensor map.

#include <cuda.h>

#include <new>

#include "common.cuh"
#include "tc_common.cuh"
#include "conv_tc_common.cuh"

namespace psld {

constexpr int AT_TILE = 128 * 64 * 2;           // one operand tile: 128 rows x 64 bf16 (128 B rows, SW128)
constexpr int AT_RING = 3;                      // ring slots

// Shared-memory plan (v2).  Everything is a [<=128 rows x 64 columns] bf16 tile of 16 KB:
//   QP region  4 tiles : the Q channel chunks during S = Q K^T, then P (4 key chunks, written by the
//                        softmax threads over Q, which is dead by then), then the normalised O (4
//                        channel chunks: the A operand of the output projection)
//   ring       3 slots : K tiles (64 channels x one 128-key half), then V tiles (one 128-key half x
//                        64 channels), then NIN_3 weight tiles (<=128 output rows x 64 input channels)
// and the accumulators share ONE 256-column TMEM window: S, then O (after every softmax thread has
// read S), then the projection Y (after O has been normalised into shared memory).  112 KB of shared
// memory and 256 TMEM columns per CTA = TWO CTAs per SM in the bf16 tier: the load / softmax /
// epilogue phases of one query tile overlap the MMA phases of another (v1 ran 1 CTA per SM with
// 231 KB and 512 columns: tensor pipe 16 %, warps active 9 %).
// kX3 = split-bf16 operands (the fp32-tolerance tier): q|k|v rows are [3C hi | 3C lo], every GEMM is
// three MMA groups hi*hi + hi*lo + lo*hi, every tile has a lo twin (QP 128 KB, ring 3 x 32 KB: one
// CTA per SM, but the 3-deep ring still overlaps loads with MMAs), the output is split bf16.
template <bool kX3>
struct AtCfg {
  static constexpr int kMul = kX3 ? 2 : 1;
  static constexpr int kQP = 4 * AT_TILE * kMul;             // hi tiles, then lo tiles
  static constexpr int kSlot = AT_TILE * kMul;               // hi | lo
  // kX3 (one CTA per SM, nothing else overlaps its serial phases): TWO warps per TMEM lane quarter share the
  // softmax, the O normalisation and the projection epilogue of a query row (columns / channels / column
  // groups split in two; row max and row sum are exchanged through 2 KB of shared memory)
  static constexpr int kParts = kX3 ? 2 : 1;
  static constexpr int kThreads = 64 + 128 * kParts;         // TMA warp, MMA warp, 4 * kParts softmax warps
  static constexpr int kXchg = kX3 ? 2048 : 0;               // row max / row sum exchange [2][2][128] floats
  static constexpr int kSmem = kQP + AT_RING * kSlot + 256 + kXchg;  // + barriers; the window must start on
                                                             // a 1024-byte boundary (it does; trap otherwise)
  static constexpr int kMinBlocks = kX3 ? 1 : 2;
};

// Optional per-CTA phase timeline (build with -DPSLD_TC_TRACE; scripts/attn_trace.py reads it)
#ifdef PSLD_TC_TRACE
__device__ long long g_at_trace[1024 * 8];
#define AT_TRACE(slot) do { if ((threadIdx.x & 31) == 0) { const int b_ = blockIdx.y * gridDim.x + blockIdx.x; if (b_ < 1024) g_at_trace[b_ * 8 + (slot)] = clock64(); } } while (0)
#else
#define AT_TRACE(slot) do { } while (0)
#endif

struct AttnTcParams {
  __nv_bfloat16* out;
  int HW, C, N;
  int q_rows;        // rows of the Q box: min(128, HW)
  int k_rows;        // rows of a K / V tile: min(128, HW)
  int w_rows;        // rows of a NIN_3 weight tile: min(128, C)
  float scale_log2;  // C^-0.5 * log2(e)
  ConvTcParams ep;   // kProj: epilogue of the fused NIN_3 projection (bias, residual, scale, stats)
};

struct AttnTcState {
  CUtensorMap tq, tkv, tw;
  bool proj, x3;
  AttnTcParams p;
  dim3 grid;
};

// kProj: the block's output projection rides along (AttnBlockpp, layerspp.py:87-91):
//   h = (NIN_3(O / rowsum) + x) * scale; the conv epilogue (bias, residual, scale, store, GroupNorm
//   statistics) finishes the tile: no O round trip through HBM, no separate 1x1 convolution launch.
template <bool kProj, bool kX3>
__global__ void __launch_bounds__(AtCfg<kX3>::kThreads, AtCfg<kX3>::kMinBlocks)
attn_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmKV,
               const __grid_constant__ CUtensorMap tmW, const AttnTcParams p) {
  using Cfg = AtCfg<kX3>;
  constexpr uint32_t QP_LO = 4u * AT_TILE;           // lo tiles of the QP region (kX3)
  constexpr uint32_t S_LO = AT_TILE;                 // lo half of a ring slot (kX3)
  extern __shared__ uint8_t smem_raw[];
  pdl_trigger_early();
  if (threadIdx.x == 0) AT_TRACE(0);
  const uint32_t base = smem_u32(smem_raw);
  if (base & 1023u) __trap();                        // SW128 atoms need 1024-byte alignment
  const uint32_t qp = base;
  const uint32_t ring = base + Cfg::kQP;
  const uint32_t bar_base = ring + AT_RING * Cfg::kSlot;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (AT_RING + s); };
  const uint32_t q_full = bar_base + 8u * (2 * AT_RING);
  const uint32_t s_full = q_full + 8u;
  const uint32_t p_ready = q_full + 16u;
  const uint32_t o_full = q_full + 24u;
  const uint32_t o_ready = q_full + 32u;
  const uint32_t y_full = q_full + 40u;
  const uint32_t tmem_slot = q_full + 48u;
  // kProj epilogue: staging tiles + additive vectors alias the (by then idle) ring
  const uint32_t stg_base = ring;
  const uint32_t addv_base = ring + 8u * 4096u;
  constexpr int kParts = Cfg::kParts;
  float* xchg = reinterpret_cast<float*>(smem_raw + (bar_base + 256u - base));   // kX3: [max | sum][part][row]
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - base));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = blockIdx.y, q0 = blockIdx.x * 128;
  const int nck = p.C / 64;                          // 64-channel chunks
  const int nkh = (p.HW + 127) / 128;                // 128-key halves
  const int nwt = (p.C + 127) / 128;                 // 128-row tiles of the NIN_3 weight
  const int lo_c = 3 * p.C;                          // kX3: lo half of a q|k|v row

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmQ) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmKV) : "memory");
    if (kProj) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmW) : "memory");
    for (int s = 0; s < AT_RING; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(q_full, 1);
    mbar_init(s_full, 1);
    mbar_init(p_ready, 128 * kParts);
    mbar_init(o_full, 1);
    mbar_init(o_ready, 128 * kParts);
    mbar_init(y_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(tmem_slot), "n"(256) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();                  // q|k|v come from the previous kernel (prologue above overlaps its tail)
  const uint32_t tmem_acc = *tmem_slot_ptr;          // 256 columns: S, then O, then Y

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      const uint32_t mul = kX3 ? 2u : 1u;
      mbar_arrive_expect_tx(q_full, (uint32_t)(nck * p.q_rows) * 128u * mul);
      for (int c = 0; c < nck; ++c) {
        tma_load_3d(qp + (uint32_t)c * AT_TILE, &tmQ, q_full, c * 64, q0, n);
        if (kX3) tma_load_3d(qp + QP_LO + (uint32_t)c * AT_TILE, &tmQ, q_full, lo_c + c * 64, q0, n);
      }
      int slot = 0;
      uint32_t phase = 0;
      auto next = [&]() { if (++slot == AT_RING) { slot = 0; phase ^= 1; } };
      // K tiles: (channel chunk, key half)
      for (int c = 0; c < nck; ++c)
        for (int h = 0; h < nkh; ++h) {
          mbar_wait(empty_bar(slot), phase ^ 1);
          mbar_arrive_expect_tx(full_bar(slot), (uint32_t)p.k_rows * 128u * mul);
          const uint32_t st = ring + (uint32_t)slot * Cfg::kSlot;
          tma_load_3d(st, &tmKV, full_bar(slot), p.C + c * 64, h * 128, n);
          if (kX3) tma_load_3d(st + S_LO, &tmKV, full_bar(slot), lo_c + p.C + c * 64, h * 128, n);
          next();
        }
      // V tiles: (channel group, key half)
      for (int g = 0; g < nck; ++g)
        for (int h = 0; h < nkh; ++h) {
          mbar_wait(empty_bar(slot), phase ^ 1);
          mbar_arrive_expect_tx(full_bar(slot), (uint32_t)p.k_rows * 128u * mul);
          const uint32_t st = ring + (uint32_t)slot * Cfg::kSlot;
          tma_load_3d(st, &tmKV, full_bar(slot), 2 * p.C + g * 64, h * 128, n);
          if (kX3) tma_load_3d(st + S_LO, &tmKV, full_bar(slot), lo_c + 2 * p.C + g * 64, h * 128, n);
          next();
        }
      if (kProj) {   // NIN_3 weight tiles: (input-channel chunk, 128-row output tile)
        for (int c = 0; c < nck; ++c)
          for (int t = 0; t < nwt; ++t) {
            mbar_wait(empty_bar(slot), phase ^ 1);
            mbar_arrive_expect_tx(full_bar(slot), (uint32_t)p.w_rows * 128u * mul);
            const uint32_t st = ring + (uint32_t)slot * Cfg::kSlot;
            tma_load_2d(st, &tmW, full_bar(slot), c * 64, t * 128);
            if (kX3) tma_load_2d(st + S_LO, &tmW, full_bar(slot), c * 64, p.C + t * 128);
            next();
          }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      int slot = 0;
      uint32_t phase = 0;
      auto next = [&]() { if (++slot == AT_RING) { slot = 0; phase ^= 1; } };
      // one (A tile, B tile) product group of 4 k-steps (64 channels); kX3: three groups
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
      // ---- S[:, h*128 ..] += Q_c K_{c,h}^T : M = 128, N = k_rows, both operands K-major
      const uint32_t idesc_s = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.k_rows >> 3) << 17) |
                               ((uint32_t)(128 >> 4) << 24);
      mbar_wait(q_full, 0);
      tc_fence_after();
      AT_TRACE(1);
      for (int c = 0; c < nck; ++c)
        for (int h = 0; h < nkh; ++h) {
          mbar_wait(full_bar(slot), phase);
          tc_fence_after();
          const uint32_t st = ring + (uint32_t)slot * Cfg::kSlot;
          kgroup(tmem_acc + (uint32_t)h * 128u, qp + (uint32_t)c * AT_TILE, st,
                 qp + QP_LO + (uint32_t)c * AT_TILE, st + S_LO, idesc_s, c == 0);
          tc_commit(empty_bar(slot));
          next();
        }
      tc_commit(s_full);
      // ---- O[:, g*64 ..] += P[:, keys of half h] V_{g,h} : M = 128, N = 64, A = P (K-major over
      // keys), B = V tile as an MN-major operand (V is [keys, channels] = contiguous along N)
      const uint32_t idesc_o = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) |
                               ((uint32_t)(64 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
      mbar_wait(p_ready, 0);           // P is in shared memory AND every thread is done reading S
      tc_fence_after();
      for (int g = 0; g < nck; ++g)
        for (int h = 0; h < nkh; ++h) {
          mbar_wait(full_bar(slot), phase);
          tc_fence_after();
          const uint32_t st = ring + (uint32_t)slot * Cfg::kSlot;
          const uint32_t d = tmem_acc + (uint32_t)g * 64u;
          for (int ks = 0; ks < p.k_rows / 16; ++ks) {
            const int kg = h * 8 + ks;                                       // global 16-key step
            const uint32_t pa = qp + (uint32_t)(kg >> 2) * AT_TILE;
            const uint64_t adesc = make_sw128_desc(pa) + (uint64_t)(2 * (kg & 3));
            const uint64_t bdesc = make_sw128_desc(st + (uint32_t)ks * 2048u);   // 16 keys x 128 B
            tc_mma_bf16(d, adesc, bdesc, idesc_o, (h > 0 || ks > 0) ? 1u : 0u);
            if (kX3) {
              const uint64_t adesc_lo = make_sw128_desc(pa + QP_LO) + (uint64_t)(2 * (kg & 3));
              const uint64_t bdesc_lo = make_sw128_desc(st + S_LO + (uint32_t)ks * 2048u);
              tc_mma_bf16(d, adesc, bdesc_lo, idesc_o, 1u);
              tc_mma_bf16(d, adesc_lo, bdesc, idesc_o, 1u);
            }
          }
          tc_commit(empty_bar(slot));
          next();
        }
      tc_commit(o_full);
      if (kProj) {
        // ---- Y[:, t*128 ..] += Onorm_c W3_{c,t}^T : A = Onorm chunk (K-major over channels, in the QP
        // region), B = weight tile (K-major), N = rows of the tile
        mbar_wait(o_ready, 0);         // normalised O is in shared memory AND O has been read from TMEM
        tc_fence_after();
        for (int c = 0; c < nck; ++c)
          for (int t = 0; t < nwt; ++t) {
            mbar_wait(full_bar(slot), phase);
            tc_fence_after();
            const int rows = (p.C - t * 128) < 128 ? (p.C - t * 128) : 128;
            const uint32_t idesc_y = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(rows >> 3) << 17) |
                                     ((uint32_t)(128 >> 4) << 24);
            const uint32_t st = ring + (uint32_t)slot * Cfg::kSlot;
            kgroup(tmem_acc + (uint32_t)t * 128u, qp + (uint32_t)c * AT_TILE, st,
                   qp + QP_LO + (uint32_t)c * AT_TILE, st + S_LO, idesc_y, c == 0);
            tc_commit(empty_bar(slot));
            next();
          }
        tc_commit(y_full);
      }
    }
  } else {
    // ===================== softmax + epilogue: 128 threads, one query row each =====================
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(quarter * 32) << 16;
    // kParts == 2: warps 2..5 take the first half of the keys / channels / column groups, warps 6..9 the
    // second; the two warps of a lane quarter meet on named barrier 2 + quarter (64 threads)
    const int part = kParts == 2 ? (warp >= 6 ? 1 : 0) : 0;
    const int k_lo = part * (p.HW / kParts), k_hi = k_lo + p.HW / kParts;
    const int c_lo = part * (p.C / kParts), c_hi = c_lo + p.C / kParts;
    auto pair_sync = [&]() {
      if (kParts == 2) asm volatile("bar.sync %0, 64;" ::"r"(2 + quarter) : "memory");
    };
    mbar_wait(s_full, 0);
    tc_fence_after();
    if (warp == 2) AT_TRACE(2);
    float mx = -INFINITY;
    for (int ch = k_lo; ch < k_hi; ch += 32) {
      uint32_t r[32];
      tmem_ld32(tmem_acc + lane_addr + (uint32_t)ch, r);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) mx = fmaxf(mx, __uint_as_float(r[j]));
    }
    if (kParts == 2) {
      xchg[part * 128 + row] = mx;
      pair_sync();
      mx = fmaxf(mx, xchg[(part ^ 1) * 128 + row]);
    }
    const float mxs = mx * p.scale_log2;
    float sum = 0.f;
    for (int ch = k_lo; ch < k_hi; ch += 32) {
      uint32_t r[32];
      tmem_ld32(tmem_acc + lane_addr + (uint32_t)ch, r);
      tmem_ld_wait();
      // P tile (ch / 64), 16-byte chunks (ch % 64) / 8 .. +3, swizzled by (row % 8); the Q tiles it
      // overwrites were last read by MMAs that completed before s_full
      const uint32_t tile = qp + (uint32_t)(ch >> 6) * AT_TILE + (uint32_t)row * 128u;
      const int cbase = (ch & 63) >> 3;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint32_t w[4], wl[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          const float e0 = exp2f(fmaf(__uint_as_float(r[q * 8 + 2 * t]), p.scale_log2, -mxs));
          const float e1 = exp2f(fmaf(__uint_as_float(r[q * 8 + 2 * t + 1]), p.scale_log2, -mxs));
          if (kX3) {
            split_bf2(e0, e1, w[t], wl[t]);
            sum += e0 + e1;
          } else {
            __nv_bfloat162 h = __floats2bfloat162_rn(e0, e1);
            // accumulate the sum from the ROUNDED values so that P / sum is a true softmax of P
            const float2 f = __bfloat1622float2(h);
            sum += f.x + f.y;
            w[t] = *reinterpret_cast<uint32_t*>(&h);
          }
        }
        const uint32_t dst = tile + (uint32_t)(((cbase + q) ^ (row & 7)) << 4);
        sts128(dst, w[0], w[1], w[2], w[3]);
        if (kX3) sts128(dst + QP_LO, wl[0], wl[1], wl[2], wl[3]);
      }
    }
    // generic-proxy smem writes -> visible to the tensor core (async proxy); the TMEM reads of S are
    // complete (tcgen05.wait::ld), so the MMA warp may overwrite the window with O
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    mbar_arrive(p_ready);
    if (warp == 2) AT_TRACE(3);
    if (kParts == 2) {
      xchg[256 + part * 128 + row] = sum;
      pair_sync();
      sum += xchg[256 + (part ^ 1) * 128 + row];
    }
    const float inv = 1.0f / sum;
    mbar_wait(o_full, 0);
    tc_fence_after();
    if (warp == 2) AT_TRACE(4);
    const int q = q0 + row;
    const bool valid = q < p.HW;
    if (kProj) {
      // normalised O -> (split) bf16 in the QP region, same swizzled K-major tiles (tile = ch / 64);
      // P was last read by MMAs that completed before o_full
      for (int ch = c_lo; ch < c_hi; ch += 32) {
        uint32_t r[32];
        tmem_ld32(tmem_acc + lane_addr + (uint32_t)ch, r);
        tmem_ld_wait();
        const uint32_t tile = qp + (uint32_t)(ch >> 6) * AT_TILE + (uint32_t)row * 128u;
        const int cbase = (ch & 63) >> 3;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint32_t w[4], wl[4];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const float o0 = __uint_as_float(r[j * 8 + 2 * t]) * inv;
            const float o1 = __uint_as_float(r[j * 8 + 2 * t + 1]) * inv;
            if (kX3) split_bf2(o0, o1, w[t], wl[t]);
            else w[t] = f2_to_bf2(o0, o1);
          }
          const uint32_t dst = tile + (uint32_t)(((cbase + j) ^ (row & 7)) << 4);
          sts128(dst, w[0], w[1], w[2], w[3]);
          if (kX3) sts128(dst + QP_LO, wl[0], wl[1], wl[2], wl[3]);
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      tc_fence_before();
      mbar_arrive(o_ready);
      if (warp == 2) AT_TRACE(5);
      mbar_wait(y_full, 0);
      tc_fence_after();
      if (warp == 2) AT_TRACE(6);
      const int m_tile = n * (p.HW >> 7) + (int)blockIdx.x;
      const int ew = warp - 2;                     // softmax / epilogue warps are warps 2..5 (kX3: 2..9)
#pragma unroll 1
      for (int half = (kParts == 2 ? part : 0); half < (kParts == 2 ? part + 1 : 2); ++half)
        tc_epilogue_tile<true, kX3 ? 32 : 64, !kX3, kX3>(p.ep, tmem_acc, 0, m_tile, 0, p.ep.block_n, quarter, half, lane,
                                                         stg_base + (uint32_t)ew * 4096u,
                                                         addv_base + (uint32_t)ew * 256u, []() {}, []() {});
    } else {
      __nv_bfloat16* orow = p.out + ((int64_t)n * p.HW + q) * (p.C * (kX3 ? 2 : 1));
      for (int ch = c_lo; ch < c_hi; ch += 32) {
        uint32_t r[32];
        tmem_ld32(tmem_acc + lane_addr + (uint32_t)ch, r);
        tmem_ld_wait();
        if (valid) {
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
        __syncwarp();
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) AT_TRACE(7);
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;"
                 ::"r"(tmem_acc), "n"(256) : "memory");
  }
}

#ifdef PSLD_TC_TRACE
extern "C" __attribute__((visibility("default"))) int psld_debug_attn_trace(long long* out) {
  return cudaMemcpyFromSymbol(out, g_at_trace, sizeof(g_at_trace)) == cudaSuccess ? 0 : 1;
}
#endif

// ---------------------------------------------------------------- host side
static int encode_qkv_map(CUtensorMap* tm, const void* ptr, int N, int HW, int C3, int rows) {
  const cuuint64_t dims[3] = {(cuuint64_t)C3, (cuuint64_t)HW, (cuuint64_t)N};
  const cuuint64_t strides[2] = {(cuuint64_t)C3 * 2, (cuuint64_t)HW * C3 * 2};
  const cuuint32_t box[3] = {64, (cuuint32_t)rows, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  return encode_bf16_map(tm, ptr, 3, dims, strides, box, estr, "qkv");
}

int prepare_attn_tc(psld_op& op) {
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
  if (HW != 64 && HW != 128 && HW != 256) return unsupported("HW must be 64, 128 or 256");
  if (!op.in[0] || !op.out[0]) { set_error("attn_tc: null pointer"); return PSLD_EINVAL; }
  AttnTcState* st = new (std::nothrow) AttnTcState();
  if (!st) { set_error("attn_tc: out of host memory"); return PSLD_ECUDA; }
  const int q_rows = HW < 128 ? HW : 128;
  st->x3 = x3;
  int rc = encode_qkv_map(&st->tq, op.in[0], N, HW, cm * 3 * C, q_rows);
  if (rc == PSLD_OK) rc = encode_qkv_map(&st->tkv, op.in[0], N, HW, cm * 3 * C, q_rows);   // 128-key halves
  if (rc != PSLD_OK) { delete st; return rc; }
  st->p.out = (__nv_bfloat16*)op.out[0];
  st->p.HW = HW; st->p.C = C; st->p.N = N; st->p.q_rows = q_rows;
  st->p.k_rows = q_rows; st->p.w_rows = C < 128 ? C : 128;
  st->p.scale_log2 = op.f[0] * 1.4426950408889634f;
  st->grid = dim3((unsigned)((HW + 127) / 128), (unsigned)N);
  // optional fused output projection (in[1] = W3 bf16 [C out, C in], in[2] = bias, in[3] = residual)
  st->proj = op.i[PSLD_ATTN_PROJ] != 0;
  if (st->proj) {
    if (HW % 128 || !op.in[1] || !op.in[3]) { delete st; return unsupported("fused projection needs HW %% 128 == 0, weight and residual"); }
    // W3 [C out, C in] (split: planes [2][C out, C in]) in <=128-row output tiles
    rc = encode_w_map(&st->tw, op.in[1], cm * C, C, C < 128 ? C : 128);
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
    cudaError_t e = cudaFuncSetAttribute(attn_tc_kernel<false, false>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, AtCfg<false>::kSmem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(attn_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               AtCfg<false>::kSmem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(attn_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               AtCfg<true>::kSmem);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(attn_tc_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               AtCfg<true>::kSmem);
    // two CTAs per SM (bf16 tier) need the maximum shared-memory carve-out
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(attn_tc_kernel<false, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(attn_tc_kernel<true, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
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

int release_attn_tc(psld_op& op) {
  if (op.aux) {
    delete (AttnTcState*)op.aux;
    op.aux = nullptr;
  }
  return PSLD_OK;
}

int run_attn_tc(const psld_op& op, cudaStream_t s) {
  const AttnTcState* st = (const AttnTcState*)op.aux;
  PSLD_CHECK_ARG(st != nullptr, "attn_tc: op not prepared (call psld_op_prepare)");
#define ATTN_LAUNCH(PROJ, X3)                                                                  \
  PSLD_CHECK_CUDA(launch_pdl(attn_tc_kernel<PROJ, X3>, st->grid, dim3(AtCfg<X3>::kThreads),       \
                             AtCfg<X3>::kSmem, s, 1, st->tq, st->tkv,                              \
                             st->tw, st->p))
  if (st->proj) { if (st->x3) ATTN_LAUNCH(true, true); else ATTN_LAUNCH(true, false); }
  else { if (st->x3) ATTN_LAUNCH(false, true); else ATTN_LAUNCH(false, false); }
#undef ATTN_LAUNCH
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}

}  // namespace psld
