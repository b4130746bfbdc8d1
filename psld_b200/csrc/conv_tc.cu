// tcgen05 / TMEM / TMA implicit-GEMM convolution for sm_100a (bf16 in, fp32 accumulate).
//
// Computes, for NHWC bf16 activations, y = scale * (conv_{KSxKS, stride 1, pad KS/2}(cat(x1,x2), W)
//                                                   + bias + temb[n,:] + residual)
// i.e. the reference's ddpm_conv3x3 / ddpm_conv1x1 / NIN call sites with their epilogue terms
// fused (layers.py:85-109,531-540; layerspp.py:242-274,75-91).  >= 97% of the network's FLOPs
// go through this kernel (SURVEY.md §8 a14/a15: conv3x3 71.09 + conv1x1 3.38 + NIN 1.24 of
// 76.43 GFLOP per sample per NFE).
//
// Design (B200-first, not a port: the reference calls cuDNN through ATen):
//   * GEMM view: M = N*H*W output pixels, N = Cout, K = KS*KS*Cin, K ordered (tap, channel).
//   * One CTA tile = 128 pixels x BLOCK_N channels; the accumulator lives in TMEM
//     (128 lanes x BLOCK_N fp32 columns), double-buffered (2 x 256 columns) so the epilogue of
//     tile i overlaps the MMAs of tile i+1.  Persistent CTAs, one per SM.
//   * A operand: for every (tap, 64-channel chunk) ONE 4-D TMA box {64 ch, BW, BH, BN} of the
//     NHWC tensor, shifted by the tap offset; out-of-image rows/columns are zero-filled by the
//     TMA unit, which is exactly the conv's zero padding - no im2col buffer, no halo code.
//     The box lands in shared memory as 128 rows x 128 B with the 128B swizzle = the canonical
//     K-major UMMA layout.
//   * B operand: weights pre-packed [Cout, K] bf16 (K-major), 2-D TMA box {64, BLOCK_N}.
//   * torch.cat([h, skip]) inputs (ncsnpp.py:374) are never materialised: the K loop walks two
//     tensor maps.
//   * Warp roles: warp 0 = A (activation) TMA producer, warp 10 = B (weight) TMA producer, warp 1 =
//     MMA issuer + TMEM allocator (all three run their loops converged, one elected lane issues),
//     warps 2-9 = epilogue (conv_tc_common.cuh: tcgen05.ld -> FFMA2 against a warp-uniform
//     (bias + temb) * scale vector -> + residual -> bf16 through a swizzled smem tile -> full-line
//     stores + GroupNorm statistics; two warps per TMEM lane quarter, each taking every other
//     64-column group, with the residual of the next group prefetched).
//   * smem ring of (A 16 KB + B 32 KB) stages, 4 deep (1-CTA) or (A 16 KB + half B 16 KB) 6 deep
//     (2-CTA cta_group::2, the default: one M = 256 MMA stream per CTA pair), mbarrier full/empty
//     pairs, tcgen05.commit releases stages and publishes accumulators.
//   * Optional K-extension: a 1x1 convolution over a second input (the residual block's Conv_2
//     shortcut) accumulated into the same tile through two more tensor maps.
//   * Programmatic dependent launch: dependents are released at entry, the A producer and the
//     epilogue warps execute griddepcontrol.wait before touching activations.

#include <cuda.h>

#include <new>

#include "common.cuh"
#include "tc_common.cuh"
#include "conv_tc_common.cuh"

namespace psld {

struct ConvTcState {
  CUtensorMap a1, a2, b, b2, e1, e2;      // b2: weight map with the N-slice box of the split tail units
  ConvTcParams p;
  int grid;
  bool pair;      // 2-CTA (cta_group::2) variant
  bool x3;        // split-bf16 operands, three MMA groups per k-block (fp32-tolerance tier)
};

// Optional per-CTA phase timeline (build with -DPSLD_TC_TRACE; scripts/tc_trace.py reads it)
#ifdef PSLD_TC_TRACE
__device__ long long g_tc_trace[160 * 8];
#define TC_TRACE(slot) do { if ((threadIdx.x & 31) == 0) g_tc_trace[blockIdx.x * 8 + (slot)] = clock64(); } while (0)
#else
#define TC_TRACE(slot) do { } while (0)
#endif

template <bool kPair, bool kX3>
__global__ void __launch_bounds__(TC_THREADS, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmA2,
               const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmB2,
               const __grid_constant__ CUtensorMap tmE1, const __grid_constant__ CUtensorMap tmE2,
               const ConvTcParams p) {
  using Cfg = TcCfg<kPair, kX3>;
  constexpr int kStages = Cfg::kStages;
  extern __shared__ uint8_t smem_raw[];
  if (threadIdx.x == 0) TC_TRACE(0);
  // PDL: the next kernel's CTAs may take this SM as soon as this CTA exits (one wave, persistent)
  pdl_launch_dependents();
  // 1024-byte alignment required by the 128B swizzle atoms
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t stg_base = base + kStages * Cfg::kStageBytes;
  const uint32_t bar_base = stg_base + Cfg::kStagingBytes;
  const uint32_t addv_base = bar_base + 256u;
  if (addv_base + Cfg::kAddvBytes > smem_u32(smem_raw) + Cfg::kSmemBytes) __trap();   // see TcCfg
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kStages + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * kStages + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * kStages + 2 + s); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * kStages + 4);
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = kPair ? cluster_ctarank() : 0u;   // 0 = leader (issues the MMAs)
  // work decomposition: a "unit" is one tile (1-CTA) or two vertically adjacent M tiles (pair)
  const int unit0 = kPair ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int unit_step = kPair ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA1) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA2) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar(s), 2);      // A producer + B producer (of the leader CTA)
      mbar_init(empty_bar(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), kPair ? 16 : 8);   // one arrive per epilogue warp (of both CTAs)
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if (kPair) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                   ::"r"(tmem_slot), "n"(TC_TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                   ::"r"(tmem_slot), "n"(TC_TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  if (kPair) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  if (threadIdx.x == 0) TC_TRACE(1);

  // K = taps x input channels, optionally followed by a 1x1 "extension" over a second input
  // (the residual block's Conv_2 shortcut accumulated into the same tile, layerspp.py:269-274)
  const int total_kb = p.taps * p.kchunks + p.ext_kchunks;
  auto decode = [&](int v, int& unit, int& nsub, int& bn) { tc_decode_unit(p, v, unit, nsub, bn); };

  if (warp == 0 || warp == 10) {
    // ===================== TMA producers (both CTAs of a pair) =====================
    // warp 0 streams the activation (A) boxes, warp 10 the weight (B) boxes: two independent
    // single-thread issue loops (one loop issuing both was the limiter: it was never blocked on a
    // free stage, i.e. it could not issue fast enough to stay ahead of the tensor core).  The
    // warp stays converged and one elected lane issues (uniform-datapath coordinates).
    {
      const bool is_a = warp == 0;
      if (is_a) pdl_wait();     // activations come from the previous kernel; weights do not
      const uint32_t tx_mul = (kPair ? 2u : 1u) * (kX3 ? 2u : 1u);
      // one A / B tile of this stage (kX3: called for the hi half, then for the lo half)
      auto load_a = [&](uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c, int x, int y, int n) {
        if (kPair) tma_load_4d_pair(dst, tm, bar, c, x, y, n);
        else tma_load_4d(dst, tm, bar, c, x, y, n);
      };
      auto load_b = [&](uint32_t dst, const CUtensorMap* tm, uint32_t bar, int k, int row) {
        if (kPair) tma_load_2d_pair(dst, tm, bar, k, row);
        else tma_load_2d(dst, tm, bar, k, row);
      };
      int stage = 0;
      uint32_t phase = 0;
      for (int v = unit0; v < p.num_virtual; v += unit_step) {
        int unit, nsub, bn;
        decode(v, unit, nsub, bn);
        const int n_tile = unit % p.n_tiles_n;
        const int m_tile = kPair ? 2 * (unit / p.n_tiles_n) + (int)rank : unit / p.n_tiles_n;
        const int n0 = (m_tile / p.tiles_y) * p.BN_img;
        const int t_img = m_tile % p.tiles_y;                      // (row group, x-tile) in the image
        const int y0 = (t_img / p.tiles_x) * p.BH * p.stride - p.pad;
        const int x0 = (t_img % p.tiles_x) * TC_BLOCK_M;           // 256-wide rows: two 128-pixel halves
        const int b_rows = kPair ? (bn >> 1) : bn;                 // weight rows this CTA loads
        const CUtensorMap* tmW = nsub < 0 ? &tmB : &tmB2;
        const int bn0 = n_tile * p.block_n + (nsub < 0 ? 0 : nsub * bn) + (kPair ? (int)rank * b_rows : 0);
        const uint32_t my_tx = (is_a ? (uint32_t)TC_A_BYTES : (uint32_t)b_rows * TC_BLOCK_K * 2) * tx_mul;
        int kb = 0;
        for (int ky = 0; ky < p.KS; ++ky) {
          for (int kx = 0; kx < p.KS; ++kx) {
            for (int cc = 0; cc < p.kchunks; ++cc, ++kb) {
              mbar_wait(empty_bar(stage), phase ^ 1);
              const uint32_t sa = base + stage * Cfg::kStageBytes;
              if (elect_one()) {
                if (!kPair || rank == 0) mbar_arrive_expect_tx(full_bar(stage), my_tx);
                if (is_a) {
                  const bool s1 = cc < p.kchunks1;
                  const CUtensorMap* tmA = s1 ? &tmA1 : &tmA2;
                  const int c0 = (s1 ? cc : cc - p.kchunks1) * TC_BLOCK_K;
                  load_a(sa, tmA, full_bar(stage), c0, x0 + kx - p.pad, y0 + ky, n0);
                  if (kX3)
                    load_a(sa + TC_A_BYTES, tmA, full_bar(stage), c0 + (s1 ? p.lo1 : p.lo2), x0 + kx - p.pad,
                           y0 + ky, n0);
                } else {
                  load_b(sa + Cfg::kBOff, tmW, full_bar(stage), kb * TC_BLOCK_K, bn0);
                  if (kX3)
                    load_b(sa + Cfg::kBOff + Cfg::kBBytes, tmW, full_bar(stage), kb * TC_BLOCK_K,
                           bn0 + p.w_lo_rows);
                }
              }
              __syncwarp();
              if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
          }
        }
        for (int cc = 0; cc < p.ext_kchunks; ++cc, ++kb) {    // shortcut input, centre tap only
          mbar_wait(empty_bar(stage), phase ^ 1);
          const uint32_t sa = base + stage * Cfg::kStageBytes;
          if (elect_one()) {
            if (!kPair || rank == 0) mbar_arrive_expect_tx(full_bar(stage), my_tx);
            if (is_a) {
              const bool s1 = cc < p.ext_kchunks1;
              const CUtensorMap* tmE = s1 ? &tmE1 : &tmE2;
              const int c0 = (s1 ? cc : cc - p.ext_kchunks1) * TC_BLOCK_K;
              load_a(sa, tmE, full_bar(stage), c0, x0, y0 + p.pad, n0);
              if (kX3)
                load_a(sa + TC_A_BYTES, tmE, full_bar(stage), c0 + (s1 ? p.loe1 : p.loe2), x0,
                       y0 + p.pad, n0);
            } else {
              load_b(sa + Cfg::kBOff, tmW, full_bar(stage), kb * TC_BLOCK_K, bn0);
              if (kX3)
                load_b(sa + Cfg::kBOff + Cfg::kBBytes, tmW, full_bar(stage), kb * TC_BLOCK_K,
                       bn0 + p.w_lo_rows);
            }
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    // The whole warp runs the loop converged (every value warp-uniform) and one elected lane
    // issues: with a divergent `lane == 0` branch around the loop ptxas wraps every tcgen05
    // instruction in an ELECT / R2UR.BROADCAST sequence and the issue loop itself (about 120
    // instructions per k-block, never waiting on a barrier) paces the tensor pipe.
    if (rank == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int v = unit0; v < p.num_virtual; v += unit_step) {
        int unit, nsub, bn;
        decode(v, unit, nsub, bn);
        // instruction descriptor: D=f32, A=B=bf16, both K-major, N=bn, M=128 (256 for a pair)
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(bn >> 3) << 17) |
                               ((uint32_t)((kPair ? 256 : 128) >> 4) << 24);
        if (kPair) mbar_wait_cluster(tempty_bar(acc), acc_phase ^ 1);
        else mbar_wait(tempty_bar(acc), acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * 256u;
        for (int kb = 0; kb < total_kb; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          if (kb == 0 && v == unit0) TC_TRACE(2);
          const uint32_t sa = base + stage * Cfg::kStageBytes;
          const uint64_t adesc = make_sw128_desc(sa);
          const uint64_t bdesc = make_sw128_desc(sa + Cfg::kBOff);
          if (elect_one()) {
            auto group = [&](uint64_t ad, uint64_t bd, bool first) {
#pragma unroll
              for (int k = 0; k < TC_BLOCK_K / 16; ++k) {
                // advance 16 bf16 = 32 B inside the swizzle atom: +2 in the (addr >> 4) field
                const uint32_t accum = (!first || kb > 0 || k > 0) ? 1u : 0u;
                if (kPair) tc_mma_bf16_pair(d_tmem, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, accum);
                else tc_mma_bf16(d_tmem, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, accum);
              }
            };
            group(adesc, bdesc, true);                               // a_hi * w_hi
            if (kX3) {
              const uint64_t adesc_lo = make_sw128_desc(sa + TC_A_BYTES);
              const uint64_t bdesc_lo = make_sw128_desc(sa + Cfg::kBOff + Cfg::kBBytes);
              group(adesc, bdesc_lo, false);                         // a_hi * w_lo
              group(adesc_lo, bdesc, false);                         // a_lo * w_hi
            }
            // frees the smem stage (in both CTAs) when these MMAs retire
            if (kPair) tc_commit_pair(empty_bar(stage)); else tc_commit(empty_bar(stage));
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        // accumulator ready for the epilogue (of both CTAs)
        if (elect_one()) {
          if (kPair) tc_commit_pair(tfull_bar(acc)); else tc_commit(tfull_bar(acc));
        }
        __syncwarp();
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
      TC_TRACE(3);
    }
  } else if (warp < 10) {
    // ===================== epilogue (warps 2..9) =====================
    const int quarter = warp & 3;        // TMEM lane quarter this warp may access (warp id % 4)
    const int half = (warp - 2) >> 2;    // this warp takes the 32-column chunks with index % 2 == half
    const uint32_t leader_tempty0 = kPair ? mapa_rank(tempty_bar(0), 0) : 0u;
    int acc = 0;
    uint32_t acc_phase = 0;
    pdl_wait();                 // residual / temb reads and every global write come after this
    for (int v = unit0; v < p.num_virtual; v += unit_step) {
      int unit, nsub, bn;
      decode(v, unit, nsub, bn);
      const int n_tile = nsub < 0 ? unit % p.n_tiles_n : (unit % p.n_tiles_n) * p.n_split + nsub;   // in units of bn
      const int m_tile = kPair ? 2 * (unit / p.n_tiles_n) + (int)rank : unit / p.n_tiles_n;
      tc_epilogue_tile<true, kX3 ? 32 : 64, !kX3, kX3>(
          p, tmem_base, acc, m_tile, n_tile, bn, quarter, half, lane,
          stg_base + (uint32_t)(warp - 2) * 4096u, addv_base + (uint32_t)(warp - 2) * 256u,
          [&]() {
            mbar_wait(tfull_bar(acc), acc_phase);
            tc_fence_after();
            if (warp == 2) TC_TRACE(4);
          },
          [&]() {
            // the accumulator is in registers: hand it back before the stores are issued
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              if (kPair) mbar_arrive_remote_relaxed(leader_tempty0 + 8u * (uint32_t)acc);
              else mbar_arrive(tempty_bar(acc));
            }
          });
      if (warp == 2) TC_TRACE(5);
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }

  tc_fence_before();
  if (kPair) cluster_sync_all(); else __syncthreads();
  if (threadIdx.x == 0) TC_TRACE(6);
  if (warp == 1) {
    tc_fence_after();
    if (kPair)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;"
                   ::"r"(tmem_base), "n"(TC_TMEM_COLS) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;"
                   ::"r"(tmem_base), "n"(TC_TMEM_COLS) : "memory");
  }
}

// ---------------------------------------------------------------- host side
// Activation map over the INPUT tensor [N, H, W, C]; the box covers BW x BH x BN output positions
// visited with element stride `stride` (TMA loads ceil(box / stride) elements per dimension).
// (split bf16: C = 2 x channels, the row holds [hi | lo])
static int encode_act_map(CUtensorMap* tm, const void* ptr, int N, int H, int W, int C, int BW,
                          int BH, int BN_img, int stride) {
  const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  const cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  const cuuint32_t box[4] = {(cuuint32_t)TC_BLOCK_K, (cuuint32_t)(BW * stride), (cuuint32_t)(BH * stride),
                             (cuuint32_t)BN_img};
  const cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
  return encode_bf16_map(tm, ptr, 4, dims, strides, box, estr, "activation");
}

static bool is_pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

int prepare_conv_tc(psld_op& op) {
  const int N = op.i[PSLD_CONV_N], H = op.i[PSLD_CONV_H], W = op.i[PSLD_CONV_W];
  const int C1 = op.i[PSLD_CONV_C1], C2 = op.i[PSLD_CONV_C2], Cout = op.i[PSLD_CONV_COUT];
  const int KS = op.i[PSLD_CONV_KS];
  auto unsupported = [&](const char* why) {
    set_error("conv_tc: not eligible (%s): N=%d H=%d W=%d C1=%d C2=%d Cout=%d KS=%d", why, N, H, W,
              C1, C2, Cout, KS);
    return PSLD_EUNSUPPORTED;
  };
  const bool head = op.i[PSLD_CONV_OUT_LAYOUT] == PSLD_NCHW;   // fp32 NCHW output head
  const int adt = op.i[PSLD_CONV_IN_DTYPE];
  if (adt != PSLD_BF16 && adt != PSLD_BF16S) return unsupported("input dtype must be bf16 or split bf16");
  const bool x3 = adt == PSLD_BF16S;
  const int cm = x3 ? 2 : 1;                                   // bf16 elements per channel in a row
  if (op.i[PSLD_CONV_OUT_DTYPE] != (head ? PSLD_F32 : adt))
    return unsupported("output must be NHWC of the input's element type, or fp32 NCHW");
  if (op.i[PSLD_CONV_IN_LAYOUT] != PSLD_NHWC) return unsupported("input layout must be NHWC");
  if (head && (op.f[1] < 1.0f || (int)op.f[1] > Cout))
    return unsupported("NCHW head needs f[1] = valid channels");
  if (head && op.in[2] && op.i[PSLD_CONV_RES_DTYPE] != PSLD_F32)
    return unsupported("NCHW head residual must be fp32 NCHW");
  const int stride = op.i[PSLD_CONV_STRIDE], pad = op.i[PSLD_CONV_PAD];
  const bool same = stride == 1 && pad == KS / 2 && (KS == 1 || KS == 3);
  const bool down2 = stride == 2 && pad == 0 && KS == 3 && C2 == 0;   // conv_downsample_2d's conv
  if (!same && !down2) return unsupported("stride 1 'same' or 3x3 stride 2 pad 0 only");
  const int OH = op.i[PSLD_CONV_OH], OW = op.i[PSLD_CONV_OW];
  if (OH != (H + 2 * pad - KS) / stride + 1 || OW != (W + 2 * pad - KS) / stride + 1) {
    set_error("conv_tc: OH/OW mismatch");
    return PSLD_EINVAL;
  }
  if (C1 % TC_BLOCK_K || C2 % TC_BLOCK_K) return unsupported("Cin %% 64 != 0");
  if (Cout % 32) return unsupported("Cout %% 32 != 0");
  if (!is_pow2(OW) || !is_pow2(OH) || OW > (same ? 256 : 128) || OW < 4)
    return unsupported("output W,H must be pow2, 4..256 (stride 1) or 4..128");
  if (!head && op.in[2] && op.i[PSLD_CONV_RES_DTYPE] != adt) return unsupported("residual dtype");
  if (x3 && !head && (OH * OW) % 32) return unsupported("split bf16 output needs H*W %% 32 == 0");
  if (!op.in[0] || !op.in[4] || !op.out[0] || (C2 > 0 && !op.in[1])) {
    set_error("conv_tc: null pointer");
    return PSLD_EINVAL;
  }
  // N tile = the widest that divides Cout.  (Measured: narrowing to N=128 to fix the wave
  // quantisation of the 16x16 layers - 7 half rounds instead of 4 - is a net loss, 2.0 -> 2.8 ms:
  // k-blocks then retire every 256 cycles and the TMA issue loops cannot keep up.)
  int block_n = 0;
  for (int cand : {256, 128, 64, 32})
    if (Cout % cand == 0) { block_n = cand; break; }
  // M tile = 128 output pixels: whole rows of BN_img images, or half a row when OW = 256
  const int BW = OW < TC_BLOCK_M ? OW : TC_BLOCK_M;
  int BH = 128 / BW;
  if (BH > OH) BH = OH;
  const int BN_img = 128 / (BW * BH);
  if (BN_img > 256) return unsupported("image too small");

  const int sms = sm_count();
  // 2-CTA pairs whenever there are at least two M tiles
  const int64_t m_tiles_all = (int64_t)((N + BN_img - 1) / BN_img) * (OH / BH) * (OW / BW);
  const bool pair = m_tiles_all >= 2 && sms >= 2;
  ConvTcState* st = new (std::nothrow) ConvTcState();
  if (!st) { set_error("conv_tc: out of host memory"); return PSLD_ECUDA; }
  int rc = encode_act_map(&st->a1, op.in[0], N, H, W, cm * C1, BW, BH, BN_img, stride);
  if (rc == PSLD_OK)
    rc = C2 > 0 ? encode_act_map(&st->a2, op.in[1], N, H, W, cm * C2, BW, BH, BN_img, stride)
                : encode_act_map(&st->a2, op.in[0], N, H, W, cm * C1, BW, BH, BN_img, stride);
  const int E1 = op.i[PSLD_CONV_EXT_C1], E2 = op.i[PSLD_CONV_EXT_C2];
  const bool ext = op.in[8] != nullptr && E1 > 0;
  if (ext && (stride != 1 || E1 % TC_BLOCK_K || E2 % TC_BLOCK_K || (E2 > 0 && !op.in[9]))) {
    delete st;
    return unsupported("1x1 extension needs stride 1 and channel counts %% 64 == 0");
  }
  if (rc == PSLD_OK)
    rc = ext ? encode_act_map(&st->e1, op.in[8], N, OH, OW, cm * E1, BW, BH, BN_img, 1)
             : encode_act_map(&st->e1, op.in[0], N, H, W, cm * C1, BW, BH, BN_img, stride);
  if (rc == PSLD_OK)
    rc = (ext && E2 > 0) ? encode_act_map(&st->e2, op.in[9], N, OH, OW, cm * E2, BW, BH, BN_img, 1)
                         : encode_act_map(&st->e2, op.in[0], N, H, W, cm * C1, BW, BH, BN_img, stride);
  const int K = KS * KS * (C1 + C2) + (ext ? E1 + E2 : 0);
  // split bf16 weights: two planes [2][Cout, K] seen as one [2*Cout, K] matrix
  if (rc == PSLD_OK) rc = encode_w_map(&st->b, op.in[4], cm * Cout, K, pair ? block_n / 2 : block_n);
  if (rc != PSLD_OK) { delete st; return rc; }
  st->b2 = st->b;

  ConvTcParams& p = st->p;
  tc_conv_params(p, op, head, OH, OW, BH, BN_img, block_n);
  if (p.mg_stats && (head || (OH * OW) % 32 != 0)) {
    delete st;
    set_error("conv_tc: micro-group stats need NHWC bf16 output and H*W %% 32 == 0");
    return PSLD_EINVAL;
  }
  st->x3 = x3;
  const int64_t m_tiles = (int64_t)((N + BN_img - 1) / BN_img) * p.tiles_y;
  const int64_t m_units = pair ? (m_tiles + 1) / 2 : m_tiles;
  p.num_tiles = (int)(m_units * p.n_tiles_n);          // work units (tiles, or tile pairs)
  st->pair = pair;
  // ---- last partial round: split its units along N when that lets the idle clusters share the work
  // (16x16 CIFAR layers at B = 256: 256 tile pairs over 74 clusters = 3 rounds + 34 units; as 68
  // half-N units the tail costs half a round: 4 -> 3.5 rounds).
  const int best = tc_plan_tail_split(p, pair ? sms / 2 : sms, 64, !head);
  if (best > 1) {
    const int sub = block_n / best;
    rc = encode_w_map(&st->b2, op.in[4], cm * Cout, K, pair ? sub / 2 : sub);
    if (rc != PSLD_OK) { delete st; return rc; }
  }
  if (pair) {
    const int pairs = sms / 2;
    st->grid = 2 * (p.num_virtual < pairs ? p.num_virtual : pairs);
  } else {
    st->grid = p.num_virtual < sms ? p.num_virtual : sms;
  }
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_tc_kernel<false, false>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         TcCfg<false, false>::kSmemBytes);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(conv_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               TcCfg<true, false>::kSmemBytes);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(conv_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               TcCfg<false, true>::kSmemBytes);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(conv_tc_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               TcCfg<true, true>::kSmemBytes);
    if (e != cudaSuccess) {
      set_error("conv_tc: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
      delete st;
      return PSLD_ECUDA;
    }
    attr_set = true;
  }
  op.aux = st;
  return PSLD_OK;
}

int release_conv_tc(psld_op& op) {
  if (op.aux) {
    delete (ConvTcState*)op.aux;
    op.aux = nullptr;
  }
  return PSLD_OK;
}

int run_conv_tc(const psld_op& op, cudaStream_t s) {
  const ConvTcState* st = (const ConvTcState*)op.aux;
  PSLD_CHECK_ARG(st != nullptr, "conv_tc: op not prepared (call psld_op_prepare)");
#define CONV_TC_LAUNCH(PAIR, X3)                                                               \
  PSLD_CHECK_CUDA(launch_pdl(conv_tc_kernel<PAIR, X3>, dim3((unsigned)st->grid), dim3(TC_THREADS), \
                             TcCfg<PAIR, X3>::kSmemBytes, s, PAIR ? 2 : 1, st->a1, st->a2, st->b,  \
                             st->b2, st->e1, st->e2, st->p))
  if (st->pair) {
    if (st->x3) CONV_TC_LAUNCH(true, true); else CONV_TC_LAUNCH(true, false);
  } else {
    if (st->x3) CONV_TC_LAUNCH(false, true); else CONV_TC_LAUNCH(false, false);
  }
#undef CONV_TC_LAUNCH
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}

}  // namespace psld

#ifdef PSLD_TC_TRACE
extern "C" __attribute__((visibility("default"))) int psld_debug_tc_trace(long long* out) {
  return (int)cudaMemcpyFromSymbol(out, psld::g_tc_trace, sizeof(psld::g_tc_trace));
}
#endif
