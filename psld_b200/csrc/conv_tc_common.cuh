// Shared pieces of the tcgen05 convolution kernels: parameters, 2-CTA (cta_group::2) PTX wrappers
// and the epilogue (TMEM -> registers -> bias/temb/residual/scale -> bf16 through a swizzled
// shared-memory tile -> coalesced global stores, plus GroupNorm micro-group statistics).
#pragma once

#include "common.cuh"
#include "tc_common.cuh"

namespace psld {

constexpr int TC_BLOCK_M = 128;
constexpr int TC_BLOCK_K = 64;        // bf16 elements = one 128-byte swizzle row
constexpr int TC_STAGES = 4;
constexpr int TC_A_BYTES = TC_BLOCK_M * TC_BLOCK_K * 2;   // 16 KB
constexpr int TC_B_BYTES = 256 * TC_BLOCK_K * 2;          // 32 KB (max BLOCK_N = 256)
constexpr int TC_STAGE_BYTES = TC_A_BYTES + TC_B_BYTES;
constexpr int TC_SMEM_BYTES = TC_STAGES * TC_STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
constexpr int TC_THREADS = 352;        // A-TMA warp + MMA warp + 8 epilogue warps + B-TMA warp
constexpr int TC_TMEM_COLS = 512;

struct ConvTcParams {
  const float* bias;
  const float* temb;
  const __nv_bfloat16* res;
  __nv_bfloat16* y;
  float* y_nchw;             // when non-null: fp32 NCHW output, first cout_valid channels only
  const float* res_nchw;     // optional fp32 NCHW residual of the y_nchw head (same shape as y_nchw)
  double* mg_stats;         // optional [N, Cout/4, 2] per-sample (sum, sumsq) of the output per 4
                             // channels, accumulated with atomics (zeroed by the caller)
  int cout_valid;
  float scale;
  int temb_off, temb_bstride;
  int H, W, HW, Cout;        // OUTPUT map size (== input size for the stride-1 'same' case)
  int stride, pad;           // 1/KS/2, or 2/0 (3x3 stride-2 conv on a pre-padded input)
  int BH, BN_img;            // output rows / images per tile: min(W,128)*BH*BN_img == 128; the TMA box
                             // is {64, min(W,128)*stride, BH*stride, BN_img} traversed with element stride
  int tiles_x;               // tiles per output row: W / 128 for W = 256 (BH = BN_img = 1), else 1
  int tiles_y;               // M tiles per BN_img images: (H / BH) * tiles_x
  int kchunks1, kchunks;     // 64-channel chunks in source 1 / in total (C1+C2)/64
  int taps, KS;
  int ext_kchunks1, ext_kchunks;   // 64-channel chunks of the fused 1x1 shortcut input (0 = none)
  int block_n, n_tiles_n;
  int num_tiles;
  int64_t M;                 // N*H*W
  // split-bf16 ("bf16x3") operands: channel offset of the lo half inside a pixel row of source
  // 1 / 2 / shortcut 1 / shortcut 2 (= the source's channel count) and row offset of the lo plane of
  // the weight matrix (= its padded Cout); the output / residual rows are [Cout hi | Cout lo]
  int lo1, lo2, loe1, loe2, w_lo_rows;
  // last partial round: units >= tail_start are processed as n_split N-slices of block_n / n_split
  // channels each ("virtual units" tail_start + (u - tail_start) * n_split + slice), so that the
  // clusters that would idle in that round share its work; num_virtual = total loop trip count
  int tail_start, n_split, num_virtual;
};


// ---------------------------------------------------------------- the kernel
// kPair = false: one CTA per tile (tcgen05 cta_group::1, M = 128).
// kPair = true : a cluster of two CTAs (one TPC) works on two vertically adjacent M tiles with ONE
//   tcgen05.mma.cta_group::2 stream (M = 256) issued by the leader CTA.  Each CTA loads its own
//   A tile and only HALF of the weight tile (block_n/2 rows); the tensor core reads the B halves
//   from both CTAs' shared memory.  Per CTA and k-block this cuts the L2->SM traffic from 48 KB to
//   32 KB and frees room for a 6-deep ring (ncu on the 1-CTA kernel: tensor pipe 75 % active with
//   the XBAR at 15.6 TB/s and only ~1.3 us of TMA lookahead).
// kX3 = the fp32-tolerance tier: activations and weights are split bf16 (hi + lo); one stage holds
//   A_hi | A_lo | B_hi | B_lo of a k-block and feeds THREE MMA groups (hi*hi, hi*lo, lo*hi) into
//   the same fp32 accumulator: products to ~2^-17 relative instead of bf16's 2^-9, at 3x the
//   tensor-pipe work and 2x the operand bytes per k-block (half as many, twice as long stages).
template <bool kPair, bool kX3 = false>
struct TcCfg {
  static constexpr int kStages = kX3 ? (kPair ? 3 : 2) : (kPair ? 6 : TC_STAGES);
  static constexpr int kBBytes = kPair ? TC_B_BYTES / 2 : TC_B_BYTES;
  static constexpr int kStageBytes = (TC_A_BYTES + kBBytes) * (kX3 ? 2 : 1);
  static constexpr int kBOff = kX3 ? 2 * TC_A_BYTES : TC_A_BYTES;   // first B tile inside a stage
  static constexpr int kStagingBytes = 8 * 4096;   // epilogue transpose buffers, 4 KB per warp
  static constexpr int kAddvBytes = 8 * 256;       // (bias + temb) * scale, 64 columns per warp
  // 768 B of alignment slack: the kernel traps if the dynamic window starts further than that
  // from a 1024-byte boundary (it starts ON one in practice); total = the 227 KB maximum
  static constexpr int kSmemBytes = kStages * kStageBytes + kStagingBytes + 256 + kAddvBytes + 768;
};

// virtual unit v -> (unit, N slice index or -1, N width): full units first, then the N-split units of
// the last partial round (ConvTcParams::tail_start / n_split)
__device__ __forceinline__ void tc_decode_unit(const ConvTcParams& p, int v, int& unit, int& nsub, int& bn) {
  if (v < p.tail_start) {
    unit = v; nsub = -1; bn = p.block_n;
  } else {
    const int t = v - p.tail_start;
    const int u = t / p.n_split;
    unit = p.tail_start + u; nsub = t - u * p.n_split; bn = p.block_n / p.n_split;
  }
}

// Host: choose the N-split of the last partial round.  `workers` = clusters (or CTAs) that run
// concurrently, `min_sub` = smallest / granularity of the N slice.  Fills tail_start / n_split /
// num_virtual and returns n_split.
static inline int tc_plan_tail_split(ConvTcParams& p, int workers, int min_sub, bool enable) {
  const int full = p.num_tiles / workers, tail = p.num_tiles % workers;
  int best = 1;
  double best_cost = full + (tail > 0 ? 1.0 : 0.0);
  if (enable && tail > 0) {
    for (int ns : {2, 4}) {
      const int sub = p.block_n / ns;
      if (p.block_n % ns || sub < min_sub || sub % min_sub) continue;
      const double cost = full + (double)((tail * ns + workers - 1) / workers) / ns;
      if (cost < best_cost - 1e-9) { best_cost = cost; best = ns; }
    }
  }
  p.n_split = best;
  p.tail_start = best > 1 ? p.num_tiles - tail : p.num_tiles;
  p.num_virtual = p.tail_start + (p.num_tiles - p.tail_start) * best;
  return best;
}

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same smem offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_rank(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr)
               : "memory");
}
// no memory ordering needed (the payload is "TMEM has been read", completed by tcgen05.wait::ld);
// the .release form costs a MEMBAR that waits for every store in flight
__device__ __forceinline__ void mbar_arrive_remote_relaxed(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait_cluster(bar, parity)) return;
  const long long t0 = clock64();
  uint32_t spins = 0;
  while (!mbar_try_wait_cluster(bar, parity)) {
    if ((++spins & 0xFFF) == 0 && clock64() - t0 > 8000000000LL) __trap();
  }
}
// 2-CTA TMA loads: data lands in THIS CTA's smem, bytes are credited to the LEADER's mbarrier
// (peer bit 24 of the shared::cluster address cleared)
__device__ __forceinline__ void tma_load_4d_pair(uint32_t dst, const CUtensorMap* tm, uint32_t bar,
                                                 int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(tm), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* tm, uint32_t bar,
                                                 int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(tm), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc,
                                                 uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

// packed fp32x2 FMA (Blackwell FFMA2): (d0, d1) = (a0, a1) * (b0, b1) + (c0, c1)
__device__ __forceinline__ void ffma2(float& d0, float& d1, float a0, float a1, float b0, float b1,
                                      float c0, float c1) {
  uint64_t a, b, c, d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(b0), "f"(b1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(c) : "f"(c0), "f"(c1));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d0), "=f"(d1) : "l"(d));
}
__device__ __forceinline__ uint4 lds128(uint32_t a) {
  uint4 q;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(q.x), "=r"(q.y), "=r"(q.z), "=r"(q.w) : "r"(a) : "memory");
  return q;
}
__device__ __forceinline__ void sts128(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w)
               : "memory");
}

// One output tile: TMEM accumulator -> (+bias +temb +residual) * scale -> bf16 NHWC (or the fp32
// NCHW network head) + GroupNorm micro-group statistics.  Called by the 8 epilogue warps;
// `quarter` = TMEM lane quarter (warp id % 4), `half` selects alternate column groups, `stg` =
// this warp's 4 KB staging tile and `addv` its 256 B additive-vector slot in shared memory.
// `bn` = N width of THIS tile (p.block_n, or a fraction of it for the N-split units of the last
// partial round), `n_tile` = index in units of `bn`.
// `acquire()` is called once before the first TMEM access (it waits for the accumulator),
// `release()` right after this warp's LAST TMEM read (it hands the accumulator back to the MMA
// warp before the global stores are issued, so the release never waits on them).
// kPrefetchRes: keep the NEXT column group's residual in registers while the current one is
// processed (GC/2 registers); kTmemAhead (GC = 64): second TMEM chunk in flight while the first is
// processed (32 registers).  Both off for kernels that are short of registers.
// kSplit: output / residual are split bf16 ([Cout hi | Cout lo] rows): GC must be 32 and `stg` holds
// two 2 KB tiles (hi, lo) per warp.
template <bool kPrefetchRes = true, int GC = 64, bool kTmemAhead = true, bool kSplit = false,
          class Acquire, class Release>
__device__ __forceinline__ void tc_epilogue_tile(const ConvTcParams& p, uint32_t tmem_base, int acc,
                                                 int m_tile, int n_tile, const int bn, int quarter, int half,
                                                 int lane, uint32_t stg, uint32_t addv,
                                                 Acquire acquire, Release release) {
  static_assert(GC == 64 || GC == 32, "staging group = 64 or 32 columns");
  static_assert(!kSplit || GC == 32, "split-bf16 output stages 32-column groups");
  constexpr int NT = kSplit ? 2 : 1;                  // staging tiles / global planes (hi, lo)
  const int64_t m = (int64_t)m_tile * TC_BLOCK_M + quarter * 32 + lane;
  const bool valid = m < p.M;
  const int slot = m_tile * 4 + quarter;             // 32-row slot of the micro-group stats
  const bool stats = p.mg_stats != nullptr && (int64_t)slot * 32 < p.M;
  if (p.y != nullptr && (bn & (GC - 1)) == 0 && (p.HW & 31) == 0) {
    // ---- staged path: GC-column groups go through a per-warp 32 x (2*GC) B shared-memory tile
    // (16-byte chunks XOR-swizzled by row) so that BOTH the residual loads and the output
    // stores hit global memory as full 128-byte (GC = 32: 64-byte) row segments, 4 (8) rows per
    // instruction, instead of 32 scattered 16-byte pieces; thread <-> TMEM row only touches its
    // own row of the tile.
    // HW % 32 == 0: the warp's 32 pixels belong to ONE image, so (bias + temb) * scale is a
    // warp-uniform vector: GC/4 lanes fetch it once per column group into `addv`, and every
    // output is one FFMA2 lane (acc * scale + addv), two with a residual.
    constexpr int RB = GC * 2;                        // staging row bytes
    constexpr int CPR = GC / 8;                       // 16-byte chunks per row
    constexpr int RPI = 32 / CPR;                     // rows per coalesced instruction
    constexpr int ITS = 32 / RPI;                     // coalesced instructions per group
    constexpr int NSUB = GC / 32;
    auto swz = [](int row) { return GC == 64 ? (row & 7) : ((row >> 1) & 3); };
    const int64_t m_base = (int64_t)m_tile * TC_BLOCK_M + quarter * 32;
    const bool full = m_base + 32 <= p.M;             // warp-uniform: no per-row bounds checks
    const int sub_row = lane / CPR, chunk = lane % CPR;
    const int ncg = bn / GC;
    constexpr uint32_t TILE = 32u * RB;               // bytes of one staging tile
    const int64_t ldo = (int64_t)p.Cout * NT;          // output / residual row stride (elements)
    const uint32_t my_row = stg + (uint32_t)lane * RB;
    const int my_swz = swz(lane);
    const float scale = p.scale;
    const float* tembw = nullptr;
    if (p.temb) tembw = p.temb + (m_base < p.M ? m_base / p.HW : 0) * p.temb_bstride + p.temb_off;
    uint4 rq[NT][ITS];
    float4 av = make_float4(0.f, 0.f, 0.f, 0.f);
    auto load_add = [&](int cg) {
      if (lane < GC / 4) {
        const int c = n_tile * bn + cg * GC + 4 * lane;
        av = p.bias ? __ldg(reinterpret_cast<const float4*>(p.bias + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (tembw) {
          const float4 t = __ldg(reinterpret_cast<const float4*>(tembw + c));
          av.x += t.x; av.y += t.y; av.z += t.z; av.w += t.w;
        }
      }
    };
    const int64_t rowstep = (int64_t)RPI * ldo;       // RPI rows (elements)
    auto load_res = [&](int cg) {
#pragma unroll
      for (int pl = 0; pl < NT; ++pl) {
        const __nv_bfloat16* rp = p.res + (int64_t)n_tile * bn + cg * GC + chunk * 8 +
                                  (m_base + sub_row) * ldo + pl * p.Cout;
        if (full) {
#pragma unroll
          for (int it = 0; it < ITS; ++it) rq[pl][it] = *reinterpret_cast<const uint4*>(rp + it * rowstep);
        } else {
#pragma unroll
          for (int it = 0; it < ITS; ++it)
            if (m_base + RPI * it + sub_row < p.M)
              rq[pl][it] = *reinterpret_cast<const uint4*>(rp + it * rowstep);
        }
      }
    };
    // one 32-column chunk: r = accumulator row fragment -> bf16 into this thread's row of the
    // staging tile (+ micro-group statistics)
    auto process = [&](uint32_t (&r)[32], int sub, int co0) {
      uint4 ad[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) ad[q] = lds128(addv + (uint32_t)(sub * 32 + q * 4) * 4u);
      float v[32];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        ffma2(v[4 * q], v[4 * q + 1], __uint_as_float(r[4 * q]), __uint_as_float(r[4 * q + 1]), scale,
              scale, __uint_as_float(ad[q].x), __uint_as_float(ad[q].y));
        ffma2(v[4 * q + 2], v[4 * q + 3], __uint_as_float(r[4 * q + 2]), __uint_as_float(r[4 * q + 3]),
              scale, scale, __uint_as_float(ad[q].z), __uint_as_float(ad[q].w));
      }
      if (p.res) {
        uint4 wq[4], wl[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          wq[q] = lds128(my_row + (uint32_t)(((sub * 4 + q) ^ my_swz) << 4));
          if (kSplit) wl[q] = lds128(my_row + TILE + (uint32_t)(((sub * 4 + q) ^ my_swz) << 4));
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint32_t w[4] = {wq[q].x, wq[q].y, wq[q].z, wq[q].w};
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[t]));
            if (kSplit) {
              const uint32_t wlo[4] = {wl[q].x, wl[q].y, wl[q].z, wl[q].w};
              const float2 g = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&wlo[t]));
              f.x += g.x;
              f.y += g.y;
            }
            ffma2(v[q * 8 + 2 * t], v[q * 8 + 2 * t + 1], f.x, f.y, scale, scale, v[q * 8 + 2 * t],
                  v[q * 8 + 2 * t + 1]);
          }
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint32_t o[4], ol[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          if (kSplit) {
            split_bf2(v[q * 8 + 2 * t], v[q * 8 + 2 * t + 1], o[t], ol[t]);
          } else {
            __nv_bfloat162 h = __floats2bfloat162_rn(v[q * 8 + 2 * t], v[q * 8 + 2 * t + 1]);
            o[t] = *reinterpret_cast<uint32_t*>(&h);
          }
        }
        sts128(my_row + (uint32_t)(((sub * 4 + q) ^ my_swz) << 4), o[0], o[1], o[2], o[3]);
        if (kSplit)
          sts128(my_row + TILE + (uint32_t)(((sub * 4 + q) ^ my_swz) << 4), ol[0], ol[1], ol[2], ol[3]);
      }
      if (stats) {
        // GroupNorm statistics of the tensor being written, at 4-channel ("micro-group")
        // granularity: (sum, sum of squares) over this warp's 32 pixels (one sample: HW % 32 ==
        // 0).  16 values per lane are transposed-and-reduced across the warp with 16 shuffles
        // (halving butterfly) and accumulated per sample with f64 atomics; the consumer
        // GroupNorm sums the micro-groups of each of its groups.
        if (!full && !valid) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0.f;
        }
        float a[16];
#pragma unroll
        for (int g = 0; g < 8; ++g) {
          const float x0 = v[4 * g], x1 = v[4 * g + 1], x2 = v[4 * g + 2], x3 = v[4 * g + 3];
          a[2 * g] = (x0 + x1) + (x2 + x3);
          a[2 * g + 1] = fmaf(x0, x0, fmaf(x1, x1, fmaf(x2, x2, x3 * x3)));
        }
#pragma unroll
        for (int w = 8; w >= 1; w >>= 1) {
          const bool hi = (lane & (2 * w)) != 0;
#pragma unroll
          for (int j = 0; j < w; ++j) {
            const float send = hi ? a[j] : a[j + w];
            const float keep = hi ? a[j + w] : a[j];
            a[j] = keep + __shfl_xor_sync(0xffffffffu, send, 2 * w);
          }
        }
        a[0] += __shfl_xor_sync(0xffffffffu, a[0], 1);
        if ((lane & 1) == 0)     // 16 lanes: 8 micro-groups x (sum, sumsq) of this warp's 32 pixels
          atomicAdd(p.mg_stats + ((m_base / p.HW) * (p.Cout >> 2) + (co0 >> 2)) * 2 + (lane >> 1),
                    (double)a[0]);
      }
    };
    if (half < ncg) {
      load_add(half);
      if (p.res) load_res(half);
    }
    acquire();
    if (half >= ncg) release();
    for (int cg = half; cg < ncg; cg += 2) {
      const int co_base = n_tile * bn + cg * GC;
      const bool more = cg + 2 < ncg;
      if (lane < GC / 4)
        sts128(addv + (uint32_t)lane * 16u, __float_as_uint(av.x * scale), __float_as_uint(av.y * scale),
               __float_as_uint(av.z * scale), __float_as_uint(av.w * scale));
      if (p.res) {
        if (!kPrefetchRes && cg != half) load_res(cg);
#pragma unroll
        for (int pl = 0; pl < NT; ++pl)
#pragma unroll
          for (int it = 0; it < ITS; ++it) {
            const int row = RPI * it + sub_row;
            sts128(stg + pl * TILE + (uint32_t)row * RB + (uint32_t)((chunk ^ swz(row)) << 4),
                   rq[pl][it].x, rq[pl][it].y, rq[pl][it].z, rq[pl][it].w);
          }
      }
      __syncwarp();
      if (more) {
        load_add(cg + 2);
        if (kPrefetchRes && p.res) load_res(cg + 2);
      }
      {
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) +
                               (uint32_t)acc * 256u + (uint32_t)(cg * GC);
        if (NSUB == 1) {
          uint32_t r[32];
          tmem_ld32(taddr, r);
          tmem_ld_wait();
          if (!more) release();
          process(r, 0, co_base);
        } else if (kTmemAhead) {
          uint32_t r0[32], r1[32];
          tmem_ld32(taddr, r0);
          tmem_ld_wait();
          tmem_ld32(taddr + 32u, r1);        // in flight while the first chunk is processed
          process(r0, 0, co_base);
          tmem_ld_wait();
          if (!more) release();
          process(r1, 1, co_base + 32);
        } else {                             // register-lean order
          uint32_t r[32];
          tmem_ld32(taddr, r);
          tmem_ld_wait();
          process(r, 0, co_base);
          tmem_ld32(taddr + 32u, r);
          tmem_ld_wait();
          if (!more) release();
          process(r, 1, co_base + 32);
        }
      }
      __syncwarp();
#pragma unroll
      for (int pl = 0; pl < NT; ++pl) {
        __nv_bfloat16* yp = p.y + co_base + chunk * 8 + (m_base + sub_row) * ldo + pl * p.Cout;
        uint4 q[ITS];
#pragma unroll
        for (int it = 0; it < ITS; ++it) {
          const int row = RPI * it + sub_row;
          q[it] = lds128(stg + pl * TILE + (uint32_t)row * RB + (uint32_t)((chunk ^ swz(row)) << 4));
        }
        if (full) {
#pragma unroll
          for (int it = 0; it < ITS; ++it) *reinterpret_cast<uint4*>(yp + it * rowstep) = q[it];
        } else {
#pragma unroll
          for (int it = 0; it < ITS; ++it)
            if (m_base + RPI * it + sub_row < p.M) *reinterpret_cast<uint4*>(yp + it * rowstep) = q[it];
        }
      }
      __syncwarp();
    }
  } else {
  if (kSplit && p.y != nullptr) __trap();     // split-bf16 NHWC output exists only on the staged path
  acquire();
  const int img = valid ? (int)(m / p.HW) : 0;
  const float* temb = p.temb ? p.temb + (int64_t)img * p.temb_bstride + p.temb_off : nullptr;
  const bool has_res = valid && p.res != nullptr;
  uint4 rq[4];                                       // residual of the chunk being processed
  if (has_res && half * 32 < bn) {
    const __nv_bfloat16* rp = p.res + m * p.Cout + n_tile * bn + half * 32;
#pragma unroll
    for (int t = 0; t < 4; ++t) rq[t] = *reinterpret_cast<const uint4*>(rp + 8 * t);
  }
  for (int ch = half * 32; ch < bn; ch += 64) {
    uint32_t r[32];
    const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) +
                           (uint32_t)acc * 256u + (uint32_t)ch;
    tmem_ld32(taddr, r);
    const int co0 = n_tile * bn + ch;
    uint4 rn[4];                                     // prefetch the next chunk's residual
    const bool more = ch + 64 < bn;
    if (has_res && more) {
      const __nv_bfloat16* rp = p.res + m * p.Cout + co0 + 64;
#pragma unroll
      for (int t = 0; t < 4; ++t) rn[t] = *reinterpret_cast<const uint4*>(rp + 8 * t);
    }
    tmem_ld_wait();
    float v[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = valid ? __uint_as_float(r[j]) : 0.f;
    if (valid) {
      const int64_t o = m * p.Cout + co0;
      if (p.bias) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + co0 + j));
          v[j] += b.x; v[j + 1] += b.y; v[j + 2] += b.z; v[j + 3] += b.w;
        }
      }
      if (temb) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 b = __ldg(reinterpret_cast<const float4*>(temb + co0 + j));
          v[j] += b.x; v[j + 1] += b.y; v[j + 2] += b.z; v[j + 3] += b.w;
        }
      }
      if (p.res) {
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          const uint4 q = rq[j >> 3];
          const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&w[t]);
            const float2 f = __bfloat1622float2(h);
            v[j + 2 * t] += f.x;
            v[j + 2 * t + 1] += f.y;
          }
        }
      }
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] *= p.scale;
      if (p.y_nchw) {
        // network output head (ncsnpp.py:430): fp32 NCHW, lanes = consecutive pixels; the output
        // pyramid of progressive=output_skip arrives as an fp32 NCHW residual (ncsnpp.py:414-418)
        const int64_t pix = m - (int64_t)img * p.HW;
        if (p.res_nchw) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int64_t o = ((int64_t)img * p.cout_valid + co0 + j) * p.HW + pix;
            if (co0 + j < p.cout_valid) p.y_nchw[o] = fmaf(p.scale, __ldg(p.res_nchw + o), v[j]);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int co = co0 + j;
            if (co < p.cout_valid)
              p.y_nchw[((int64_t)img * p.cout_valid + co) * p.HW + pix] = v[j];
          }
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          uint32_t w[4];
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            __nv_bfloat162 h = __floats2bfloat162_rn(v[j + 2 * t], v[j + 2 * t + 1]);
            w[t] = *reinterpret_cast<uint32_t*>(&h);
          }
          *reinterpret_cast<uint4*>(p.y + o + j) = make_uint4(w[0], w[1], w[2], w[3]);
        }
      }
    }
    if (has_res && more) {
#pragma unroll
      for (int t = 0; t < 4; ++t) rq[t] = rn[t];
    }
    __syncwarp();
    if (stats) {
      // GroupNorm statistics of the tensor being written, at 4-channel ("micro-group")
      // granularity: (sum, sum of squares) over this warp's 32 pixels.  16 values per lane are
      // transposed-and-reduced across the warp with 16 shuffles (halving butterfly); the
      // consumer GroupNorm combines micro-groups into its groups (gn_finalize_kernel).
      float a[16];
#pragma unroll
      for (int g = 0; g < 8; ++g) {
        const float x0 = v[4 * g], x1 = v[4 * g + 1], x2 = v[4 * g + 2], x3 = v[4 * g + 3];
        a[2 * g] = (x0 + x1) + (x2 + x3);
        a[2 * g + 1] = fmaf(x0, x0, fmaf(x1, x1, fmaf(x2, x2, x3 * x3)));
      }
#pragma unroll
      for (int w = 8; w >= 1; w >>= 1) {
        const bool hi = (lane & (2 * w)) != 0;
#pragma unroll
        for (int j = 0; j < w; ++j) {
          const float send = hi ? a[j] : a[j + w];
          const float keep = hi ? a[j + w] : a[j];
          a[j] = keep + __shfl_xor_sync(0xffffffffu, send, 2 * w);
        }
      }
      a[0] += __shfl_xor_sync(0xffffffffu, a[0], 1);
      if ((lane & 1) == 0) {
        const int idx = lane >> 1;     // = bit4*8 + bit3*4 + bit2*2 + bit1
        atomicAdd(p.mg_stats + (((int64_t)slot * 32 / p.HW) * (p.Cout >> 2) + (co0 >> 2)) * 2 + idx,
                  (double)a[0]);
      }
    }
  }
  release();
  }  // legacy (non-staged) path
}

// Host: [rows, K] bf16 weight matrix, K contiguous (split bf16: the planes [2][Cout, K] as one
// [2*Cout, K] matrix); box = one 64-wide K chunk x box_rows rows.
static inline int encode_w_map(CUtensorMap* tm, const void* ptr, int rows, int K, int box_rows) {
  const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)K * 2};
  const cuuint32_t box[2] = {(cuuint32_t)TC_BLOCK_K, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  return encode_bf16_map(tm, ptr, 2, dims, strides, box, estr, "weight");
}

// Host: SMs of the current device (148 if the query fails).
static inline int sm_count() {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
    cudaGetLastError();
    sms = 148;
  }
  return sms;
}

// Host: the ConvTcParams fields that follow from a validated conv op record and its tiling (OH x OW
// output, M tiles of BH rows x BN_img images, N tiles of block_n channels).  num_tiles and the tail
// split are left to the caller.
static inline void tc_conv_params(ConvTcParams& p, const psld_op& op, bool head, int OH, int OW, int BH,
                                  int BN_img, int block_n) {
  const int N = op.i[PSLD_CONV_N], C1 = op.i[PSLD_CONV_C1], C2 = op.i[PSLD_CONV_C2];
  const int Cout = op.i[PSLD_CONV_COUT], KS = op.i[PSLD_CONV_KS];
  const int E1 = op.i[PSLD_CONV_EXT_C1], E2 = op.i[PSLD_CONV_EXT_C2];
  const bool ext = op.in[8] != nullptr && E1 > 0;
  p.bias = (const float*)op.in[5];
  p.temb = (const float*)op.in[3];
  p.res = head ? nullptr : (const __nv_bfloat16*)op.in[2];
  p.y = head ? nullptr : (__nv_bfloat16*)op.out[0];
  p.y_nchw = head ? (float*)op.out[0] : nullptr;
  p.res_nchw = head ? (const float*)op.in[2] : nullptr;
  p.cout_valid = head ? (int)op.f[1] : Cout;
  p.mg_stats = (double*)op.out[1];
  p.scale = op.f[0];
  p.temb_off = op.i[PSLD_CONV_TEMB_OFF];
  p.temb_bstride = op.i[PSLD_CONV_TEMB_BSTRIDE];
  p.H = OH; p.W = OW; p.HW = OH * OW; p.Cout = Cout;
  p.stride = op.i[PSLD_CONV_STRIDE]; p.pad = op.i[PSLD_CONV_PAD];
  p.BH = BH; p.BN_img = BN_img;
  p.tiles_x = OW > TC_BLOCK_M ? OW / TC_BLOCK_M : 1;
  p.tiles_y = OH / BH * p.tiles_x;
  p.kchunks1 = C1 / TC_BLOCK_K; p.kchunks = (C1 + C2) / TC_BLOCK_K;
  p.taps = KS * KS; p.KS = KS;
  p.ext_kchunks1 = ext ? E1 / TC_BLOCK_K : 0;
  p.ext_kchunks = ext ? (E1 + E2) / TC_BLOCK_K : 0;
  p.block_n = block_n; p.n_tiles_n = Cout / block_n;
  p.M = (int64_t)N * OH * OW;
  p.lo1 = C1; p.lo2 = C2; p.loe1 = E1; p.loe2 = E2; p.w_lo_rows = Cout;
}

}  // namespace psld
