// GroupNorm+SiLU-on-load 3x3 convolution: tcgen05 (cta_group::2) implicit GEMM whose A operand is
// normalised INSIDE the kernel, so the separate GroupNorm "apply" pass over HBM (read x, write
// silu(gn(x)), 20 % of the sampler step) disappears for the layers this kernel takes.
//
//   y = scale * ( conv3x3( silu( x * sc[n,c] + sh[n,c] ) ) + bias + temb + residual )
//
// with (sc, sh) the per-(sample, channel) affine form of GroupNorm (gn_affine_micro_kernel) — i.e.
// ResnetBlockBigGANpp's  act(GroupNorm_k(.)) -> Conv_k  pairs (reference layerspp.py:243,259,266).
//
// How the normalisation is applied once per element although a 3x3 conv reads every pixel 9 times:
// per (tile, 64-channel chunk) the RAW tile plus its vertical halo ((BH+2) x W pixels, out-of-image
// rows zero-filled by TMA) is loaded ONCE; eight "transform" warps normalise it in shared memory and
// write three operand tiles: centre, shifted left and shifted right by one pixel (image-edge
// columns zeroed = the conv's horizontal padding).  The 9 taps are then plain descriptor offsets:
// kx selects the variant, ky adds ky*W rows (a multiple of the 1024-byte swizzle atom for
// W = 16, 32), so no tap needs its own load.  L2->SM traffic for A drops from 9 x 16 KB to 24 KB
// per chunk; weights stream per tap through a 4-stage ring (half tile per CTA, as in conv_tc).
// The three centre-column taps are issued first: the centre slot (where the raw tile lands) is
// released after a third of a chunk's MMAs, so the next-but-one raw tile is in flight early.
// An optional 1x1 "extension" over a second, un-normalised input (the block's Conv_2 shortcut)
// adds one-tap chunks that bypass the transform.  In THIS (bf16) kernel they travel through the two
// big operand sets, whose latency a one-tap chunk cannot hide, so the bf16 plan keeps shortcut blocks
// on conv_tc + an apply pass; the split-bf16 kernel below
// streams them through a ring of their own and takes them by default.
//
// Warps (640 threads): 0 = raw-tile TMA, 1 = MMA issuer (leader CTA) + TMEM allocator,
// 2 = weight TMA, 3 idle, 4..11 = epilogue (shared with conv_tc), 12..19 = transform.

#include <cuda.h>

#include <new>

#include "common.cuh"
#include "tc_common.cuh"
#include "conv_tc_common.cuh"

namespace psld {

constexpr int GN_TRANSFORM_WARPS = 8;
constexpr int GN_THREADS = (12 + GN_TRANSFORM_WARPS) * 32;   // 640 = 5 warpgroups
constexpr int GN_B_STAGES = 4;
constexpr int GN_B_BYTES = 128 * 128;            // half weight tile per CTA (<= 128 rows x 128 B)
constexpr int GN_MAX_ROWS = 192;                 // (BH+2)*W: 6x32 or 10x16
constexpr int GN_VAR_BYTES = GN_MAX_ROWS * 128;  // one operand variant (24 KB)
constexpr int GN_ABUF_BYTES = 3 * GN_VAR_BYTES;  // left | centre | right
constexpr int GN_STAGING_BYTES = 8 * 2048;     // 32-column staging groups (frees a 4th B stage)
constexpr int GN_ADDV_BYTES = 8 * 256;
// 768 B of alignment slack (the kernel traps if that is not enough); total = the 227 KB maximum
constexpr int GN_SMEM_BYTES = 2 * GN_ABUF_BYTES + GN_B_STAGES * GN_B_BYTES + GN_STAGING_BYTES + 256 + GN_ADDV_BYTES + 768;

struct ConvGnParams {
  ConvTcParams c;
  const float* affine;     // [N, Cin, 2] (scale, shift) of the GroupNorm feeding this conv
  int cin;                 // C1 + C2
  int silu;
  int rows_in;             // (BH + 2) * W
  int w_shift;             // log2(W)
  int n_images;
};

struct ConvGnState {
  CUtensorMap a1, a2, b, b2, e1, e2;     // b2: weight map with the N-slice box of the split tail units
  ConvGnParams p;
  int grid;
  bool x3;       // split-bf16 operands: conv_gn_x3_kernel
};

// tap issue order: the three centre-column taps first, so that the centre slot (where the next
// raw tile lands) is released after a third of the chunk's MMAs
__device__ __forceinline__ int gn_tap(int t9) {
  const int kx = t9 < 3 ? 1 : (t9 < 6 ? 0 : 2);
  const int ky = t9 < 3 ? t9 : (t9 < 6 ? t9 - 3 : t9 - 6);
  return ky * 3 + kx;
}

__device__ __forceinline__ float silu_fast(float x) {
  const float h = 0.5f * x;
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}

__global__ void __launch_bounds__(GN_THREADS, 1)
conv_gn_tc_kernel(const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmA2,
                  const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmB2,
                  const __grid_constant__ CUtensorMap tmE1,
                  const __grid_constant__ CUtensorMap tmE2, const ConvGnParams gp) {
  const ConvTcParams& p = gp.c;
  extern __shared__ uint8_t smem_raw[];
  pdl_launch_dependents();      // single wave of persistent CTAs (see conv_tc.cu)
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  auto abuf = [&](int b) { return base + (uint32_t)b * GN_ABUF_BYTES; };
  const uint32_t bring = base + 2 * GN_ABUF_BYTES;
  const uint32_t stg_base = bring + GN_B_STAGES * GN_B_BYTES;
  const uint32_t bar_base = stg_base + GN_STAGING_BYTES;
  const uint32_t addv_base = bar_base + 256u;
  if (addv_base + GN_ADDV_BYTES > smem_u32(smem_raw) + GN_SMEM_BYTES) __trap();
  auto raw_full = [&](int b) { return bar_base + 8u * b; };
  auto a_ready = [&](int b) { return bar_base + 8u * (2 + b); };
  auto a_empty = [&](int b) { return bar_base + 8u * (4 + b); };
  auto b_full = [&](int s) { return bar_base + 8u * (6 + s); };
  auto b_empty = [&](int s) { return bar_base + 8u * (6 + GN_B_STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (6 + 2 * GN_B_STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (8 + 2 * GN_B_STAGES + s); };
  auto c_empty = [&](int b) { return bar_base + 8u * (10 + 2 * GN_B_STAGES + b); };
  const uint32_t tmem_slot = bar_base + 8u * (12 + 2 * GN_B_STAGES);
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int unit0 = (int)(blockIdx.x >> 1), unit_step = (int)(gridDim.x >> 1);

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA1) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA2) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    if (p.ext_kchunks > 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tmE1) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&tmE2) : "memory");
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(raw_full(b), 1);
      mbar_init(a_ready(b), 2);       // one elected arrive per CTA of the pair
      mbar_init(a_empty(b), 1);
      mbar_init(c_empty(b), 1);
      mbar_init(tfull_bar(b), 1);
      mbar_init(tempty_bar(b), 16);
    }
    for (int s = 0; s < GN_B_STAGES; ++s) {
      mbar_init(b_full(s), 1);
      mbar_init(b_empty(s), 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(tmem_slot), "n"(TC_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  // (setmaxnreg re-balancing between the warpgroups was tried: ptxas lowers the budget of the
  // .dec branches but does not raise the epilogue's above the launch-bound value, so it only
  // added spills; all warps keep the launch allocation.)
  const uint32_t raw_bytes = (uint32_t)gp.rows_in * 128u;
  // K = 9 taps x normalised input chunks, then the 1x1 shortcut chunks over a second, raw input
  const int total_chunks = p.kchunks + p.ext_kchunks;

  if (warp == 0) {
    // ===================== raw activation tile producer =====================
    pdl_wait();
    if (lane == 0) {
      int buf = 0;
      uint32_t ph = 0;
      for (int v = unit0; v < p.num_virtual; v += unit_step) {
        int unit, nsub, bn;
        tc_decode_unit(p, v, unit, nsub, bn);
        const int m_tile = 2 * (unit / p.n_tiles_n) + (int)rank;
        const int n0 = m_tile / p.tiles_y;
        const int y0 = (m_tile % p.tiles_y) * p.BH - 1;
        for (int cc = 0; cc < total_chunks; ++cc) {
          mbar_wait(c_empty(buf), ph ^ 1);      // centre slot free (its 3 taps are issued first)
          mbar_arrive_expect_tx(raw_full(buf), raw_bytes);
          const CUtensorMap* tmA;
          int c0;
          if (cc < p.kchunks) {
            tmA = cc < p.kchunks1 ? &tmA1 : &tmA2;
            c0 = (cc < p.kchunks1 ? cc : cc - p.kchunks1) * TC_BLOCK_K;
          } else {                              // un-normalised shortcut input (centre tap only)
            const int e = cc - p.kchunks;
            tmA = e < p.ext_kchunks1 ? &tmE1 : &tmE2;
            c0 = (e < p.ext_kchunks1 ? e : e - p.ext_kchunks1) * TC_BLOCK_K;
          }
          tma_load_4d(abuf(buf) + GN_VAR_BYTES, tmA, raw_full(buf), c0, 0, y0, n0);  // centre slot
          if (++buf == 2) { buf = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 2) {
    // ===================== weight producer (half tile per CTA, credited to the leader) ======
    {
      int stage = 0;
      uint32_t ph = 0;
      for (int v = unit0; v < p.num_virtual; v += unit_step) {
        int unit, nsub, bn;
        tc_decode_unit(p, v, unit, nsub, bn);
        const int n_tile = unit % p.n_tiles_n;
        const int b_rows = bn >> 1;
        const CUtensorMap* tmW = nsub < 0 ? &tmB : &tmB2;
        const int bn0 = n_tile * p.block_n + (nsub < 0 ? 0 : nsub * bn) + (int)rank * b_rows;
        const uint32_t tx = (uint32_t)b_rows * 128u * 2u;
        for (int cc = 0; cc < total_chunks; ++cc) {
          const int ntap = cc < p.kchunks ? 9 : 1;
          for (int t9 = 0; t9 < ntap; ++t9) {
            const int kblk = cc < p.kchunks ? gn_tap(t9) * p.kchunks + cc : 8 * p.kchunks + cc;
            mbar_wait(b_empty(stage), ph ^ 1);
            if (elect_one()) {
              if (rank == 0) mbar_arrive_expect_tx(b_full(stage), tx);
              tma_load_2d_pair(bring + (uint32_t)stage * GN_B_BYTES, tmW, b_full(stage),
                               kblk * TC_BLOCK_K, bn0);
            }
            __syncwarp();
            if (++stage == GN_B_STAGES) { stage = 0; ph ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA) =====================
    // whole warp converged, one elected lane issues (see conv_tc.cu)
    if (rank == 0) {
      int buf = 0, stage = 0, acc = 0;
      uint32_t aph = 0, bph = 0, acc_phase = 0;
      const uint32_t row_step = (uint32_t)p.W * 128u;       // ky * W rows
      for (int v = unit0; v < p.num_virtual; v += unit_step) {
        int unit, nsub, bn;
        tc_decode_unit(p, v, unit, nsub, bn);
        mbar_wait_cluster(tempty_bar(acc), acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * 256u;
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(bn >> 3) << 17) |
                               ((uint32_t)(256 >> 4) << 24);
        for (int cc = 0; cc < total_chunks; ++cc) {
          mbar_wait_cluster(a_ready(buf), aph);
          tc_fence_after();
          const int ntap = cc < p.kchunks ? 9 : 1;     // shortcut chunks: the centre tap of the raw tile
          for (int t9 = 0; t9 < ntap; ++t9) {
            const int tap = ntap == 9 ? gn_tap(t9) : 4;
            const int ky = tap / 3, kx = tap - ky * 3;
            mbar_wait(b_full(stage), bph);
            tc_fence_after();
            // variant kx: 0 = shifted so that row (y,x) holds t(y,x-1), 1 = centre, 2 = t(y,x+1)
            const uint64_t adesc = make_sw128_desc(abuf(buf) + (uint32_t)kx * GN_VAR_BYTES +
                                                   (uint32_t)ky * row_step);
            const uint64_t bdesc = make_sw128_desc(bring + (uint32_t)stage * GN_B_BYTES);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < TC_BLOCK_K / 16; ++k)
                tc_mma_bf16_pair(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc,
                                 (cc > 0 || t9 > 0 || k > 0) ? 1u : 0u);
              tc_commit_pair(b_empty(stage));
              if (t9 == 2 || ntap == 1) tc_commit_pair(c_empty(buf));   // raw tile of chunk cc+2 may land
              if (t9 == ntap - 1) tc_commit_pair(a_empty(buf));
            }
            __syncwarp();
            if (++stage == GN_B_STAGES) { stage = 0; bph ^= 1; }
          }
          if (++buf == 2) { buf = 0; aph ^= 1; }
        }
        if (elect_one()) tc_commit_pair(tfull_bar(acc));
        __syncwarp();
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= 12) {
    // ===================== transform warps: GroupNorm + SiLU, three shifted operand tiles =====
    constexpr int TT = GN_TRANSFORM_WARPS * 32;     // transform threads
    constexpr int RSTEP = TT / 8;                   // rows covered per pass
    constexpr int ITEMS = (GN_MAX_ROWS + RSTEP - 1) / RSTEP;
    const int tt = (int)threadIdx.x - 12 * 32;      // 0..TT-1
    const int j = tt & 7;                           // 16-byte chunk = channels 8j .. 8j+7
    const int r0 = tt >> 3;                         // rows r0, r0+RSTEP, ...
    const uint32_t leader_ready0 = mapa_rank(a_ready(0), 0);
    const int Wm = p.W - 1;
    const uint32_t sm0 = smem_u32(smem_raw);
    auto sptr = [&](uint32_t a) { return reinterpret_cast<uint4*>(smem_raw + (a - sm0)); };
    int buf = 0;
    uint32_t ph = 0;
    pdl_wait();                 // the affine table comes from the GroupNorm fold just before
    for (int v = unit0; v < p.num_virtual; v += unit_step) {
        int unit, nsub, bn;
        tc_decode_unit(p, v, unit, nsub, bn);
      const int m_tile = 2 * (unit / p.n_tiles_n) + (int)rank;
      const int n0 = m_tile / p.tiles_y;
      const int y0 = (m_tile % p.tiles_y) * p.BH - 1;
      const bool img_ok = n0 < gp.n_images;
      for (int cc = 0; cc < total_chunks; ++cc) {
        if (cc >= p.kchunks) {
          // shortcut chunk: the tensor core reads the raw centre tile as it landed; only relay
          // "this CTA's tile is in place" to the leader (same barrier protocol as a transform)
          mbar_wait(raw_full(buf), ph);
          mbar_wait(a_empty(buf), ph ^ 1);
          asm volatile("bar.sync 1, %0;" ::"n"(GN_TRANSFORM_WARPS * 32) : "memory");
          if (tt == 0) mbar_arrive_remote(leader_ready0 + 8u * (uint32_t)buf);
          if (++buf == 2) { buf = 0; ph ^= 1; }
          continue;
        }
        float sc[8], sh[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) { sc[q] = 0.f; sh[q] = 0.f; }
        if (img_ok) {
          const float4* ap = reinterpret_cast<const float4*>(
              gp.affine + ((int64_t)n0 * gp.cin + cc * TC_BLOCK_K + j * 8) * 2);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 v = __ldg(ap + q);
            sc[2 * q] = v.x; sh[2 * q] = v.y; sc[2 * q + 1] = v.z; sh[2 * q + 1] = v.w;
          }
        }
        mbar_wait(raw_full(buf), ph);
        const uint32_t L = abuf(buf), Cc = L + GN_VAR_BYTES, R = Cc + GN_VAR_BYTES;
        // all of this thread's rows at once: independent load -> normalise -> store chains
        uint4 t[ITEMS];
        bool inb[ITEMS], valid[ITEMS];
#pragma unroll
        for (int u = 0; u < ITEMS; ++u) {
          const int r = r0 + RSTEP * u;
          inb[u] = r < gp.rows_in;
          const int gy = y0 + (r >> gp.w_shift);
          valid[u] = inb[u] && img_ok && gy >= 0 && gy < p.H;
          t[u] = make_uint4(0u, 0u, 0u, 0u);
          if (valid[u]) t[u] = *sptr(Cc + (uint32_t)r * 128u + (uint32_t)((j ^ (r & 7)) << 4));
        }
#pragma unroll
        for (int u = 0; u < ITEMS; ++u) {
          if (valid[u]) {
            uint32_t* ww = reinterpret_cast<uint32_t*>(&t[u]);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&ww[q]));
              float a = fmaf(f.x, sc[2 * q], sh[2 * q]);
              float b = fmaf(f.y, sc[2 * q + 1], sh[2 * q + 1]);
              if (gp.silu) { a = silu_fast(a); b = silu_fast(b); }
              __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
              ww[q] = *reinterpret_cast<uint32_t*>(&h);
            }
          }
        }
        mbar_wait(a_empty(buf), ph ^ 1);          // left / right variants no longer being read
#pragma unroll
        for (int u = 0; u < ITEMS; ++u) {
          if (!inb[u]) continue;
          const int r = r0 + RSTEP * u;
          const int x = r & Wm;
          const uint32_t off = (uint32_t)r * 128u + (uint32_t)((j ^ (r & 7)) << 4);
          *sptr(Cc + off) = t[u];                                    // centre: t(y, x)
          if (x < Wm) {                                              // left variant: (y, x+1) <- t(y, x)
            const int rn = r + 1;
            *sptr(L + (uint32_t)rn * 128u + (uint32_t)((j ^ (rn & 7)) << 4)) = t[u];
          }
          if (x == 0) *sptr(L + off) = make_uint4(0u, 0u, 0u, 0u);    // left image edge
          if (x > 0) {                                               // right variant: (y, x-1) <- t(y, x)
            const int rp = r - 1;
            *sptr(R + (uint32_t)rp * 128u + (uint32_t)((j ^ (rp & 7)) << 4)) = t[u];
          }
          if (x == Wm) *sptr(R + off) = make_uint4(0u, 0u, 0u, 0u);   // right image edge
        }
        // generic-proxy writes -> visible to the tensor core (async proxy), then tell the leader
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("bar.sync 1, %0;" ::"n"(GN_TRANSFORM_WARPS * 32) : "memory");
        if (tt == 0) mbar_arrive_remote(leader_ready0 + 8u * (uint32_t)buf);
        if (++buf == 2) { buf = 0; ph ^= 1; }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (warps 4..11), shared with conv_tc =====================
    const int quarter = warp & 3;
    const int half = (warp - 4) >> 2;
    const uint32_t leader_tempty0 = mapa_rank(tempty_bar(0), 0);
    int acc = 0;
    uint32_t acc_phase = 0;
    pdl_wait();
    for (int v = unit0; v < p.num_virtual; v += unit_step) {
        int unit, nsub, bn;
        tc_decode_unit(p, v, unit, nsub, bn);
      const int n_tile = nsub < 0 ? unit % p.n_tiles_n : (unit % p.n_tiles_n) * p.n_split + nsub;
      const int m_tile = 2 * (unit / p.n_tiles_n) + (int)rank;
      tc_epilogue_tile<true, 32, false>(
          p, tmem_base, acc, m_tile, n_tile, bn, quarter, half, lane,
          stg_base + (uint32_t)(warp - 4) * 2048u, addv_base + (uint32_t)(warp - 4) * 256u,
          [&]() {
            mbar_wait(tfull_bar(acc), acc_phase);
            tc_fence_after();
          },
          [&]() {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote_relaxed(leader_tempty0 + 8u * (uint32_t)acc);
          });
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;"
                 ::"r"(tmem_base), "n"(TC_TMEM_COLS) : "memory");
  }
}

// =====================================================================================
// Split-bf16 ("bf16x3") variant: the fp32-tolerance tier's GroupNorm-on-load convolution.
//
// Every operand tile has a hi and a lo twin, so the three column-shifted variants are SIX tiles of
// 24 KB: 144 KB, which fits shared memory once, not twice.  Instead of double-buffering the whole
// operand set, the transform runs in TWO phases around a single set, using the centre-taps-first
// issue order:
//   * the raw (hi, lo) tile of chunk c+1 lands in the CENTRE slots as soon as the three centre taps
//     of chunk c have retired (c_empty); the transform warps normalise it in place (fp32 GroupNorm
//     + SiLU, split back into hi/lo) while the tensor core is still busy with the six SIDE taps of
//     chunk c, and publish it (c_ready);
//   * the MMA warp goes straight from the side taps of chunk c to the centre taps of chunk c+1;
//     meanwhile (lr_empty) the transform warps write the left / right shifted copies from registers
//     and publish them (lr_ready) before the centre taps are through.
// A k-block = (tap, 64-channel chunk) feeds three MMA groups (a_hi w_hi, a_hi w_lo, a_lo w_hi) from
// one weight stage holding W_hi | W_lo.  Four epilogue warps (each handles both column halves; the
// tile's MMA phase is 3x longer than in the bf16 kernel, so the epilogue has time) keep the split
// staging tiles at 16 KB.
// The 1x1 shortcut extension (the block's Conv_2 over the RAW block input, accumulated into the same
// tile as extra centre-tap k-blocks) follows the 9-tap chunks of a tile: its tiles need no halo and no
// transform, so they stream through a 3-deep ring of 32 KB (hi | lo) slots carved out of the left /
// right variant region (idle by then), loaded by their own producer warp with 2-CTA TMA (credited to
// the leader's barrier, as in conv_tc); the centre slots stay free, so the next tile's first raw tile
// lands and is normalised while the shortcut k-blocks run.
//
// Warps (384 threads, so that the split epilogue keeps its accumulator rows in registers: 170 regs):
// 0 = raw-tile TMA, 1 = MMA issuer (leader CTA) + TMEM allocator, 2 = weight TMA, 3 = shortcut-tile
// TMA, 4..7 = epilogue, 8..11 = transform.
constexpr int GX_THREADS = 384;
constexpr int GX_TRANSFORM_WARPS = 4;
constexpr int GX_B_STAGES = 2;
constexpr int GX_B_STAGE = 2 * GN_B_BYTES;          // W_hi | W_lo half tiles (32 KB)
constexpr int GX_ABUF_BYTES = 6 * GN_VAR_BYTES;     // C_hi C_lo L_hi L_lo R_hi R_lo
constexpr int GX_STAGING_BYTES = 4 * 4096;          // 4 epilogue warps x (hi, lo) 2 KB tiles
constexpr int GX_ADDV_BYTES = 4 * 256;
constexpr int GX_SMEM_BYTES = GX_ABUF_BYTES + GX_B_STAGES * GX_B_STAGE + GX_STAGING_BYTES + 256 + GX_ADDV_BYTES + 768;

__device__ __forceinline__ float silu_x3(float x) { return __fdividef(x, 1.0f + __expf(-x)); }

__global__ void __launch_bounds__(GX_THREADS, 1)
conv_gn_x3_kernel(const __grid_constant__ CUtensorMap tmA1, const __grid_constant__ CUtensorMap tmA2,
                  const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmB2,
                  const __grid_constant__ CUtensorMap tmE1, const __grid_constant__ CUtensorMap tmE2,
                  const ConvGnParams gp) {
  const ConvTcParams& p = gp.c;
  extern __shared__ uint8_t smem_raw[];
  pdl_launch_dependents();
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  // variant v in {0: centre, 1: left, 2: right}, plane pl in {0: hi, 1: lo}
  auto var = [&](int v, int pl) { return base + (uint32_t)(2 * v + pl) * GN_VAR_BYTES; };
  // shortcut ring: 3 slots of (hi 16 KB | lo 16 KB) over the left / right variant region (96 KB)
  auto ext_slot = [&](int k) { return base + 2u * GN_VAR_BYTES + (uint32_t)k * 32768u; };
  const uint32_t bring = base + GX_ABUF_BYTES;
  const uint32_t stg_base = bring + GX_B_STAGES * GX_B_STAGE;
  const uint32_t bar_base = stg_base + GX_STAGING_BYTES;
  const uint32_t addv_base = bar_base + 256u;
  if (addv_base + GX_ADDV_BYTES > smem_u32(smem_raw) + GX_SMEM_BYTES) __trap();
  const uint32_t raw_full = bar_base, c_ready = bar_base + 8u, lr_ready = bar_base + 16u;
  const uint32_t c_empty = bar_base + 24u, lr_empty = bar_base + 32u;
  auto b_full = [&](int s) { return bar_base + 40u + 8u * s; };
  auto b_empty = [&](int s) { return bar_base + 40u + 8u * (GX_B_STAGES + s); };
  auto tfull_bar = [&](int s) { return bar_base + 40u + 8u * (2 * GX_B_STAGES + s); };
  auto tempty_bar = [&](int s) { return bar_base + 40u + 8u * (2 * GX_B_STAGES + 2 + s); };
  const uint32_t tmem_slot = bar_base + 40u + 8u * (2 * GX_B_STAGES + 4);
  auto ext_full = [&](int k) { return tmem_slot + 8u + 8u * k; };
  auto ext_empty = [&](int k) { return tmem_slot + 32u + 8u * k; };
  const uint32_t ext_done = tmem_slot + 56u;
  volatile uint32_t* tmem_slot_ptr =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int unit0 = (int)(blockIdx.x >> 1), unit_step = (int)(gridDim.x >> 1);

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA1) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA2) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    mbar_init(raw_full, 1);
    mbar_init(c_ready, 2);          // one elected arrive per CTA of the pair
    mbar_init(lr_ready, 2);
    mbar_init(c_empty, 1);
    mbar_init(lr_empty, 1);
    for (int k = 0; k < 3; ++k) {
      mbar_init(ext_full(k), 1);
      mbar_init(ext_empty(k), 1);
    }
    mbar_init(ext_done, 1);
    for (int s = 0; s < GX_B_STAGES; ++s) {
      mbar_init(b_full(s), 1);
      mbar_init(b_empty(s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(tfull_bar(b), 1);
      mbar_init(tempty_bar(b), 8);  // 4 epilogue warps x 2 CTAs
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                 ::"r"(tmem_slot), "n"(TC_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  const uint32_t raw_bytes = (uint32_t)gp.rows_in * 128u;
  const int total_chunks = p.kchunks;

  if (warp == 0) {
    // ===================== raw activation tiles (hi, lo) -> the centre slots =====================
    pdl_wait();
    if (lane == 0) {
      uint32_t ph = 0;
      for (int v = unit0; v < p.num_virtual; v += unit_step) {
        int unit, nsub, bn;
        tc_decode_unit(p, v, unit, nsub, bn);
        const int m_tile = 2 * (unit / p.n_tiles_n) + (int)rank;
        const int n0 = m_tile / p.tiles_y;
        const int y0 = (m_tile % p.tiles_y) * p.BH - 1;
        for (int cc = 0; cc < total_chunks; ++cc) {
          mbar_wait(c_empty, ph ^ 1);             // centre taps of the previous chunk have retired
          mbar_arrive_expect_tx(raw_full, 2u * raw_bytes);
          const bool s1 = cc < p.kchunks1;
          const CUtensorMap* tmA = s1 ? &tmA1 : &tmA2;
          const int c0 = (s1 ? cc : cc - p.kchunks1) * TC_BLOCK_K;
          tma_load_4d(var(0, 0), tmA, raw_full, c0, 0, y0, n0);
          tma_load_4d(var(0, 1), tmA, raw_full, c0 + (s1 ? p.lo1 : p.lo2), 0, y0, n0);
          ph ^= 1;
        }
      }
    }
  } else if (warp == 2) {
    // ===================== weight producer: W_hi | W_lo half tiles per (tap, chunk) =============
    int stage = 0;
    uint32_t ph = 0;
    for (int v = unit0; v < p.num_virtual; v += unit_step) {
        int unit, nsub, bn;
        tc_decode_unit(p, v, unit, nsub, bn);
      const int n_tile = unit % p.n_tiles_n;
      const int b_rows = bn >> 1;
      const CUtensorMap* tmW = nsub < 0 ? &tmB : &tmB2;
      const int bn0 = n_tile * p.block_n + (nsub < 0 ? 0 : nsub * bn) + (int)rank * b_rows;
      const uint32_t tx = (uint32_t)b_rows * 128u * 2u * 2u;       // (hi + lo) x both CTAs
      for (int cc = 0; cc < total_chunks + p.ext_kchunks; ++cc) {
        const int ntap = cc < total_chunks ? 9 : 1;
        for (int t9 = 0; t9 < ntap; ++t9) {
          const int kblk = ntap == 9 ? gn_tap(t9) * p.kchunks + cc : 8 * p.kchunks + cc;
          mbar_wait(b_empty(stage), ph ^ 1);
          if (elect_one()) {
            if (rank == 0) mbar_arrive_expect_tx(b_full(stage), tx);
            const uint32_t dst = bring + (uint32_t)stage * GX_B_STAGE;
            tma_load_2d_pair(dst, tmW, b_full(stage), kblk * TC_BLOCK_K, bn0);
            tma_load_2d_pair(dst + GN_B_BYTES, tmW, b_full(stage), kblk * TC_BLOCK_K, bn0 + p.w_lo_rows);
          }
          __syncwarp();
          if (++stage == GX_B_STAGES) { stage = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 3) {
    // ===================== shortcut tiles (raw hi, lo; no halo, no transform) =====================
    if (p.ext_kchunks > 0) {
      pdl_wait();
      int eslot = 0;
      uint32_t eph = 0, lph = 0;
      for (int v = unit0; v < p.num_virtual; v += unit_step) {
        int unit, nsub, bn;
        tc_decode_unit(p, v, unit, nsub, bn);
        const int m_tile = 2 * (unit / p.n_tiles_n) + (int)rank;
        const int n0 = m_tile / p.tiles_y;
        const int y0 = (m_tile % p.tiles_y) * p.BH;
        // the ring lives in the left / right variant region: wait until the side taps of EVERY 9-tap
        // chunk of this tile have retired (every lr_empty phase must be observed, in order)
        for (int cc = 0; cc < total_chunks; ++cc) { mbar_wait(lr_empty, lph); lph ^= 1; }
        for (int e = 0; e < p.ext_kchunks; ++e) {
          mbar_wait(ext_empty(eslot), eph ^ 1);
          if (elect_one()) {
            if (rank == 0) mbar_arrive_expect_tx(ext_full(eslot), 4u * TC_A_BYTES);   // (hi + lo) x both CTAs
            const bool s1 = e < p.ext_kchunks1;
            const CUtensorMap* tmE = s1 ? &tmE1 : &tmE2;
            const int c0 = (s1 ? e : e - p.ext_kchunks1) * TC_BLOCK_K;
            tma_load_4d_pair(ext_slot(eslot), tmE, ext_full(eslot), c0, 0, y0, n0);
            tma_load_4d_pair(ext_slot(eslot) + 16384u, tmE, ext_full(eslot), c0 + (s1 ? p.loe1 : p.loe2), 0, y0, n0);
          }
          __syncwarp();
          if (++eslot == 3) { eslot = 0; eph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA) =====================
    if (rank == 0) {
      int stage = 0, acc = 0, eslot = 0;
      uint32_t cph = 0, bph = 0, acc_phase = 0, eph = 0;
      const uint32_t row_step = (uint32_t)p.W * 128u;       // ky * W rows
      for (int v = unit0; v < p.num_virtual; v += unit_step) {
        int unit, nsub, bn;
        tc_decode_unit(p, v, unit, nsub, bn);
        mbar_wait_cluster(tempty_bar(acc), acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * 256u;
        const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(bn >> 3) << 17) |
                               ((uint32_t)(256 >> 4) << 24);
        for (int cc = 0; cc < total_chunks; ++cc) {
          for (int t9 = 0; t9 < 9; ++t9) {
            if (t9 == 0) { mbar_wait_cluster(c_ready, cph); tc_fence_after(); }
            if (t9 == 3) {
              // side variants written (the transform warps are done READING the centre tiles too):
              // once the three centre taps issued so far retire, the next raw tile may land
              mbar_wait_cluster(lr_ready, cph);
              tc_fence_after();
              if (elect_one()) tc_commit_pair(c_empty);
              __syncwarp();
            }
            const int tap = gn_tap(t9);
            const int ky = tap / 3, kx = tap - ky * 3;
            const int v = kx == 1 ? 0 : (kx == 0 ? 1 : 2);   // centre / left / right variant
            mbar_wait(b_full(stage), bph);
            tc_fence_after();
            const uint64_t a_hi = make_sw128_desc(var(v, 0) + (uint32_t)ky * row_step);
            const uint64_t a_lo = make_sw128_desc(var(v, 1) + (uint32_t)ky * row_step);
            const uint64_t b_hi = make_sw128_desc(bring + (uint32_t)stage * GX_B_STAGE);
            const uint64_t b_lo = make_sw128_desc(bring + (uint32_t)stage * GX_B_STAGE + GN_B_BYTES);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < TC_BLOCK_K / 16; ++k)
                tc_mma_bf16_pair(d_tmem, a_hi + (uint64_t)(2 * k), b_hi + (uint64_t)(2 * k), idesc,
                                 (cc > 0 || t9 > 0 || k > 0) ? 1u : 0u);
#pragma unroll
              for (int k = 0; k < TC_BLOCK_K / 16; ++k)
                tc_mma_bf16_pair(d_tmem, a_hi + (uint64_t)(2 * k), b_lo + (uint64_t)(2 * k), idesc, 1u);
#pragma unroll
              for (int k = 0; k < TC_BLOCK_K / 16; ++k)
                tc_mma_bf16_pair(d_tmem, a_lo + (uint64_t)(2 * k), b_hi + (uint64_t)(2 * k), idesc, 1u);
              tc_commit_pair(b_empty(stage));
              if (t9 == 8) tc_commit_pair(lr_empty);     // side variants free
            }
            __syncwarp();
            if (++stage == GX_B_STAGES) { stage = 0; bph ^= 1; }
          }
          cph ^= 1;
        }
        // 1x1 shortcut k-blocks: raw (hi, lo) tiles of the block input from the 3-slot ring
        for (int e = 0; e < p.ext_kchunks; ++e) {
          mbar_wait(ext_full(eslot), eph);
          mbar_wait(b_full(stage), bph);
          tc_fence_after();
          const uint64_t a_hi = make_sw128_desc(ext_slot(eslot));
          const uint64_t a_lo = make_sw128_desc(ext_slot(eslot) + 16384u);
          const uint64_t b_hi = make_sw128_desc(bring + (uint32_t)stage * GX_B_STAGE);
          const uint64_t b_lo = make_sw128_desc(bring + (uint32_t)stage * GX_B_STAGE + GN_B_BYTES);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < TC_BLOCK_K / 16; ++k)
              tc_mma_bf16_pair(d_tmem, a_hi + (uint64_t)(2 * k), b_hi + (uint64_t)(2 * k), idesc, 1u);
#pragma unroll
            for (int k = 0; k < TC_BLOCK_K / 16; ++k)
              tc_mma_bf16_pair(d_tmem, a_hi + (uint64_t)(2 * k), b_lo + (uint64_t)(2 * k), idesc, 1u);
#pragma unroll
            for (int k = 0; k < TC_BLOCK_K / 16; ++k)
              tc_mma_bf16_pair(d_tmem, a_lo + (uint64_t)(2 * k), b_hi + (uint64_t)(2 * k), idesc, 1u);
            tc_commit_pair(b_empty(stage));
            tc_commit_pair(ext_empty(eslot));
            if (e == p.ext_kchunks - 1) tc_commit_pair(ext_done);   // left / right region free again
          }
          __syncwarp();
          if (++stage == GX_B_STAGES) { stage = 0; bph ^= 1; }
          if (++eslot == 3) { eslot = 0; eph ^= 1; }
        }
        if (elect_one()) tc_commit_pair(tfull_bar(acc));
        __syncwarp();
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= 8) {
    // ===================== transform warps: fp32 GroupNorm + SiLU, two phases =====================
    constexpr int TT = GX_TRANSFORM_WARPS * 32;
    constexpr int RSTEP = TT / 8;
    constexpr int ITEMS = (GN_MAX_ROWS + RSTEP - 1) / RSTEP;
    const int tt = (int)threadIdx.x - 8 * 32;
    const int j = tt & 7;                           // 16-byte chunk = channels 8j .. 8j+7
    const int r0 = tt >> 3;
    const uint32_t leader_c = mapa_rank(c_ready, 0), leader_lr = mapa_rank(lr_ready, 0);
    const int Wm = p.W - 1;
    const uint32_t sm0 = smem_u32(smem_raw);
    auto sptr = [&](uint32_t a) { return reinterpret_cast<uint4*>(smem_raw + (a - sm0)); };
    uint32_t ph = 0, tph = 0;
    pdl_wait();
    for (int v = unit0; v < p.num_virtual; v += unit_step) {
        int unit, nsub, bn;
        tc_decode_unit(p, v, unit, nsub, bn);
      const int m_tile = 2 * (unit / p.n_tiles_n) + (int)rank;
      const int n0 = m_tile / p.tiles_y;
      const int y0 = (m_tile % p.tiles_y) * p.BH - 1;
      const bool img_ok = n0 < gp.n_images;
      for (int cc = 0; cc < total_chunks; ++cc) {
        float sc[8], sh[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) { sc[q] = 0.f; sh[q] = 0.f; }
        if (img_ok) {
          const float4* ap = reinterpret_cast<const float4*>(
              gp.affine + ((int64_t)n0 * gp.cin + cc * TC_BLOCK_K + j * 8) * 2);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float4 v = __ldg(ap + q);
            sc[2 * q] = v.x; sh[2 * q] = v.y; sc[2 * q + 1] = v.z; sh[2 * q + 1] = v.w;
          }
        }
        mbar_wait(raw_full, ph);
        const uint32_t Ch = var(0, 0), Cl = var(0, 1);
        // ---- phase 1: normalise the centre tiles in place (three rows in flight per thread)
#pragma unroll 3
        for (int u = 0; u < ITEMS; ++u) {
          const int r = r0 + RSTEP * u;
          if (r >= gp.rows_in) continue;
          const int gy = y0 + (r >> gp.w_shift);
          const bool valid = img_ok && gy >= 0 && gy < p.H;
          const uint32_t off = (uint32_t)r * 128u + (uint32_t)((j ^ (r & 7)) << 4);
          uint4 th = make_uint4(0u, 0u, 0u, 0u), tl = th;     // rows outside the image: zero padding
          if (valid) {
            th = *sptr(Ch + off);
            tl = *sptr(Cl + off);
            uint32_t* wh = reinterpret_cast<uint32_t*>(&th);
            uint32_t* wl = reinterpret_cast<uint32_t*>(&tl);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float2 fh = bf2_to_f2(wh[q]), fl = bf2_to_f2(wl[q]);
              float a = fmaf(fh.x + fl.x, sc[2 * q], sh[2 * q]);
              float b = fmaf(fh.y + fl.y, sc[2 * q + 1], sh[2 * q + 1]);
              if (gp.silu) { a = silu_x3(a); b = silu_x3(b); }
              split_bf2(a, b, wh[q], wl[q]);
            }
          }
          *sptr(Ch + off) = th;
          *sptr(Cl + off) = tl;
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("bar.sync 1, %0;" ::"n"(GX_TRANSFORM_WARPS * 32) : "memory");
        if (tt == 0) mbar_arrive_remote(leader_c);
        // ---- phase 2: left / right shifted copies of the normalised centre tiles, once the side taps
        // of the previous chunk have retired (the centre tiles stay put until lr_ready: see the MMA warp)
        mbar_wait(lr_empty, ph ^ 1);
        if (cc == 0 && p.ext_kchunks > 0) { mbar_wait(ext_done, tph ^ 1); tph ^= 1; }   // previous tile's shortcut ring
#pragma unroll 3
        for (int u = 0; u < ITEMS; ++u) {
          const int r = r0 + RSTEP * u;
          if (r >= gp.rows_in) continue;
          const int x = r & Wm;
          const uint32_t off = (uint32_t)r * 128u + (uint32_t)((j ^ (r & 7)) << 4);
          const uint4 th = *sptr(Ch + off), tl = *sptr(Cl + off);
          const uint4 z = make_uint4(0u, 0u, 0u, 0u);
          if (x < Wm) {                                              // left variant: (y, x+1) <- t(y, x)
            const int rn = r + 1;
            const uint32_t o2 = (uint32_t)rn * 128u + (uint32_t)((j ^ (rn & 7)) << 4);
            *sptr(var(1, 0) + o2) = th;
            *sptr(var(1, 1) + o2) = tl;
          }
          if (x == 0) { *sptr(var(1, 0) + off) = z; *sptr(var(1, 1) + off) = z; }     // left image edge
          if (x > 0) {                                               // right variant: (y, x-1) <- t(y, x)
            const int rp = r - 1;
            const uint32_t o2 = (uint32_t)rp * 128u + (uint32_t)((j ^ (rp & 7)) << 4);
            *sptr(var(2, 0) + o2) = th;
            *sptr(var(2, 1) + o2) = tl;
          }
          if (x == Wm) { *sptr(var(2, 0) + off) = z; *sptr(var(2, 1) + off) = z; }    // right image edge
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("bar.sync 1, %0;" ::"n"(GX_TRANSFORM_WARPS * 32) : "memory");
        if (tt == 0) mbar_arrive_remote(leader_lr);
        ph ^= 1;
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (warps 4..7): both column halves per warp =====================
    const int quarter = warp & 3;
    const uint32_t leader_tempty0 = mapa_rank(tempty_bar(0), 0);
    int acc = 0;
    uint32_t acc_phase = 0;
    pdl_wait();
    for (int v = unit0; v < p.num_virtual; v += unit_step) {
        int unit, nsub, bn;
        tc_decode_unit(p, v, unit, nsub, bn);
      const int n_tile = nsub < 0 ? unit % p.n_tiles_n : (unit % p.n_tiles_n) * p.n_split + nsub;
      const int m_tile = 2 * (unit / p.n_tiles_n) + (int)rank;
      const uint32_t stg = stg_base + (uint32_t)(warp - 4) * 4096u;
      const uint32_t addv = addv_base + (uint32_t)(warp - 4) * 256u;
      tc_epilogue_tile<false, 32, false, true>(
          p, tmem_base, acc, m_tile, n_tile, bn, quarter, 0, lane, stg, addv,
          [&]() {
            mbar_wait(tfull_bar(acc), acc_phase);
            tc_fence_after();
          },
          []() {});
      tc_epilogue_tile<false, 32, false, true>(
          p, tmem_base, acc, m_tile, n_tile, bn, quarter, 1, lane, stg, addv, []() {},
          [&]() {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote_relaxed(leader_tempty0 + 8u * (uint32_t)acc);
          });
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;"
                 ::"r"(tmem_base), "n"(TC_TMEM_COLS) : "memory");
  }
}

// ---------------------------------------------------------------- host side
static int encode_raw_map(CUtensorMap* tm, const void* ptr, int N, int H, int W, int C, int rows_y) {
  const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  const cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  const cuuint32_t box[4] = {(cuuint32_t)TC_BLOCK_K, (cuuint32_t)W, (cuuint32_t)rows_y, 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  return encode_bf16_map(tm, ptr, 4, dims, strides, box, estr, "raw tile");
}

// Returns PSLD_EUNSUPPORTED when the shape must take the unfused route (GroupNorm apply + conv_tc).
int prepare_conv_gn_tc(psld_op& op) {
  const int N = op.i[PSLD_CONV_N], H = op.i[PSLD_CONV_H], W = op.i[PSLD_CONV_W];
  const int C1 = op.i[PSLD_CONV_C1], C2 = op.i[PSLD_CONV_C2], Cout = op.i[PSLD_CONV_COUT];
  const int KS = op.i[PSLD_CONV_KS];
  auto unsupported = [&](const char* why) {
    set_error("conv_gn_tc: not eligible (%s): N=%d H=%d W=%d C1=%d C2=%d Cout=%d KS=%d", why, N, H,
              W, C1, C2, Cout, KS);
    return PSLD_EUNSUPPORTED;
  };
  // network head (ncsnpp.py:430): fp32 NCHW output, first f[1] channels of a zero-padded Cout
  const bool head = op.i[PSLD_CONV_OUT_LAYOUT] == PSLD_NCHW && op.i[PSLD_CONV_OUT_DTYPE] == PSLD_F32;
  const int adt = op.i[PSLD_CONV_IN_DTYPE];
  if ((adt != PSLD_BF16 && adt != PSLD_BF16S) || (!head && op.i[PSLD_CONV_OUT_DTYPE] != adt))
    return unsupported("bf16 or split-bf16 in/out only");
  const bool x3 = adt == PSLD_BF16S;
  const int cm = x3 ? 2 : 1;
  if (op.i[PSLD_CONV_IN_LAYOUT] != PSLD_NHWC || (!head && op.i[PSLD_CONV_OUT_LAYOUT] != PSLD_NHWC))
    return unsupported("NHWC only");
  if (head && op.out[1]) return unsupported("head: no statistics");
  if (head && op.in[2] && op.i[PSLD_CONV_RES_DTYPE] != PSLD_F32)
    return unsupported("head residual must be fp32 NCHW");
  if (KS != 3 || op.i[PSLD_CONV_STRIDE] != 1 || op.i[PSLD_CONV_PAD] != 1) return unsupported("3x3 s1 p1 only");
  if (C1 % TC_BLOCK_K || C2 % TC_BLOCK_K) return unsupported("Cin %% 64 != 0");
  if (Cout % 64 || Cout > 256 && Cout % 256) return unsupported("Cout");
  if (!((W == 32 && H >= 4) || (W == 16 && H >= 8)) || (H & (H - 1))) return unsupported("map must be 16x16+ / 32x32+ wide tiles");
  if (!head && op.in[2] && op.i[PSLD_CONV_RES_DTYPE] != adt) return unsupported("residual dtype");
  if (!op.in[0] || !op.in[4] || !op.in[6] || !op.out[0] || (C2 > 0 && !op.in[1])) {
    set_error("conv_gn_tc: null pointer");
    return PSLD_EINVAL;
  }
  int block_n = 0;
  for (int cand : {256, 128, 64})
    if (Cout % cand == 0) { block_n = cand; break; }
  const int BH = 128 / W;
  const int rows_in = (BH + 2) * W;
  if (rows_in > GN_MAX_ROWS) return unsupported("tile rows");
  const int64_t m_tiles = (int64_t)N * (H / BH);
  if (m_tiles < 2) return unsupported("single tile");
  ConvGnState* st = new (std::nothrow) ConvGnState();
  if (!st) { set_error("conv_gn_tc: out of host memory"); return PSLD_ECUDA; }
  st->x3 = x3;
  int rc = encode_raw_map(&st->a1, op.in[0], N, H, W, cm * C1, BH + 2);
  if (rc == PSLD_OK)
    rc = C2 > 0 ? encode_raw_map(&st->a2, op.in[1], N, H, W, cm * C2, BH + 2)
                : encode_raw_map(&st->a2, op.in[0], N, H, W, cm * C1, BH + 2);
  // optional 1x1 shortcut over a second, un-normalised input cat(e1, e2): extra K-blocks
  const int E1 = op.i[PSLD_CONV_EXT_C1], E2 = op.i[PSLD_CONV_EXT_C2];
  const bool ext = op.in[8] != nullptr && E1 > 0;
  if (ext && (E1 % TC_BLOCK_K || E2 % TC_BLOCK_K || (E2 > 0 && !op.in[9]))) {
    delete st;
    return unsupported("shortcut extension needs E %% 64 == 0");
  }
  if (rc == PSLD_OK)
    // split-bf16 kernel: the shortcut tile is the tile's own BH rows (no halo), [hi | lo] channels
    rc = ext ? encode_raw_map(&st->e1, op.in[8], N, H, W, cm * E1, x3 ? BH : BH + 2)
             : encode_raw_map(&st->e1, op.in[0], N, H, W, cm * C1, BH + 2);
  if (rc == PSLD_OK)
    rc = (ext && E2 > 0) ? encode_raw_map(&st->e2, op.in[9], N, H, W, cm * E2, x3 ? BH : BH + 2)
                         : encode_raw_map(&st->e2, op.in[0], N, H, W, cm * C1, BH + 2);
  const int K = 9 * (C1 + C2) + (ext ? E1 + E2 : 0);
  // split bf16: weight planes [2][Cout, K] seen as one [2*Cout, K] matrix
  if (rc == PSLD_OK) rc = encode_w_map(&st->b, op.in[4], cm * Cout, K, block_n / 2);
  if (rc != PSLD_OK) { delete st; return rc; }
  ConvGnParams& g = st->p;
  ConvTcParams& p = g.c;
  tc_conv_params(p, op, head, H, W, BH, 1, block_n);
  p.num_tiles = (int)(((m_tiles + 1) / 2) * p.n_tiles_n);
  g.affine = (const float*)op.in[6];
  g.cin = C1 + C2;
  g.silu = op.i[PSLD_CONV_GN_SILU];
  g.rows_in = rows_in;
  g.w_shift = W == 32 ? 5 : 4;
  g.n_images = N;
  const int pairs = sm_count() / 2;
  st->b2 = st->b;
  const int ns = tc_plan_tail_split(p, pairs, 64, !head);
  if (ns > 1) {
    rc = encode_w_map(&st->b2, op.in[4], cm * Cout, K, block_n / ns / 2);
    if (rc != PSLD_OK) { delete st; return rc; }
  }
  st->grid = 2 * (p.num_virtual < pairs ? p.num_virtual : pairs);
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_gn_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         GN_SMEM_BYTES);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(conv_gn_x3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GX_SMEM_BYTES);
    if (e != cudaSuccess) {
      set_error("conv_gn_tc: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
      delete st;
      return PSLD_ECUDA;
    }
    attr_set = true;
  }
  op.aux = st;
  return PSLD_OK;
}

int release_conv_gn_tc(psld_op& op) {
  if (op.aux) {
    delete (ConvGnState*)op.aux;
    op.aux = nullptr;
  }
  return PSLD_OK;
}

int run_conv_gn_tc(const psld_op& op, cudaStream_t s) {
  const ConvGnState* st = (const ConvGnState*)op.aux;
  PSLD_CHECK_ARG(st != nullptr, "conv_gn_tc: op not prepared (call psld_op_prepare)");
  if (st->x3)
    PSLD_CHECK_CUDA(launch_pdl(conv_gn_x3_kernel, dim3((unsigned)st->grid), dim3(GX_THREADS), GX_SMEM_BYTES,
                               s, 2, st->a1, st->a2, st->b, st->b2, st->e1, st->e2, st->p));
  else
    PSLD_CHECK_CUDA(launch_pdl(conv_gn_tc_kernel, dim3((unsigned)st->grid), dim3(GN_THREADS), GN_SMEM_BYTES,
                               s, 2, st->a1, st->a2, st->b, st->b2, st->e1, st->e2, st->p));
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}

}  // namespace psld
