// CUDA-core (fp32 FFMA) implicit-GEMM convolution and attention core.
//
// This is the reference-faithful fp32 path (true fp32 products and accumulation, like the
// reference's CPU ATen conv/einsum) and the engine for shapes the tensor-core kernel does
// not take (Cin = 6 input conv, Cout = 6 output conv, stride-2 pyramid conv, tiny nets).
//
// Reference lines: ddpm_conv3x3 / ddpm_conv1x1 layers.py:85-109; NIN layers.py:531-540;
// conv_downsample_2d's F.conv2d(stride=2) up_or_down_sampling.py:178; epilogue terms
// (+Dense_0(temb), +shortcut, /sqrt(2)) layerspp.py:262-274,88-91, ncsnpp.py:353-356;
// attention layerspp.py:82-86.

#include "common.cuh"

namespace psld {

struct ConvP {
  const void* x1; const void* x2; const void* res; const float* temb;
  const float* w; const float* bias; void* y;
  int N, H, W, C1, C2, Cout, KS, stride, pad, OH, OW;
  int in_layout, out_layout, temb_off, temb_bstride;
  float scale;
};

constexpr int BM = 64, BN = 64, BK = 16;

template <typename TI>
__device__ __forceinline__ float load_in(const ConvP& p, int n, int iy, int ix, int c) {
  if (p.in_layout == PSLD_NCHW) {  // fp32 NCHW network input (C2 == 0)
    return ((const float*)p.x1)[(((int64_t)n * p.C1 + c) * p.H + iy) * p.W + ix];
  }
  const int64_t pix = ((int64_t)n * p.H + iy) * p.W + ix;
  constexpr int M = Elt<TI>::kMul;
  if (c < p.C1) return ld_elt<TI>((const TI*)p.x1 + pix * (p.C1 * M) + c, p.C1);
  return ld_elt<TI>((const TI*)p.x2 + pix * (p.C2 * M) + (c - p.C1), p.C2);
}

template <typename TI, typename TO>
__global__ void __launch_bounds__(256)
conv_simt_kernel(const ConvP p) {
  pdl_wait();
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Bs[BK][BN + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int64_t M = (int64_t)p.N * p.OH * p.OW;
  const int64_t m0 = (int64_t)blockIdx.x * BM;
  const int n0 = blockIdx.y * BN;
  const int Cin = p.C1 + p.C2;
  const int K = p.KS * p.KS * Cin;

  // A-load assignment: this thread loads k = tid % 16 for pixels (tid/16) + 16*j
  const int ak = tid & 15;
  int an[4], aoy[4], aox[4];
  bool av[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int64_t m = m0 + (tid >> 4) + 16 * j;
    av[j] = m < M;
    const int64_t mm = av[j] ? m : 0;
    aox[j] = (int)(mm % p.OW);
    const int64_t r = mm / p.OW;
    aoy[j] = (int)(r % p.OH);
    an[j] = (int)(r / p.OH);
  }
  // B-load assignment: column tid % 64, rows tid/64 + 4*j
  const int bn = tid & 63, bk = tid >> 6;

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < K; k0 += BK) {
    {
      const int kk = k0 + ak;
      const bool kv = kk < K;
      const int tap = kv ? kk / Cin : 0;
      const int c = kk - tap * Cin;
      const int ky = tap / p.KS, kx = tap - ky * p.KS;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float v = 0.f;
        if (kv && av[j]) {
          const int iy = aoy[j] * p.stride - p.pad + ky;
          const int ix = aox[j] * p.stride - p.pad + kx;
          if (iy >= 0 && iy < p.H && ix >= 0 && ix < p.W) v = load_in<TI>(p, an[j], iy, ix, c);
        }
        As[ak][(tid >> 4) + 16 * j] = v;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int kr = bk + 4 * j;
        const int kk2 = k0 + kr;
        float v = 0.f;
        if (kk2 < K && n0 + bn < p.Cout) v = p.w[(int64_t)kk2 * p.Cout + n0 + bn];
        Bs[kr][bn] = v;
      }
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float av4[4] = {a.x, a.y, a.z, a.w}, bv4[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av4[i], bv4[j], acc[i][j]);
    }
    __syncthreads();
  }

  // epilogue: y = scale * (acc + bias + temb[n] + residual)
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t m = m0 + ty * 4 + i;
    if (m >= M) continue;
    const int ox = (int)(m % p.OW);
    const int64_t r = m / p.OW;
    const int oy = (int)(r % p.OH);
    const int n = (int)(r / p.OH);
    float o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int co = n0 + tx * 4 + j;
      float v = acc[i][j];
      if (co < p.Cout) {
        if (p.bias) v += p.bias[co];
        if (p.temb) v += p.temb[(int64_t)n * p.temb_bstride + p.temb_off + co];
        if (p.res) {
          if (p.out_layout == PSLD_NCHW)     // fp32 NCHW residual of the NCHW head
            v += ((const float*)p.res)[(((int64_t)n * p.Cout + co) * p.OH + oy) * p.OW + ox];
          else
            v += ld_elt<TO>((const TO*)p.res + m * (p.Cout * Elt<TO>::kMul) + co, p.Cout);
        }
        v *= p.scale;
      }
      o[j] = v;
    }
    const int co0 = n0 + tx * 4;
    if (p.out_layout == PSLD_NCHW) {
      float* y = (float*)p.y;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (co0 + j < p.Cout) y[(((int64_t)n * p.Cout + co0 + j) * p.OH + oy) * p.OW + ox] = o[j];
    } else {
      TO* y = (TO*)p.y + m * (p.Cout * Elt<TO>::kMul) + co0;
      if ((p.Cout & 3) == 0 && co0 + 3 < p.Cout) {
        Vec4<TO>::store(y, make_float4(o[0], o[1], o[2], o[3]), p.Cout);
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (co0 + j < p.Cout) st_elt<TO>(y + j, o[j], p.Cout);
      }
    }
  }
}

int run_conv_simt(const psld_op& op, cudaStream_t s) {
  ConvP p;
  p.x1 = op.in[0]; p.x2 = op.in[1]; p.res = op.in[2]; p.temb = (const float*)op.in[3];
  p.w = (const float*)op.in[4]; p.bias = (const float*)op.in[5]; p.y = op.out[0];
  p.N = op.i[PSLD_CONV_N]; p.H = op.i[PSLD_CONV_H]; p.W = op.i[PSLD_CONV_W];
  p.C1 = op.i[PSLD_CONV_C1]; p.C2 = op.i[PSLD_CONV_C2]; p.Cout = op.i[PSLD_CONV_COUT];
  p.KS = op.i[PSLD_CONV_KS]; p.stride = op.i[PSLD_CONV_STRIDE]; p.pad = op.i[PSLD_CONV_PAD];
  p.OH = op.i[PSLD_CONV_OH]; p.OW = op.i[PSLD_CONV_OW];
  p.in_layout = op.i[PSLD_CONV_IN_LAYOUT]; p.out_layout = op.i[PSLD_CONV_OUT_LAYOUT];
  p.temb_off = op.i[PSLD_CONV_TEMB_OFF]; p.temb_bstride = op.i[PSLD_CONV_TEMB_BSTRIDE];
  p.scale = op.f[0];
  const int idt = op.i[PSLD_CONV_IN_DTYPE], odt = op.i[PSLD_CONV_OUT_DTYPE];
  PSLD_CHECK_ARG(p.x1 && p.w && p.y, "conv: null pointer");
  PSLD_CHECK_ARG(p.N > 0 && p.H > 0 && p.W > 0 && p.C1 > 0 && p.C2 >= 0 && p.Cout > 0,
                 "conv: bad sizes");
  PSLD_CHECK_ARG(p.C2 == 0 || p.x2, "conv: C2 > 0 needs x2");
  PSLD_CHECK_ARG(p.KS == 1 || p.KS == 3, "conv: kernel size must be 1 or 3");
  PSLD_CHECK_ARG(p.stride >= 1 && p.pad >= 0, "conv: bad stride/pad");
  PSLD_CHECK_ARG(p.OH == (p.H + 2 * p.pad - p.KS) / p.stride + 1 &&
                 p.OW == (p.W + 2 * p.pad - p.KS) / p.stride + 1, "conv: OH/OW mismatch");
  PSLD_CHECK_ARG(p.in_layout == PSLD_NHWC || (idt == PSLD_F32 && p.C2 == 0),
                 "conv: NCHW input must be fp32 single-source");
  PSLD_CHECK_ARG(p.out_layout == PSLD_NHWC || odt == PSLD_F32, "conv: NCHW output must be fp32");
  PSLD_CHECK_ARG(!p.res || op.i[PSLD_CONV_RES_DTYPE] == odt, "conv: residual dtype != out dtype");
  const int64_t M = (int64_t)p.N * p.OH * p.OW;
  dim3 grid((unsigned)ceil_div(M, BM), (unsigned)ceil_div(p.Cout, BN));
  if (idt == PSLD_F32 && odt == PSLD_F32) launch_pdl(conv_simt_kernel<float, float>, dim3(grid), dim3(256), 0, s, 1, p);
  else if (idt == PSLD_BF16 && odt == PSLD_BF16)
    launch_pdl(conv_simt_kernel<__nv_bfloat16, __nv_bfloat16>, dim3(grid), dim3(256), 0, s, 1, p);
  else if (idt == PSLD_BF16 && odt == PSLD_F32)
    launch_pdl(conv_simt_kernel<__nv_bfloat16, float>, dim3(grid), dim3(256), 0, s, 1, p);
  else if (idt == PSLD_F32 && odt == PSLD_BF16)
    launch_pdl(conv_simt_kernel<float, __nv_bfloat16>, dim3(grid), dim3(256), 0, s, 1, p);
  else if (idt == PSLD_BF16S && odt == PSLD_BF16S)
    launch_pdl(conv_simt_kernel<bf16s, bf16s>, dim3(grid), dim3(256), 0, s, 1, p);
  else if (idt == PSLD_BF16S && odt == PSLD_F32)
    launch_pdl(conv_simt_kernel<bf16s, float>, dim3(grid), dim3(256), 0, s, 1, p);
  else if (idt == PSLD_F32 && odt == PSLD_BF16S)
    launch_pdl(conv_simt_kernel<float, bf16s>, dim3(grid), dim3(256), 0, s, 1, p);
  else { set_error("conv: unsupported dtypes %d -> %d", idt, odt); return PSLD_EINVAL; }
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}

// ======================================================================== attention (SIMT)
// One CTA = one sample x 32 queries.  q|k|v are packed along the channel axis of one [N,HW,3C] tensor
// produced by a single fused NIN GEMM.  Keys are taken in chunks of KC: S = scale * Q K^T of a chunk
// lives in shared memory ([TQ][KC + 1] floats).
//   KC >= HW (every score row fits, HW <= 1518): one pass with an exact softmax, P = softmax(S),
//            O = P V (the S block is computed once and reused by every 256-channel block)
//   KC <  HW: online softmax per chunk: m_new = max(m, rowmax), P = exp(S - m_new),
//            l = l * exp(m - m_new) + rowsum(P), O = O * exp(m - m_new) + P V;  out = O / l.
//            Each 256-channel block recomputes its chunks' S (O stays in registers).
constexpr int TQ = 32;
constexpr int ATTN_TILE = TQ * 33 + 256 * 33 > 32 * 256 ? TQ * 33 + 256 * 33 : 32 * 256;   // floats

template <typename T>
__global__ void __launch_bounds__(256)
attn_simt_kernel(const T* __restrict__ qkv, T* __restrict__ out, int HW, int C, int KC, float scale) {
  pdl_wait();
  extern __shared__ float smem[];
  const int ldS = KC + 1;
  float* S = smem;                               // [TQ][KC + 1]
  float* buf = smem + TQ * ldS;                  // tile buffers
  float* rowst = buf + ATTN_TILE;                // KC < HW: [running max | running sum | rescale][TQ]
  const bool one = KC >= HW;
  const int n = blockIdx.y, q0 = blockIdx.x * TQ;
  const int tid = threadIdx.x;
  const int tq = tid >> 3, tk = tid & 7;
  const int lo = 3 * C;                          // split-bf16 lo offset of a q|k|v row
  const int ld = lo * Elt<T>::kMul;
  const T* base = qkv + (int64_t)n * HW * ld;
  float* Qs = buf;                 // phase 1: [TQ][33]
  float* Ks = buf + TQ * 33;       //          [256][33]
  float* Vs = buf;                 // phase 3: [32][256]

  for (int cb = 0; cb < C; cb += 256) {
    float acc[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = 0.f;
    for (int kc0 = 0; kc0 < HW; kc0 += KC) {
      const int kn = HW - kc0 < KC ? HW - kc0 : KC;
      if (!one || cb == 0) {
        // ---- phase 1: S = scale * Q K^T over the chunk's keys, key blocks of 256, channel chunks of 32
        for (int kb = 0; kb < kn; kb += 256) {
          float sacc[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) sacc[i] = 0.f;
          for (int c0 = 0; c0 < C; c0 += 32) {
            for (int e = tid; e < TQ * 32; e += 256) {
              const int r = e >> 5, cc = e & 31;
              const int q = q0 + r;
              Qs[r * 33 + cc] = (q < HW && c0 + cc < C) ? ld_elt<T>(base + (int64_t)q * ld + c0 + cc, lo) : 0.f;
            }
            for (int e = tid; e < 256 * 32; e += 256) {
              const int r = e >> 5, cc = e & 31;
              const int key = kb + r;
              Ks[r * 33 + cc] = (key < kn && c0 + cc < C)
                                    ? ld_elt<T>(base + (int64_t)(kc0 + key) * ld + C + c0 + cc, lo) : 0.f;
            }
            __syncthreads();
#pragma unroll 4
            for (int cc = 0; cc < 32; ++cc) {
              const float qv = Qs[tq * 33 + cc];
#pragma unroll
              for (int i = 0; i < 32; ++i) sacc[i] = fmaf(qv, Ks[(tk + 8 * i) * 33 + cc], sacc[i]);
            }
            __syncthreads();
          }
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int key = kb + tk + 8 * i;
            if (key < kn) S[tq * ldS + key] = sacc[i] * scale;   // einsum then * C^-0.5 (layerspp.py:82)
          }
        }
        __syncthreads();

        // ---- phase 2: row softmax (F.softmax over keys, layerspp.py:84)
        {
          const int warp = tid >> 5, lane = tid & 31;
          for (int r = warp; r < TQ; r += 8) {
            float* row = S + r * ldS;
            float mx = -INFINITY;
            for (int k = lane; k < kn; k += 32) mx = fmaxf(mx, row[k]);
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, d));
            const float m_old = (one || kc0 == 0) ? -INFINITY : rowst[r];
            const float m_new = fmaxf(m_old, mx);
            float sum = 0.f;
            for (int k = lane; k < kn; k += 32) {
              const float e = expf(row[k] - m_new);
              row[k] = e;
              sum += e;
            }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
            if (one) {
              const float inv = 1.0f / sum;
              for (int k = lane; k < kn; k += 32) row[k] *= inv;
            } else if (lane == 0) {
              const float a = kc0 == 0 ? 0.f : expf(m_old - m_new);
              rowst[r] = m_new;
              rowst[TQ + r] = (kc0 == 0 ? 0.f : rowst[TQ + r] * a) + sum;
              rowst[2 * TQ + r] = a;
            }
          }
        }
        __syncthreads();
      }

      // ---- phase 3: O (+)= P V over the chunk's keys, key chunks of 32
      if (!one) {
        const float a = rowst[2 * TQ + tq];
#pragma unroll
        for (int i = 0; i < 32; ++i) acc[i] *= a;
      }
      for (int k0 = 0; k0 < kn; k0 += 32) {
        for (int e = tid; e < 32 * 256; e += 256) {
          const int r = e >> 8, cc = e & 255;
          const int key = k0 + r;
          Vs[e] = (key < kn && cb + cc < C) ? ld_elt<T>(base + (int64_t)(kc0 + key) * ld + 2 * C + cb + cc, lo) : 0.f;
        }
        __syncthreads();
#pragma unroll 4
        for (int kk = 0; kk < 32; ++kk) {
          const float pv = (k0 + kk < kn) ? S[tq * ldS + k0 + kk] : 0.f;
#pragma unroll
          for (int i = 0; i < 32; ++i) acc[i] = fmaf(pv, Vs[kk * 256 + tk + 8 * i], acc[i]);
        }
        __syncthreads();
      }
    }
    const int q = q0 + tq;
    if (q < HW) {
      const float inv = one ? 1.0f : 1.0f / rowst[TQ + tq];
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const int c = cb + tk + 8 * i;
        if (c < C) st_elt<T>(out + ((int64_t)n * HW + q) * (C * Elt<T>::kMul) + c, one ? acc[i] : acc[i] * inv, C);
      }
    }
  }
}

int run_attn_simt(const psld_op& op, cudaStream_t s) {
  const int N = op.i[PSLD_ATTN_N], HW = op.i[PSLD_ATTN_HW], C = op.i[PSLD_ATTN_C];
  const int dt = op.i[PSLD_ATTN_DTYPE];
  PSLD_CHECK_ARG(N > 0 && HW > 0 && C > 0 && op.in[0] && op.out[0], "attn: bad arguments");
  // the whole score row in one chunk when it fits; otherwise the largest multiple of 256 keys that fits
  // beside the row statistics
  constexpr size_t kMaxSmem = 227 * 1024;
  int KC = HW;
  size_t smem = ((size_t)TQ * (HW + 1) + ATTN_TILE) * sizeof(float);
  if (smem > kMaxSmem) {
    KC = (int)((kMaxSmem / sizeof(float) - ATTN_TILE - 3 * TQ) / TQ - 1) / 256 * 256;
    smem = ((size_t)TQ * (KC + 1) + ATTN_TILE + 3 * TQ) * sizeof(float);
  }
  dim3 grid((unsigned)ceil_div(HW, TQ), (unsigned)N);
  if (dt == PSLD_BF16) {
    PSLD_CHECK_CUDA(cudaFuncSetAttribute(attn_simt_kernel<__nv_bfloat16>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    launch_pdl(attn_simt_kernel<__nv_bfloat16>, dim3(grid), dim3(256), smem, s, 1, (const __nv_bfloat16*)op.in[0],
               (__nv_bfloat16*)op.out[0], HW, C, KC, op.f[0]);
  } else if (dt == PSLD_BF16S) {
    PSLD_CHECK_CUDA(cudaFuncSetAttribute(attn_simt_kernel<bf16s>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    launch_pdl(attn_simt_kernel<bf16s>, dim3(grid), dim3(256), smem, s, 1, (const bf16s*)op.in[0],
               (bf16s*)op.out[0], HW, C, KC, op.f[0]);
  } else {
    PSLD_CHECK_CUDA(cudaFuncSetAttribute(attn_simt_kernel<float>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    launch_pdl(attn_simt_kernel<float>, dim3(grid), dim3(256), smem, s, 1, (const float*)op.in[0], (float*)op.out[0],
               HW, C, KC, op.f[0]);
  }
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}

}  // namespace psld
