// Fused phase-space update kernels: one vectorised pass over HBM per sampler step.
//
// Reference (mandt-lab/PSLD) lines these kernels compute:
//   SSCSSampler.analytical_dynamics ... main/samplers/sde.py:294-312  (stages HALF_*)
//   SSCSSampler.euler_score_dynamics .. main/samplers/sde.py:314-329  (stage SCORE)
//   PSLD.get_score (fp32 coefficients)  main/models/sde/psld.py:230-260
//   EulerMaruyamaSampler.predictor_update_fn / denoising_fn ... sde.py:16-36, 338-348
//   PSLD.sde / reverse_sde ............ main/models/sde/psld.py:330-364
//   PSLD.prior_sampling ............... main/models/sde/psld.py:366-370
//
// The reference spends ~619 aten launches + 9 host syncs per SSCS step on this algebra
// (SURVEY.md §3.1); here all per-step scalars arrive as kernel parameters computed once
// on the host in float64, and every pair (x, m) is read once and written once.
//
// Memory-bound: 4 pairs per thread, 128-bit loads/stores, grid sized to cover the data
// (one wave is >> 148 SMs at the BASELINE batch sizes).

#include <string.h>

#include "common.cuh"

namespace psld {

// ---------------------------------------------------------------- Philox4x32-10
struct Philox {
  static __device__ __forceinline__ uint4 draw(uint64_t seed, uint64_t stream, uint64_t index) {
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    uint4 c = make_uint4((uint32_t)index, (uint32_t)(index >> 32), (uint32_t)stream,
                         (uint32_t)(stream >> 32));
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
      uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
      c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
      k0 += 0x9E3779B9u;
      k1 += 0xBB67AE85u;
    }
    return c;
  }
  // 4 standard normals from one draw (Box-Muller on two uniform pairs).  The radius uses the
  // full-accuracy logf (the tail is where a relative error of the logarithm would show); the angle
  // is drawn on [-pi, pi), the interval on which sin.approx / cos.approx are specified to 2^-21.4
  // absolute error, i.e. below the fp32 rounding of the state the noise is added to (sincospif
  // would cost 96 more instructions per 4 pairs and take the fused update at 2^24 pairs from
  // bandwidth-bound to issue-bound).  The radius uniform
  // is (n + 0.5) 2^-32 in (0, 1): the tail reaches sqrt(-2 ln 2^-33) = 6.76 sigma.  Statistical
  // checks on 2.5e7 draws per stream: tests/test_gpu_kernels.py::test_philox_normal_quality.
  static __device__ __forceinline__ float4 normal4(uint64_t seed, uint64_t stream, uint64_t index) {
    uint4 r = draw(seed, stream, index);
    const float k = 2.3283064365386963e-10f;  // 2^-32
    float u0 = ((float)r.x + 0.5f) * k, u1 = (float)r.y * k;
    float u2 = ((float)r.z + 0.5f) * k, u3 = (float)r.w * k;
    u0 = fminf(u0, 0.99999994f);
    u2 = fminf(u2, 0.99999994f);
    float ra = sqrtf(-2.0f * logf(u0)), rb = sqrtf(-2.0f * logf(u2));
    float sa, ca, sb, cb;
    // angle uniform on [-pi, pi): the range where sin.approx / cos.approx are specified to
    // 2^-21.4 ABSOLUTE error (the former code fed them [0, 2 pi), outside that range)
    __sincosf(6.283185307179586f * (u1 - 0.5f), &sa, &ca);
    __sincosf(6.283185307179586f * (u3 - 0.5f), &sb, &cb);
    return make_float4(ra * ca, ra * sa, rb * cb, rb * sb);
  }
};

template <typename S>
struct St4 { S v[4]; };

template <typename S>
__device__ __forceinline__ St4<S> load4(const S* p);
template <>
__device__ __forceinline__ St4<float> load4<float>(const float* p) {
  float4 t = *reinterpret_cast<const float4*>(p);
  return {{t.x, t.y, t.z, t.w}};
}
template <>
__device__ __forceinline__ St4<double> load4<double>(const double* p) {
  double2 a = *reinterpret_cast<const double2*>(p);
  double2 b = *reinterpret_cast<const double2*>(p + 2);
  return {{a.x, a.y, b.x, b.y}};
}
template <typename S>
__device__ __forceinline__ void store4(S* p, const St4<S>& v);
template <>
__device__ __forceinline__ void store4<float>(float* p, const St4<float>& v) {
  *reinterpret_cast<float4*>(p) = make_float4(v.v[0], v.v[1], v.v[2], v.v[3]);
}
template <>
__device__ __forceinline__ void store4<double>(double* p, const St4<double>& v) {
  *reinterpret_cast<double2*>(p) = make_double2(v.v[0], v.v[1]);
  *reinterpret_cast<double2*>(p + 2) = make_double2(v.v[2], v.v[3]);
}

struct HalfF {  // psld_half_step in the state's arithmetic type
  template <typename S>
  struct T { S a_xx, a_xm, a_mx, a_mm, c11, c12, c21, c22; };
};

template <typename S>
__device__ __forceinline__ void apply_half(const psld_half_step& h, S (&x)[4], S (&m)[4],
                                           const float4& zx, const float4& zm) {
  const S axx = (S)h.a_xx, axm = (S)h.a_xm, amx = (S)h.a_mx, amm = (S)h.a_mm;
  const S c11 = (S)h.c11, c12 = (S)h.c12, c21 = (S)h.c21, c22 = (S)h.c22;
  const float zxa[4] = {zx.x, zx.y, zx.z, zx.w}, zma[4] = {zm.x, zm.y, zm.z, zm.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    S nx = axx * x[i] + axm * m[i] + (c11 * (S)zxa[i] + c12 * (S)zma[i]);
    S nm = amx * x[i] + amm * m[i] + (c21 * (S)zxa[i] + c22 * (S)zma[i]);
    x[i] = nx;
    m[i] = nm;
  }
}

// score = -L^{-T} eps evaluated exactly as the reference does in fp32:
//   s_x = (-li11)*e_x - li12*e_m ; s_m = (-li21)*e_x - li22*e_m   (psld.py:252-259)
__device__ __forceinline__ void score_from_eps(const psld_score_step& sc, float ex, float em,
                                               float& sx, float& sm) {
  if (sc.mode == 0) {
    sx = __fsub_rn(__fmul_rn(-sc.li11, ex), __fmul_rn(sc.li12, em));
    sm = __fsub_rn(__fmul_rn(-sc.li21, ex), __fmul_rn(sc.li22, em));
  } else if (sc.mode == 1) {  // score_m: eps is the momentum channel only (psld.py:240-243)
    sx = 0.0f;
    sm = __fmul_rn(-sc.li22, ex);
  } else {                    // score_x (psld.py:245-248)
    sx = __fmul_rn(-sc.li11, ex);
    sm = 0.0f;
  }
}

__device__ __forceinline__ void load_eps(const float* eps, int mode, int64_t b, int64_t j,
                                         int64_t chw, float4& ex, float4& em) {
  if (mode == 0) {
    const float* p = eps + b * 2 * chw + j;
    ex = *reinterpret_cast<const float4*>(p);
    em = *reinterpret_cast<const float4*>(p + chw);
  } else {
    ex = *reinterpret_cast<const float4*>(eps + b * chw + j);
    em = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

__device__ __forceinline__ void get_noise(const float* z, uint64_t seed, uint64_t draw,
                                          int64_t b, int64_t j, int64_t chw, float4& zx,
                                          float4& zm) {
  if (z != nullptr) {
    const float* p = z + b * 2 * chw + j;
    zx = *reinterpret_cast<const float4*>(p);
    zm = *reinterpret_cast<const float4*>(p + chw);
  } else {
    uint64_t pair4 = (uint64_t)(b * chw + j) >> 1;  // 2 draws of 4 normals per 4 pairs
    zx = Philox::normal4(seed, draw, pair4);
    zm = Philox::normal4(seed, draw, pair4 + 1);
  }
}

struct SscsParams {
  psld_sscs_coeffs c;
  const psld_sscs_coeffs* table;   // optional device table indexed by *step_ptr (CUDA-graph replay)
  const int* step_ptr;
  const float* eps;
  const float* z_a;
  const float* z_b;
  const float* z_c;
  float* net_in;
  uint64_t seed, step;
  int64_t B, chw;
  int stages;
};

template <typename S>
__device__ __forceinline__ void sscs_update_body(S* __restrict__ u_out, const S* __restrict__ u_in,
                                                 const SscsParams& p) {
  const int64_t nvec = p.B * (p.chw >> 2);
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec;
       v += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = v / (p.chw >> 2);
    const int64_t j = (v - b * (p.chw >> 2)) << 2;
    const int64_t ox = b * 2 * p.chw + j;
    St4<S> xs = load4<S>(u_in + ox), ms = load4<S>(u_in + ox + p.chw);
    S(&x)[4] = xs.v;
    S(&m)[4] = ms.v;
    float4 zx, zm;
    if (p.stages & PSLD_STAGE_HALF_A) {
      get_noise(p.z_a, p.seed, 2 * p.step, b, j, p.chw, zx, zm);
      apply_half<S>(p.c.half_a, x, m, zx, zm);
    }
    if (p.stages & PSLD_STAGE_SCORE) {
      float4 ex, em;
      load_eps(p.eps, p.c.score.mode, b, j, p.chw, ex, em);
      const float exa[4] = {ex.x, ex.y, ex.z, ex.w}, ema[4] = {em.x, em.y, em.z, em.w};
      const S kx = (S)p.c.score.k_x, km = (S)p.c.score.k_m, mi = (S)p.c.score.m_inv;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float sx, sm;
        score_from_eps(p.c.score, exa[i], ema[i], sx, sm);
        x[i] = x[i] + kx * ((S)sx + x[i]);             // sde.py:325
        m[i] = m[i] + km * ((S)sm + mi * m[i]);        // sde.py:326-328
      }
    }
    if (p.stages & PSLD_STAGE_HALF_B) {
      get_noise(p.z_b, p.seed, 2 * p.step + 1, b, j, p.chw, zx, zm);
      apply_half<S>(p.c.half_b, x, m, zx, zm);
    }
    if (p.stages & PSLD_STAGE_HALF_C) {
      get_noise(p.z_c, p.seed, 2 * p.step + 2, b, j, p.chw, zx, zm);
      apply_half<S>(p.c.half_c, x, m, zx, zm);
    }
    store4<S>(u_out + ox, xs);
    store4<S>(u_out + ox + p.chw, ms);
    if (p.net_in != nullptr) {
      *reinterpret_cast<float4*>(p.net_in + ox) =
          make_float4((float)x[0], (float)x[1], (float)x[2], (float)x[3]);
      *reinterpret_cast<float4*>(p.net_in + ox + p.chw) =
          make_float4((float)m[0], (float)m[1], (float)m[2], (float)m[3]);
    }
  }
}


// coefficients as a by-value kernel parameter (constant bank)
template <typename S>
__global__ void __launch_bounds__(256)
sscs_update_kernel(S* __restrict__ u_out, const S* __restrict__ u_in, const SscsParams p) {
  pdl_wait();
  sscs_update_body<S>(u_out, u_in, p);
}

// CUDA-graph replay: coefficients = row *step_ptr of a device table, staged in shared memory
template <typename S>
__global__ void __launch_bounds__(256)
sscs_update_table_kernel(S* __restrict__ u_out, const S* __restrict__ u_in, const SscsParams pp) {
  pdl_wait();
  __shared__ SscsParams p;
  const int step = *pp.step_ptr;
  const uint32_t* src = reinterpret_cast<const uint32_t*>(pp.table + step);
  uint32_t* dst = reinterpret_cast<uint32_t*>(&p.c);
  for (int i = threadIdx.x; i < (int)(sizeof(psld_sscs_coeffs) / 4); i += blockDim.x) dst[i] = src[i];
  if (threadIdx.x == 0) {
    p.eps = pp.eps; p.z_a = pp.z_a; p.z_b = pp.z_b; p.z_c = pp.z_c; p.net_in = pp.net_in;
    p.seed = pp.seed; p.step = (uint64_t)step;
    p.B = pp.B; p.chw = pp.chw; p.stages = pp.stages;
  }
  __syncthreads();
  sscs_update_body<S>(u_out, u_in, p);
}

struct EmParams {
  psld_score_step c;
  const psld_score_step* table;
  const int* step_ptr;
  const float* eps;
  const float* z;
  float* net_in;
  uint64_t seed, step;
  int64_t B, chw;
  int use_philox;
  const float* guide;      // optional [B,2C,H,W]: fbar += g^2 * (guide * guide_scale)   (sde.py:86-93)
  double guide_scale;
};

template <typename S>
__device__ __forceinline__ void em_update_body(S* __restrict__ u_out, const S* __restrict__ u_in,
                                               const EmParams& p) {
  const int64_t nvec = p.B * (p.chw >> 2);
  const S hb = (S)p.c.half_beta, mi = (S)p.c.m_inv, ga = (S)p.c.gamma, nu = (S)p.c.nu;
  const S g2x = (S)p.c.g2_x, g2m = (S)p.c.g2_m, dt = (S)p.c.dt;
  const S gsx = (S)p.c.gs_x, gsm = (S)p.c.gs_m;
  const bool noisy = (p.z != nullptr) || p.use_philox;
  const bool guided = p.guide != nullptr;
  const S gsc = (S)p.guide_scale;
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec;
       v += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = v / (p.chw >> 2);
    const int64_t j = (v - b * (p.chw >> 2)) << 2;
    const int64_t ox = b * 2 * p.chw + j;
    St4<S> xs = load4<S>(u_in + ox), ms = load4<S>(u_in + ox + p.chw);
    float4 ex, em, zx = make_float4(0, 0, 0, 0), zm = zx;
    load_eps(p.eps, p.c.mode, b, j, p.chw, ex, em);
    if (noisy) get_noise(p.z, p.seed, p.step, b, j, p.chw, zx, zm);
    const float exa[4] = {ex.x, ex.y, ex.z, ex.w}, ema[4] = {em.x, em.y, em.z, em.w};
    const float zxa[4] = {zx.x, zx.y, zx.z, zx.w}, zma[4] = {zm.x, zm.y, zm.z, zm.w};
    float gxa[4] = {0.f, 0.f, 0.f, 0.f}, gma[4] = {0.f, 0.f, 0.f, 0.f};
    if (guided) {
      const float4 a = *reinterpret_cast<const float4*>(p.guide + ox);
      const float4 c = *reinterpret_cast<const float4*>(p.guide + ox + p.chw);
      gxa[0] = a.x; gxa[1] = a.y; gxa[2] = a.z; gxa[3] = a.w;
      gma[0] = c.x; gma[1] = c.y; gma[2] = c.z; gma[3] = c.w;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const S x = xs.v[i], m = ms.v[i];
      float sx, sm;
      score_from_eps(p.c, exa[i], ema[i], sx, sm);
      const S fx = hb * (mi * m - ga * x);              // psld.py:336
      const S fm = hb * (-nu * m - x);                  // psld.py:337
      S fbx = -fx + g2x * (S)sx;                        // psld.py:359
      S fbm = -fm + g2m * (S)sm;
      if (guided) {                                     // classifier guidance, sde.py:93
        fbx = fbx + g2x * ((S)gxa[i] * gsc);
        fbm = fbm + g2m * ((S)gma[i] * gsc);
      }
      S nx = x + fbx * dt, nm = m + fbm * dt;           // sde.py:23
      if (noisy) {
        nx = nx + gsx * (S)zxa[i];                      // sde.py:24-25
        nm = nm + gsm * (S)zma[i];
      }
      xs.v[i] = nx;
      ms.v[i] = nm;
    }
    store4<S>(u_out + ox, xs);
    store4<S>(u_out + ox + p.chw, ms);
    if (p.net_in != nullptr) {
      *reinterpret_cast<float4*>(p.net_in + ox) =
          make_float4((float)xs.v[0], (float)xs.v[1], (float)xs.v[2], (float)xs.v[3]);
      *reinterpret_cast<float4*>(p.net_in + ox + p.chw) =
          make_float4((float)ms.v[0], (float)ms.v[1], (float)ms.v[2], (float)ms.v[3]);
    }
  }
}


template <typename S>
__global__ void __launch_bounds__(256)
em_update_kernel(S* __restrict__ u_out, const S* __restrict__ u_in, const EmParams p) {
  pdl_wait();
  em_update_body<S>(u_out, u_in, p);
}

template <typename S>
__global__ void __launch_bounds__(256)
em_update_table_kernel(S* __restrict__ u_out, const S* __restrict__ u_in, const EmParams pp) {
  pdl_wait();
  __shared__ EmParams p;
  const int step = *pp.step_ptr;
  const uint32_t* src = reinterpret_cast<const uint32_t*>(pp.table + step);
  uint32_t* dst = reinterpret_cast<uint32_t*>(&p.c);
  for (int i = threadIdx.x; i < (int)(sizeof(psld_score_step) / 4); i += blockDim.x) dst[i] = src[i];
  if (threadIdx.x == 0) {
    p.eps = pp.eps; p.z = pp.z; p.net_in = pp.net_in; p.seed = pp.seed; p.step = (uint64_t)step;
    p.B = pp.B; p.chw = pp.chw; p.use_philox = pp.use_philox;
    p.guide = pp.guide; p.guide_scale = pp.guide_scale;
  }
  __syncthreads();
  em_update_body<S>(u_out, u_in, p);
}

__global__ void __launch_bounds__(256)
prior_kernel(float* __restrict__ u, float m_std, uint64_t seed, int64_t B, int64_t chw) {
  pdl_wait();
  const int64_t nvec = B * (chw >> 2);
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec;
       v += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = v / (chw >> 2);
    const int64_t j = (v - b * (chw >> 2)) << 2;
    float4 zx, zm;
    get_noise(nullptr, seed, ~0ull, b, j, chw, zx, zm);
    float* p = u + b * 2 * chw + j;
    *reinterpret_cast<float4*>(p) = zx;
    *reinterpret_cast<float4*>(p + chw) =
        make_float4(zm.x * m_std, zm.y * m_std, zm.z * m_std, zm.w * m_std);
  }
}

// SimpleImageWriter + save_as_images of the reference (main/callbacks.py:103-107,
// main/util.py:147-158) as one pass: keep the position half, x*0.5+0.5, *255, clip to [0,255],
// truncate to uint8, NCHW -> NHWC.  Arithmetic in the state's own type, like the reference.
template <typename S>
__global__ void __launch_bounds__(256)
quantize_kernel(const S* __restrict__ u, uint8_t* __restrict__ out, int64_t B, int C, int HW) {
  pdl_wait();
  const int64_t total = B * HW * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const int64_t r = i / C;
    const int p = (int)(r % HW);
    const int64_t b = r / HW;
    S v = u[(b * 2 * C + c) * HW + p] * (S)0.5 + (S)0.5;
    v = v * (S)255;
    v = v < (S)0 ? (S)0 : (v > (S)255 ? (S)255 : v);
    out[i] = (uint8_t)v;
  }
}

static inline int grid_for(int64_t nvec) {
  // enough CTAs for >= 8 resident per SM on 148 SMs, capped so small problems stay 1 wave
  int64_t g = ceil_div(nvec, 256);
  const int64_t cap = 148 * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace psld

using namespace psld;

namespace psld {
__global__ void step_inc_kernel(int* p) {
  pdl_wait(); *p += 1; }

int launch_step_inc(int* step_ptr, cudaStream_t s) {
  launch_pdl(step_inc_kernel, dim3((unsigned)(1)), dim3(1), 0, s, 1, step_ptr);
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}

// graph-replay variants: coefficients come from row *step_ptr of a device table
int launch_sscs_table(void* u, int state_dtype, float* net_in, const float* eps,
                      const psld_sscs_coeffs* table, const int* step_ptr, int stages, uint64_t seed,
                      int64_t B, int64_t chw, cudaStream_t s) {
  SscsParams p;
  memset(&p, 0, sizeof(p));
  p.table = table; p.step_ptr = step_ptr;
  p.eps = eps; p.net_in = net_in; p.seed = seed; p.B = B; p.chw = chw; p.stages = stages;
  const int grid = grid_for(B * (chw / 4));
  if (state_dtype == PSLD_F64)
    launch_pdl(sscs_update_table_kernel<double>, dim3(grid), dim3(256), 0, s, 1, (double*)u, (const double*)u, p);
  else
    launch_pdl(sscs_update_table_kernel<float>, dim3(grid), dim3(256), 0, s, 1, (float*)u, (const float*)u, p);
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}

int launch_em_table(void* u, int state_dtype, float* net_in, const float* eps,
                    const psld_score_step* table, const int* step_ptr, uint64_t seed, int64_t B,
                    int64_t chw, cudaStream_t s) {
  EmParams p;
  memset(&p, 0, sizeof(p));
  p.table = table; p.step_ptr = step_ptr;
  p.eps = eps; p.net_in = net_in; p.seed = seed; p.B = B; p.chw = chw; p.use_philox = 1;
  const int grid = grid_for(B * (chw / 4));
  if (state_dtype == PSLD_F64)
    launch_pdl(em_update_table_kernel<double>, dim3(grid), dim3(256), 0, s, 1, (double*)u, (const double*)u, p);
  else
    launch_pdl(em_update_table_kernel<float>, dim3(grid), dim3(256), 0, s, 1, (float*)u, (const float*)u, p);
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}
}  // namespace psld

extern "C" int psld_sscs_update(void* u_out, const void* u_in, int state_dtype, float* net_in,
                                const float* eps, const float* z_a, const float* z_b,
                                const float* z_c, const psld_sscs_coeffs* coeffs, int stages,
                                uint64_t seed, uint64_t step, int64_t B, int64_t chw,
                                psld_stream_t stream) {
  PSLD_CHECK_ARG(u_out && u_in && coeffs, "psld_sscs_update: null pointer");
  PSLD_CHECK_ARG(B > 0 && chw > 0 && chw % 4 == 0, "psld_sscs_update: need chw %% 4 == 0");
  PSLD_CHECK_ARG(stages > 0 && stages < 16, "psld_sscs_update: bad stage mask %d", stages);
  PSLD_CHECK_ARG(!(stages & PSLD_STAGE_SCORE) || eps, "psld_sscs_update: SCORE needs eps");
  PSLD_CHECK_ARG(state_dtype == PSLD_F64 || state_dtype == PSLD_F32,
                 "psld_sscs_update: state dtype must be f64 or f32");
  SscsParams p;
  p.c = *coeffs;
  p.table = nullptr; p.step_ptr = nullptr;
  p.eps = eps; p.z_a = z_a; p.z_b = z_b; p.z_c = z_c; p.net_in = net_in;
  p.seed = seed; p.step = step; p.B = B; p.chw = chw; p.stages = stages;
  const int grid = grid_for(B * (chw / 4));
  cudaStream_t s = (cudaStream_t)stream;
  if (state_dtype == PSLD_F64)
    launch_pdl(sscs_update_kernel<double>, dim3(grid), dim3(256), 0, s, 1, (double*)u_out, (const double*)u_in, p);
  else
    launch_pdl(sscs_update_kernel<float>, dim3(grid), dim3(256), 0, s, 1, (float*)u_out, (const float*)u_in, p);
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}

extern "C" int psld_em_update(void* u_out, const void* u_in, int state_dtype, float* net_in,
                              const float* eps, const float* z, int use_philox,
                              const psld_score_step* coeffs, uint64_t seed, uint64_t step,
                              int64_t B, int64_t chw, psld_stream_t stream) {
  return psld_em_update_guided(u_out, u_in, state_dtype, net_in, eps, nullptr, 0.0, z, use_philox, coeffs,
                               seed, step, B, chw, stream);
}

extern "C" int psld_em_update_guided(void* u_out, const void* u_in, int state_dtype, float* net_in,
                                     const float* eps, const float* guide, double guide_scale,
                                     const float* z, int use_philox, const psld_score_step* coeffs,
                                     uint64_t seed, uint64_t step, int64_t B, int64_t chw,
                                     psld_stream_t stream) {
  PSLD_CHECK_ARG(u_out && u_in && coeffs && eps, "psld_em_update: null pointer");
  PSLD_CHECK_ARG(B > 0 && chw > 0 && chw % 4 == 0, "psld_em_update: need chw %% 4 == 0");
  PSLD_CHECK_ARG(state_dtype == PSLD_F64 || state_dtype == PSLD_F32,
                 "psld_em_update: state dtype must be f64 or f32");
  EmParams p;
  p.c = *coeffs;
  p.table = nullptr; p.step_ptr = nullptr;
  p.eps = eps; p.z = z; p.net_in = net_in; p.seed = seed; p.step = step;
  p.B = B; p.chw = chw; p.use_philox = use_philox;
  p.guide = guide; p.guide_scale = guide_scale;
  const int grid = grid_for(B * (chw / 4));
  cudaStream_t s = (cudaStream_t)stream;
  if (state_dtype == PSLD_F64)
    launch_pdl(em_update_kernel<double>, dim3(grid), dim3(256), 0, s, 1, (double*)u_out, (const double*)u_in, p);
  else
    launch_pdl(em_update_kernel<float>, dim3(grid), dim3(256), 0, s, 1, (float*)u_out, (const float*)u_in, p);
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}

// ---------------------------------------------------------------- VP-SDE Euler-Maruyama
template <typename S>
__global__ void __launch_bounds__(256)
vp_em_update_kernel(S* __restrict__ xo, const S* __restrict__ xi, float* __restrict__ net_in,
                    const float* __restrict__ eps, const float* __restrict__ z, int use_philox,
                    psld_vp_step c, uint64_t seed, uint64_t step, int64_t n) {
  pdl_wait();
  const int64_t total = n / 4;
  const S hb = (S)c.half_beta, g2 = (S)c.g2, nis = (S)c.neg_inv_std, dt = (S)c.dt, gs = (S)c.gs;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    St4<S> x = load4<S>(xi + 4 * i);
    const float4 e = *reinterpret_cast<const float4*>(eps + 4 * i);
    float4 zz = make_float4(0.f, 0.f, 0.f, 0.f);
    if (z) zz = *reinterpret_cast<const float4*>(z + 4 * i);
    else if (use_philox) zz = Philox::normal4(seed, step, (uint64_t)i);
    const float ea[4] = {e.x, e.y, e.z, e.w}, za[4] = {zz.x, zz.y, zz.z, zz.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const S score = (S)ea[k] * nis;                       // vpsde.py:27-28
      const S fbar = hb * x.v[k] + g2 * score;              // vpsde.py:60-68
      x.v[k] = (x.v[k] + fbar * dt) + gs * (S)za[k];        // sde.py:23-25
    }
    store4<S>(xo + 4 * i, x);
    if (net_in)
      *reinterpret_cast<float4*>(net_in + 4 * i) =
          make_float4((float)x.v[0], (float)x.v[1], (float)x.v[2], (float)x.v[3]);
  }
}

extern "C" int psld_vp_em_update(void* x_out, const void* x_in, int state_dtype, float* net_in,
                                 const float* eps, const float* z, int use_philox,
                                 const psld_vp_step* coeffs, uint64_t seed, uint64_t step, int64_t n,
                                 psld_stream_t stream) {
  PSLD_CHECK_ARG(x_out && x_in && eps && coeffs && n > 0 && n % 4 == 0,
                 "psld_vp_em_update: bad arguments");
  PSLD_CHECK_ARG(state_dtype == PSLD_F64 || state_dtype == PSLD_F32,
                 "psld_vp_em_update: state dtype must be f64 or f32");
  const int grid = grid_for(n / 4);
  cudaStream_t s = (cudaStream_t)stream;
  if (state_dtype == PSLD_F64)
    launch_pdl(vp_em_update_kernel<double>, dim3(grid), dim3(256), 0, s, 1, (double*)x_out,
               (const double*)x_in, net_in, eps, z, use_philox, *coeffs, seed, step, n);
  else
    launch_pdl(vp_em_update_kernel<float>, dim3(grid), dim3(256), 0, s, 1, (float*)x_out,
               (const float*)x_in, net_in, eps, z, use_philox, *coeffs, seed, step, n);
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}

// ---------------------------------------------------------------- inpainting combine
template <typename S>
__global__ void __launch_bounds__(256)
inpaint_combine_kernel(S* __restrict__ u, float* __restrict__ net_in, const float* __restrict__ x0,
                       const float* __restrict__ mask, const float* __restrict__ z_m0,
                       const float* __restrict__ z_eps, psld_inpaint_step c, uint64_t seed,
                       uint64_t step, int64_t B, int64_t chw) {
  pdl_wait();
  const int64_t q = chw / 4;
  const int64_t total = B * q;
  const S axx = (S)c.a_xx, axm = (S)c.a_xm, amx = (S)c.a_mx, amm = (S)c.a_mm;
  const S c11 = (S)c.c11, c12 = (S)c.c12, c21 = (S)c.c21, c22 = (S)c.c22, ms = (S)c.m0_std;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / q, j = (i - b * q) * 4;
    S* px = u + b * 2 * chw + j;
    S* pm = px + chw;
    St4<S> x = load4<S>(px), m = load4<S>(pm);
    const float4 x0v = *reinterpret_cast<const float4*>(x0 + b * chw + j);
    const float4 mkv = *reinterpret_cast<const float4*>(mask + b * chw + j);
    float4 zm, ex, em;
    if (z_eps) {
      zm = z_m0 ? *reinterpret_cast<const float4*>(z_m0 + b * chw + j) : make_float4(0, 0, 0, 0);
      ex = *reinterpret_cast<const float4*>(z_eps + b * 2 * chw + j);
      em = *reinterpret_cast<const float4*>(z_eps + b * 2 * chw + chw + j);
    } else {      // three independent Philox streams per step, disjoint from the predictor's
      zm = Philox::normal4(seed, (step << 2) | (1ull << 62), (uint64_t)i);
      ex = Philox::normal4(seed, (step << 2) | (1ull << 62) | 1ull, (uint64_t)i);
      em = Philox::normal4(seed, (step << 2) | (1ull << 62) | 2ull, (uint64_t)i);
    }
    const float x0a[4] = {x0v.x, x0v.y, x0v.z, x0v.w}, mka[4] = {mkv.x, mkv.y, mkv.z, mkv.w};
    const float zma[4] = {zm.x, zm.y, zm.z, zm.w}, exa[4] = {ex.x, ex.y, ex.z, ex.w};
    const float ema[4] = {em.x, em.y, em.z, em.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const S xo = (S)x0a[k], mk = (S)mka[k];
      const S m0 = ms * (S)zma[k];
      S xk = axx * xo + axm * m0, mkk = amx * xo + amm * m0;
      if (!c.mean_only) {
        xk += c11 * (S)exa[k] + c12 * (S)ema[k];
        mkk += c21 * (S)exa[k] + c22 * (S)ema[k];
      }
      x.v[k] = x.v[k] * ((S)1 - mk) + xk * mk;
      m.v[k] = m.v[k] * ((S)1 - mk) + mkk * mk;
    }
    store4<S>(px, x);
    store4<S>(pm, m);
    if (net_in) {
      *reinterpret_cast<float4*>(net_in + b * 2 * chw + j) =
          make_float4((float)x.v[0], (float)x.v[1], (float)x.v[2], (float)x.v[3]);
      *reinterpret_cast<float4*>(net_in + b * 2 * chw + chw + j) =
          make_float4((float)m.v[0], (float)m.v[1], (float)m.v[2], (float)m.v[3]);
    }
  }
}

extern "C" int psld_inpaint_combine(void* u, int state_dtype, float* net_in, const float* x0,
                                    const float* mask, const float* z_m0, const float* z_eps,
                                    const psld_inpaint_step* coeffs, uint64_t seed, uint64_t step,
                                    int64_t B, int64_t chw, psld_stream_t stream) {
  PSLD_CHECK_ARG(u && x0 && mask && coeffs && B > 0 && chw > 0 && chw % 4 == 0,
                 "psld_inpaint_combine: bad arguments");
  PSLD_CHECK_ARG(state_dtype == PSLD_F64 || state_dtype == PSLD_F32,
                 "psld_inpaint_combine: state dtype must be f64 or f32");
  PSLD_CHECK_ARG(!(z_m0 && !z_eps), "psld_inpaint_combine: z_m0 given without z_eps");
  const int grid = grid_for(B * (chw / 4));
  cudaStream_t s = (cudaStream_t)stream;
  if (state_dtype == PSLD_F64)
    launch_pdl(inpaint_combine_kernel<double>, dim3(grid), dim3(256), 0, s, 1, (double*)u, net_in, x0,
               mask, z_m0, z_eps, *coeffs, seed, step, B, chw);
  else
    launch_pdl(inpaint_combine_kernel<float>, dim3(grid), dim3(256), 0, s, 1, (float*)u, net_in, x0,
               mask, z_m0, z_eps, *coeffs, seed, step, B, chw);
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}

extern "C" int psld_prior_sample(float* u, double m_std, uint64_t seed, int64_t B, int64_t chw,
                                 psld_stream_t stream) {
  PSLD_CHECK_ARG(u && B > 0 && chw > 0 && chw % 4 == 0, "psld_prior_sample: bad arguments");
  launch_pdl(prior_kernel, dim3((unsigned)(grid_for(B * (chw / 4)))), dim3(256), 0, (cudaStream_t)stream, 1, u, (float)m_std, seed,
                                                                         B, chw);
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}

extern "C" int psld_quantize_images(const void* state, int state_dtype, uint8_t* out_nhwc, int64_t B,
                                    int C, int HW, psld_stream_t stream) {
  PSLD_CHECK_ARG(state && out_nhwc && B > 0 && C > 0 && HW > 0, "psld_quantize_images: bad arguments");
  PSLD_CHECK_ARG(state_dtype == PSLD_F64 || state_dtype == PSLD_F32,
                 "psld_quantize_images: state dtype must be f64 or f32");
  const int grid = grid_for(B * HW * C);
  cudaStream_t s = (cudaStream_t)stream;
  if (state_dtype == PSLD_F64)
    launch_pdl(quantize_kernel<double>, dim3(grid), dim3(256), 0, s, 1, (const double*)state, out_nhwc, B, C, HW);
  else
    launch_pdl(quantize_kernel<float>, dim3(grid), dim3(256), 0, s, 1, (const float*)state, out_nhwc, B, C, HW);
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}

// ---------------------------------------------------------------- probability-flow ODE (bb_ode)
// Reverse drift alone, PSLD.reverse_sde (psld.py:345-364): fbar = -f + g^2 * (score_scale * score),
// score_scale = 0.5 for the probability-flow formulation (BBODESampler.ode_fn, ode.py:42-46).  The
// state is read in its own type (the reference evaluates f on the batch-dtype copy of y); fbar is
// always float64 (vec_t is float64, psld.py:333-337 promotes).
template <typename S>
__global__ void __launch_bounds__(256)
reverse_drift_kernel(double* __restrict__ out, const S* __restrict__ u, const float* __restrict__ eps,
                     psld_score_step c, double score_scale, int64_t B, int64_t chw) {
  pdl_wait();
  const int64_t nvec = B * (chw >> 2);
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec;
       v += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = v / (chw >> 2);
    const int64_t j = (v - b * (chw >> 2)) << 2;
    const int64_t ox = b * 2 * chw + j;
    St4<S> xs = load4<S>(u + ox), ms = load4<S>(u + ox + chw);
    float4 ex, em;
    load_eps(eps, c.mode, b, j, chw, ex, em);
    const float exa[4] = {ex.x, ex.y, ex.z, ex.w}, ema[4] = {em.x, em.y, em.z, em.w};
    St4<double> fx4, fm4;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float sx, sm;
      score_from_eps(c, exa[i], ema[i], sx, sm);
      // psld.py:336-337: `0.5 * beta_t * (m_inv * m - gamma * x)`: the bracket is evaluated in the
      // STATE's dtype (python scalars times a float32 tensor stay float32, op by op, no fusion),
      // the float64 beta_t then promotes the product
      double bx, bm;
      if (sizeof(S) == 4) {
        const float x = (float)xs.v[i], m = (float)ms.v[i];
        bx = (double)__fsub_rn(__fmul_rn((float)c.m_inv, m), __fmul_rn((float)c.gamma, x));
        bm = (double)__fsub_rn(__fmul_rn(-(float)c.nu, m), x);
      } else {
        const double x = (double)xs.v[i], m = (double)ms.v[i];
        bx = c.m_inv * m - c.gamma * x;
        bm = -c.nu * m - x;
      }
      // the reference scales the fp32 score by 0.5 in fp32 (exact), then promotes (psld.py:356-359)
      const double fx = c.half_beta * bx;
      const double fm = c.half_beta * bm;
      fx4.v[i] = -fx + c.g2_x * (double)(sx * (float)score_scale);
      fm4.v[i] = -fm + c.g2_m * (double)(sm * (float)score_scale);
    }
    store4<double>(out + ox, fx4);
    store4<double>(out + ox + chw, fm4);
  }
}

// VP-SDE twin (vpsde.py:42-67 with probability_flow): f = (-0.5 beta) x, score = -eps / std, halved,
// fbar = -f + g^2 score, all in float64 (beta_t, std are float64 tensors in the reference, so the
// float32 state / eps promote before the first product).  x: [n] elements.
template <typename S>
__global__ void __launch_bounds__(256)
vp_reverse_drift_kernel(double* __restrict__ out, const S* __restrict__ x, const float* __restrict__ eps,
                        psld_vp_step c, double score_scale, int64_t n) {
  pdl_wait();
  const int64_t nvec = n >> 2;
  const double nhb = -c.half_beta;
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec;
       v += (int64_t)gridDim.x * blockDim.x) {
    St4<S> xs = load4<S>(x + 4 * v);
    const float4 e = *reinterpret_cast<const float4*>(eps + 4 * v);
    const float ea[4] = {e.x, e.y, e.z, e.w};
    St4<double> f4;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const double f = nhb * (double)xs.v[i];
      const double score = score_scale * ((double)ea[i] * c.neg_inv_std);
      f4.v[i] = -f + c.g2 * score;
    }
    store4<double>(out + 4 * v, f4);
  }
}

// out = y + h * sum_j coef[j] K[j]   (one Runge-Kutta stage / solution combination, float64), with
// optional rounded copies: out32 (the state as a float32 batch sees it, and the network input).
struct RkCoef { double c[8]; };

__global__ void __launch_bounds__(256)
rk_combine_kernel(double* __restrict__ out, float* __restrict__ out32, const double* __restrict__ y,
                  const double* __restrict__ K, RkCoef co, int terms, double h, int64_t n) {
  pdl_wait();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    double acc = 0.0;
    for (int j = 0; j < terms; ++j) acc += K[(int64_t)j * n + i] * co.c[j];
    const double v = y[i] + acc * h;
    if (out) out[i] = v;
    if (out32) out32[i] = (float)v;
  }
}

// sum_out += sum_i ( (h * sum_j e[j] K[j][i]) / (atol + max(|y_i|, |ynew_i|) * rtol) )^2
__global__ void __launch_bounds__(256)
rk_error_kernel(const double* __restrict__ y, const double* __restrict__ y_new,
                const double* __restrict__ K, RkCoef e, int terms, double h, double atol, double rtol,
                int64_t n, double* __restrict__ sum_out) {
  pdl_wait();
  double local = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    double acc = 0.0;
    for (int j = 0; j < terms; ++j) acc += K[(int64_t)j * n + i] * e.c[j];
    const double sc = atol + fmax(fabs(y[i]), fabs(y_new[i])) * rtol;
    const double r = acc * h / sc;
    local += r * r;
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) local += __shfl_xor_sync(0xffffffffu, local, d);
  __shared__ double sh[8];
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += sh[w];
    atomicAdd(sum_out, t);
  }
}

extern "C" int psld_reverse_drift(double* out, const void* u, int state_dtype, const float* eps,
                                  const psld_score_step* coeffs, double score_scale, int64_t B,
                                  int64_t chw, psld_stream_t stream) {
  PSLD_CHECK_ARG(out && u && eps && coeffs, "psld_reverse_drift: null pointer");
  PSLD_CHECK_ARG(B > 0 && chw > 0 && chw % 4 == 0, "psld_reverse_drift: need chw %% 4 == 0");
  PSLD_CHECK_ARG(state_dtype == PSLD_F64 || state_dtype == PSLD_F32, "psld_reverse_drift: state dtype");
  const int grid = grid_for(B * (chw / 4));
  cudaStream_t s = (cudaStream_t)stream;
  if (state_dtype == PSLD_F64)
    launch_pdl(reverse_drift_kernel<double>, dim3(grid), dim3(256), 0, s, 1, out, (const double*)u, eps,
               *coeffs, score_scale, B, chw);
  else
    launch_pdl(reverse_drift_kernel<float>, dim3(grid), dim3(256), 0, s, 1, out, (const float*)u, eps,
               *coeffs, score_scale, B, chw);
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}

extern "C" int psld_vp_reverse_drift(double* out, const void* x, int state_dtype, const float* eps,
                                     const psld_vp_step* coeffs, double score_scale, int64_t n,
                                     psld_stream_t stream) {
  PSLD_CHECK_ARG(out && x && eps && coeffs && n > 0 && n % 4 == 0, "psld_vp_reverse_drift: bad arguments");
  PSLD_CHECK_ARG(state_dtype == PSLD_F64 || state_dtype == PSLD_F32, "psld_vp_reverse_drift: state dtype");
  const int grid = grid_for(n / 4);
  cudaStream_t s = (cudaStream_t)stream;
  if (state_dtype == PSLD_F64)
    launch_pdl(vp_reverse_drift_kernel<double>, dim3(grid), dim3(256), 0, s, 1, out, (const double*)x, eps,
               *coeffs, score_scale, n);
  else
    launch_pdl(vp_reverse_drift_kernel<float>, dim3(grid), dim3(256), 0, s, 1, out, (const float*)x, eps,
               *coeffs, score_scale, n);
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}

extern "C" int psld_rk_combine(double* out, float* out32, const double* y, const double* K,
                               const double* coef /* host */, int terms, double h, int64_t n,
                               psld_stream_t stream) {
  PSLD_CHECK_ARG(y && (out || out32) && (terms == 0 || (K && coef)) && terms >= 0 && terms <= 8 && n > 0,
                 "psld_rk_combine: bad arguments");
  RkCoef co;
  for (int j = 0; j < 8; ++j) co.c[j] = j < terms ? coef[j] : 0.0;
  launch_pdl(rk_combine_kernel, dim3((unsigned)grid_for(n)), dim3(256), 0, (cudaStream_t)stream, 1, out,
             out32, y, K, co, terms, h, n);
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}

extern "C" int psld_rk_error(const double* y, const double* y_new, const double* K,
                             const double* e /* host */, int terms, double h, double atol, double rtol,
                             int64_t n, double* sum_out, psld_stream_t stream) {
  PSLD_CHECK_ARG(y && y_new && K && e && sum_out && terms > 0 && terms <= 8 && n > 0,
                 "psld_rk_error: bad arguments");
  RkCoef co;
  for (int j = 0; j < 8; ++j) co.c[j] = j < terms ? e[j] : 0.0;
  launch_pdl(rk_error_kernel, dim3((unsigned)grid_for(n)), dim3(256), 0, (cudaStream_t)stream, 1, y,
             y_new, K, co, terms, h, atol, rtol, n, sum_out);
  PSLD_CHECK_LAUNCH();
  return PSLD_OK;
}
