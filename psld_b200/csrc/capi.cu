// C-ABI glue: error state, op dispatch, program replay and the native sampling loop.
//
// psld_sampler_run replaces the Python loops SSCSSampler.sample / EulerMaruyamaSampler.sample
// (main/samplers/sde.py:350-370, 38-58): per step it replays the NCSN++ program (one score_fn
// call, sde.py:320 / psld.py:354) and launches ONE fused phase-space kernel, with every scalar
// of the step precomputed on the host.  No host synchronisation inside the loop (the reference
// incurs 9 `.item()` syncs per SSCS step, SURVEY.md §3.1).

#include <stdarg.h>
#include <string.h>

#include "common.cuh"

namespace psld {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static int op_launch_count(const psld_op& op) {
  switch (op.kind) {
    case PSLD_OP_LAYOUT: return 1;
    case PSLD_OP_TEMB: return 4;
    case PSLD_OP_GN:             // producer-side statistics: apply (or affine) only; else + stats pass
      return (op.in[4] && (op.i[PSLD_GN_C2] == 0 || op.in[5])) ? 1 : 2;
    case PSLD_OP_FIR: return 1;
    case PSLD_OP_CONV: return 1;
    case PSLD_OP_ATTN: return 1;
    case PSLD_OP_AXPBY: return 1;
    default: return 0;
  }
}

static int dispatch(const psld_op& op, cudaStream_t s) {
  switch (op.kind) {
    case PSLD_OP_LAYOUT: return run_layout(op, s);
    case PSLD_OP_TEMB: return run_temb(op, s);
    case PSLD_OP_GN: return run_gn(op, s);
    case PSLD_OP_FIR: return run_fir(op, s);
    case PSLD_OP_CONV:
      if (op.engine == PSLD_ENGINE_TC_GN) return run_conv_gn_tc(op, s);
      return op.engine == PSLD_ENGINE_TC ? run_conv_tc(op, s) : run_conv_simt(op, s);
    case PSLD_OP_ATTN:
      return op.engine == PSLD_ENGINE_TC ? run_attn_tc(op, s) : run_attn_simt(op, s);
    case PSLD_OP_AXPBY: return run_axpby(op, s);
    case PSLD_OP_ZERO: {         // statistics accumulators (a memset node, not a kernel of ours)
      const size_t bytes = (size_t)op.i[0] | ((size_t)op.i[1] << 31);
      if (bytes == 0) return PSLD_OK;
      PSLD_CHECK_ARG(op.out[0] != nullptr, "zero: null pointer");
      PSLD_CHECK_CUDA(cudaMemsetAsync(op.out[0], 0, bytes, s));
      return PSLD_OK;
    }
    default:
      set_error("unknown op kind %d", op.kind);
      return PSLD_EINVAL;
  }
}

}  // namespace psld

using namespace psld;

extern "C" int psld_version(void) { return PSLD_B200_VERSION; }

extern "C" const char* psld_last_error(void) { return g_err; }

extern "C" int psld_device_info(int* sm_count, int* cc_major, int* cc_minor) {
  int dev = 0;
  PSLD_CHECK_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  PSLD_CHECK_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (cc_major) *cc_major = prop.major;
  if (cc_minor) *cc_minor = prop.minor;
  return PSLD_OK;
}

extern "C" int psld_axpby(float* out, float a, const float* x, float b, const float* y, int64_t n,
                          psld_stream_t stream) {
  return launch_axpby(out, a, x, b, y, n, (cudaStream_t)stream);
}

extern "C" int psld_op_prepare(psld_op* op) {
  PSLD_CHECK_ARG(op != nullptr, "psld_op_prepare: null op");
  if (op->kind == PSLD_OP_CONV && op->engine == PSLD_ENGINE_TC) return prepare_conv_tc(*op);
  if (op->kind == PSLD_OP_CONV && op->engine == PSLD_ENGINE_TC_GN) return prepare_conv_gn_tc(*op);
  if (op->kind == PSLD_OP_ATTN && op->engine == PSLD_ENGINE_TC) return prepare_attn_tc(*op);
  return PSLD_OK;
}

extern "C" int psld_op_release(psld_op* op) {
  PSLD_CHECK_ARG(op != nullptr, "psld_op_release: null op");
  if (op->kind == PSLD_OP_CONV && op->engine == PSLD_ENGINE_TC) return release_conv_tc(*op);
  if (op->kind == PSLD_OP_CONV && op->engine == PSLD_ENGINE_TC_GN) return release_conv_gn_tc(*op);
  if (op->kind == PSLD_OP_ATTN && op->engine == PSLD_ENGINE_TC) return release_attn_tc(*op);
  return PSLD_OK;
}

extern "C" int psld_op_run(const psld_op* op, psld_stream_t stream) {
  PSLD_CHECK_ARG(op != nullptr, "psld_op_run: null op");
  return dispatch(*op, (cudaStream_t)stream);
}

extern "C" int psld_program_run(const psld_op* ops, int n_ops, psld_stream_t stream) {
  PSLD_CHECK_ARG(ops != nullptr && n_ops >= 0, "psld_program_run: bad program");
  for (int i = 0; i < n_ops; ++i) {
    const int rc = dispatch(ops[i], (cudaStream_t)stream);
    if (rc != PSLD_OK) {
      char inner[400];
      strncpy(inner, g_err, sizeof(inner) - 1);
      inner[sizeof(inner) - 1] = 0;
      set_error("op %d (kind %d): %s", i, ops[i].kind, inner);
      return rc;
    }
  }
  return PSLD_OK;
}

extern "C" int psld_program_launches(const psld_op* ops, int n_ops) {
  if (!ops || n_ops < 0) return 0;
  int n = 0;
  for (int i = 0; i < n_ops; ++i) n += op_launch_count(ops[i]);
  return n;
}

static int run_net(const psld_op* ops, int n_ops, int temb_op, const float* time_ptr,
                   cudaStream_t s, int* step_counter = nullptr) {
  for (int i = 0; i < n_ops; ++i) {
    int rc;
    // every time-embedding op of the program gets this call's time: a classifier-free-guidance
    // program holds two networks (temb_op indexes the first)
    if (i == temb_op || ops[i].kind == PSLD_OP_TEMB) {
      psld_op t = ops[i];
      t.in[0] = time_ptr;      // this call's (log) time, identical for the whole batch
      t.out[2] = step_counter; // graph replay: row index read on the device
      rc = dispatch(t, s);
    } else {
      rc = dispatch(ops[i], s);
    }
    if (rc != PSLD_OK) return rc;
  }
  return PSLD_OK;
}

extern "C" int psld_sampler_run(const psld_op* ops, int n_ops, const psld_sampler_desc* d,
                                psld_stream_t stream) {
  PSLD_CHECK_ARG(ops && d && n_ops > 0, "psld_sampler_run: null argument");
  PSLD_CHECK_ARG(d->state && d->net_in && d->eps && d->time_table, "psld_sampler_run: null buffer");
  PSLD_CHECK_ARG(d->n_steps >= 0 && d->B > 0 && d->chw > 0 && d->chw % 4 == 0,
                 "psld_sampler_run: bad sizes");
  PSLD_CHECK_ARG(d->temb_op >= 0 && d->temb_op < n_ops && ops[d->temb_op].kind == PSLD_OP_TEMB,
                 "psld_sampler_run: temb_op does not index a TEMB op");
  PSLD_CHECK_ARG(d->sampler == 0 ? d->sscs != nullptr : d->em != nullptr,
                 "psld_sampler_run: missing coefficient table");
  PSLD_CHECK_ARG(!d->denoise || d->den, "psld_sampler_run: denoise needs coefficients");
  PSLD_CHECK_ARG(!(d->record && d->fuse_halves), "psld_sampler_run: record requires fuse_halves=0");
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t per_draw = d->B * 2 * d->chw;
  const size_t state_bytes = (size_t)per_draw * dtype_size(d->state_dtype);
  auto z = [&](int64_t k) -> const float* { return d->noise ? d->noise + k * per_draw : nullptr; };
  const int n = d->n_steps;
  int rc = PSLD_OK;

  const bool graph = d->step_counter != nullptr && d->noise == nullptr && d->record == nullptr &&
                     n > 1 && (d->sampler == 0 ? d->sscs_dev != nullptr : d->em_dev != nullptr);
  if (graph) {
    // -------- CUDA-graph replay: capture ONE predictor step, launch it for every step.
    PSLD_CHECK_ARG(s != nullptr, "psld_sampler_run: graph replay needs a non-default stream");
    const int fuse = d->sampler == 0 ? d->fuse_halves : 0;
    if (d->sampler == 0 && fuse && n > 0) {
      rc = psld_sscs_update(d->state, d->state, d->state_dtype, d->net_in, nullptr, nullptr, nullptr,
                            nullptr, &d->sscs[0], PSLD_STAGE_HALF_A, d->seed, 0, d->B, d->chw, s);
      if (rc) return rc;
    }
    // with fuse_halves == 1 the last step has no HALF_C stage: it runs outside the graph
    const int n_graph = (d->sampler == 0 && fuse == 1) ? n - 1 : n;
    cudaGraph_t g = nullptr;
    cudaGraphExec_t ge = nullptr;
    PSLD_CHECK_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
    rc = PSLD_OK;
    if (d->sampler == 0) {
      if (!fuse)
        rc = launch_sscs_table(d->state, d->state_dtype, d->net_in, nullptr, d->sscs_dev,
                               d->step_counter, PSLD_STAGE_HALF_A, d->seed, d->B, d->chw, s);
      if (!rc) rc = run_net(ops, n_ops, d->temb_op, d->time_table, s, d->step_counter);
      int stages = PSLD_STAGE_SCORE | PSLD_STAGE_HALF_B;
      if (fuse == 1) stages |= PSLD_STAGE_HALF_C;
      if (!rc)
        rc = launch_sscs_table(d->state, d->state_dtype, d->net_in, d->eps, d->sscs_dev,
                               d->step_counter, stages, d->seed, d->B, d->chw, s);
    } else {
      rc = run_net(ops, n_ops, d->temb_op, d->time_table, s, d->step_counter);
      if (!rc)
        rc = launch_em_table(d->state, d->state_dtype, d->net_in, d->eps, d->em_dev,
                             d->step_counter, d->seed, d->B, d->chw, s);
    }
    if (!rc) rc = launch_step_inc(d->step_counter, s);
    cudaError_t ce = cudaStreamEndCapture(s, &g);
    if (rc) { if (g) cudaGraphDestroy(g); return rc; }
    if (ce != cudaSuccess) { set_error("cudaStreamEndCapture: %s", cudaGetErrorString(ce)); return PSLD_ECUDA; }
    ce = cudaGraphInstantiate(&ge, g, 0);
    cudaGraphDestroy(g);
    if (ce != cudaSuccess) { set_error("cudaGraphInstantiate: %s", cudaGetErrorString(ce)); return PSLD_ECUDA; }
    for (int i = 0; i < n_graph && ce == cudaSuccess; ++i) ce = cudaGraphLaunch(ge, s);
    if (ce == cudaSuccess && n_graph < n) {
      const int i = n - 1;
      rc = run_net(ops, n_ops, d->temb_op, d->time_table + i, s);
      if (!rc)
        rc = psld_sscs_update(d->state, d->state, d->state_dtype, d->net_in, d->eps, nullptr, nullptr,
                              nullptr, &d->sscs[i], PSLD_STAGE_SCORE | PSLD_STAGE_HALF_B, d->seed, i,
                              d->B, d->chw, s);
    }
    // the executable graph must outlive its launches: drain the stream before destroying it
    cudaError_t se = cudaStreamSynchronize(s);
    cudaGraphExecDestroy(ge);
    if (ce != cudaSuccess) { set_error("cudaGraphLaunch: %s", cudaGetErrorString(ce)); return PSLD_ECUDA; }
    if (se != cudaSuccess) { set_error("graph replay failed: %s", cudaGetErrorString(se)); return PSLD_ECUDA; }
    if (rc) return rc;
  } else if (d->sampler == 0) {
    // -------- SSCS: half step -> score step -> half step (sde.py:331-336)
    if (d->fuse_halves && n > 0) {
      rc = psld_sscs_update(d->state, d->state, d->state_dtype, d->net_in, nullptr, z(0), nullptr,
                            nullptr, &d->sscs[0], PSLD_STAGE_HALF_A, d->seed, 0, d->B, d->chw, s);
      if (rc) return rc;
    }
    for (int i = 0; i < n; ++i) {
      if (!d->fuse_halves) {
        rc = psld_sscs_update(d->state, d->state, d->state_dtype, d->net_in, nullptr, z(2 * i),
                              nullptr, nullptr, &d->sscs[i], PSLD_STAGE_HALF_A, d->seed, i, d->B,
                              d->chw, s);
        if (rc) return rc;
      }
      rc = run_net(ops, n_ops, d->temb_op, d->time_table + i, s);
      if (rc) return rc;
      int stages = PSLD_STAGE_SCORE | PSLD_STAGE_HALF_B;
      // fuse_halves 1: half C (= half A of step i+1) as a separate draw in the same pass;
      // fuse_halves 2: the host merged B and C into one half-step with one draw (exact in law)
      if (d->fuse_halves == 1 && i + 1 < n) stages |= PSLD_STAGE_HALF_C;
      rc = psld_sscs_update(d->state, d->state, d->state_dtype, d->net_in, d->eps, nullptr,
                            z(2 * i + 1), z(2 * i + 2), &d->sscs[i], stages, d->seed, i, d->B,
                            d->chw, s);
      if (rc) return rc;
      if (d->record)
        PSLD_CHECK_CUDA(cudaMemcpyAsync((char*)d->record + (size_t)i * state_bytes, d->state,
                                        state_bytes, cudaMemcpyDeviceToDevice, s));
    }
  } else {
    // -------- Euler-Maruyama (sde.py:16-26, 38-58)
    for (int i = 0; i < n; ++i) {
      rc = run_net(ops, n_ops, d->temb_op, d->time_table + i, s);
      if (rc) return rc;
      rc = psld_em_update(d->state, d->state, d->state_dtype, d->net_in, d->eps, z(i),
                          d->noise ? 0 : 1, &d->em[i], d->seed, i, d->B, d->chw, s);
      if (rc) return rc;
      if (d->record)
        PSLD_CHECK_CUDA(cudaMemcpyAsync((char*)d->record + (size_t)i * state_bytes, d->state,
                                        state_bytes, cudaMemcpyDeviceToDevice, s));
    }
  }
  if (d->denoise) {
    // x + fbar * eps at t = T - eps (sde.py:28-36, 338-348); net_in already holds f32(state)
    rc = run_net(ops, n_ops, d->temb_op, d->time_table + n, s);
    if (rc) return rc;
    rc = psld_em_update(d->state, d->state, d->state_dtype, d->net_in, d->eps, nullptr, 0, d->den,
                        d->seed, n, d->B, d->chw, s);
    if (rc) return rc;
  }
  return PSLD_OK;
}
