#!/usr/bin/env python
"""bench.py — PSLD CIFAR-10 SSCS sampling throughput (samples/sec) on N B200s.

Contract (driver): ``python bench.py --gpus N --steps K --warmup W`` (N>1 under torchrun) prints
ONE JSON line on rank 0.  A "step" is one SSCS predictor step (one NCSN++ score_fn call + one
fused phase-space update) over the per-GPU batch; samples/sec = batch_total / (NFE * step time)
with NFE = 1000 network calls per sample (BASELINE.json configs[1]: n_discrete_steps=1000).

  value ...... device-timed (CUDA events, max over ranks), inputs resident in HBM
  e2e ........ the same metric through the public API ``SSCSSampler.sample`` from a pinned HOST
               prior to a HOST result, full 1000-NFE run, H2D/D2H inside the timed region
  roofline ... dominant kernel (tcgen05 implicit-GEMM conv): algorithmic FLOPs / CUDA-event time
               vs the measured cuBLAS bf16 peak in MEASURED_PEAKS.json
  cpu_baseline the CPU oracle port of the reference path on the host cores (rank 0, N=1)

``--impl reference`` times the reference's CPU implementation of the path (oracle port; the
reference is Python and cannot travel to the GPU box) on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NFE = 1000
METRIC = "PSLD CIFAR-10 samples/sec (SSCS sampler)"
UNIT = "samples/sec"


WORKLOADS = {
    # name: (config factory, GFLOP/sample/NFE from BASELINE.md §2, default per-GPU batch, description)
    "cifar10": ("cifar10_config", 76.43e9, 256,
                "PSLD CIFAR-10 NCSN++ (nf=128, ch_mult=[2,2,2], 8 res blocks, attn@16, fir, fourier), "
                "SSCS sampler, 1000 NFE, random-init weights (BASELINE configs[1])"),
    "celeba64": ("celeba64_config", 84.06e9, 64,
                 "PSLD CelebA-64 NCSN++ (nf=128, ch_mult=[1,2,2,2], 4 res blocks, attn@16, fir, fourier), "
                 "SSCS sampler, 1000 NFE, random-init weights (BASELINE configs[3])"),
    # classifier-free guidance: two score_fn passes per step (two random-init networks), w = 1.5
    "cifar10_cfg": ("cifar10_config", 2 * 76.43e9, 128,
                    "PSLD CIFAR-10 NCSN++ x2 (conditional + unconditional network, classifier-free guidance "
                    "eps = (1+w) eps_c - w eps_u, w = 1.5: two score_fn passes per step), SSCS sampler, 1000 NFE, "
                    "random-init weights (BASELINE configs[4]: --batch-total 1024 on 8 GPUs)"),
}
CFG_WEIGHT = 1.5


def metric_name(workload):
    return METRIC.replace("CIFAR-10", "CelebA-64") if workload == "celeba64" else METRIC


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (weak scaling); 0 = workload default")
    ap.add_argument("--workload", default="cifar10", choices=["cifar10", "celeba64", "cifar10_cfg"],
                    help="cifar10 = BASELINE configs[1] (headline); celeba64 = configs[3]; "
                         "cifar10_cfg = configs[4] (classifier-free guidance, two passes per step)")
    ap.add_argument("--batch-total", type=int, default=0,
                    help="fixed TOTAL batch sharded over the GPUs (strong scaling; BASELINE configs[2]: 2048, "
                         "configs[3]: 512); overrides --batch")
    ap.add_argument("--precision", default="bf16x3", choices=["bf16x3", "bf16", "fp32"],
                    help="tier on the main line (the other tensor-core tier is reported as <tier>_path)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the other tensor-core tier")
    ap.add_argument("--no-gpu-eager", action="store_true", help="skip the PyTorch-eager GPU context baseline")
    ap.add_argument("--state", default="float64", choices=["float32", "float64"],
                    help="sampler state dtype (the reference's state is float64 after the first step)")
    ap.add_argument("--e2e-nfe", type=int, default=NFE, help="0 disables the end-to-end run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-batch", type=int, default=8)
    ap.add_argument("--cpu-steps", type=int, default=2)
    ap.add_argument("--profile-ops", type=int, default=2, help="per-op event timing iterations")
    ap.add_argument("--profiler-range", action="store_true",
                    help="cudaProfilerStart/Stop around the timed steps (for ncu --profile-from-start off)")
    ap.add_argument("--no-graph", dest="graph", action="store_false",
                    help="launch every kernel from the host instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the main tier computed as DIR/<name>.npy: the sampler state after the "
                         "last timed step (rank 0's shard) and the end-to-end samples")
    return ap.parse_args()


DUMP_LIMIT = 64 * 10**6


def dump_outputs(path, arrays, limit=DUMP_LIMIT):
    """Writes every array as ``path/<name>.npy`` in float64 or float32.  When the files would come to
    more than ``limit`` bytes, each keeps a fixed, seeded sample of its leading (batch) rows."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    arrays = {k: v if v.dtype == np.float64 else v.astype(np.float32) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    budget = limit - 4096 * len(arrays)          # room for the .npy headers
    for name, v in arrays.items():
        if total > budget:
            keep = max(1, v.shape[0] * budget // total)
            v = v[np.sort(np.random.default_rng(0).choice(v.shape[0], keep, replace=False))]
        np.save(os.path.join(path, name + ".npy"), v)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm": float(d["hbm_gbs"]), "tf_burst": float(d["bf16_tflops"]),
                "tf_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "src": "measured (MEASURED_PEAKS.json)"}
    return {"hbm": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0,
            "src": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ======================================================================== reference arm (CPU)
def run_cpu_port(cfg, batch, steps, warmup, threads=None, guided=False):
    """Times the oracle port of SSCSSampler.sample on the host cores: `steps` predictor steps
    (one score_fn call + the half-step algebra each) on `batch` samples."""
    import numpy as np
    import torch
    from oracle import psld_oracle as O
    from oracle.weights import fill_state_dict, noise_bank, prior
    from psld_b200 import NCSNpp
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    H = cfg.data.image_size
    shapes = {k: tuple(v.shape) for k, v in NCSNpp(cfg).state_dict().items()}
    sd = fill_state_dict(shapes, 0)
    score = O.OracleScoreFn(cfg, sd)
    if guided:
        score = O.GuidedScoreFn(score, O.OracleScoreFn(cfg, fill_state_dict(shapes, 1)), CFG_WEIGHT)
    ts, n = O.time_grid(cfg)
    u0 = prior((batch, 3, H, H), 0.5, 1)

    def go(k):
        nb = noise_bank(2 * k, (batch, 6, H, H), 2)
        t0 = time.perf_counter()
        O.sscs_sample(cfg, score, u0, ts, k, nb, denoise=False)
        return time.perf_counter() - t0

    if warmup > 0:
        go(warmup)
    dt = go(steps)
    per_step = dt / steps
    return {"value": batch / (NFE * per_step), "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"oracle port of SSCSSampler.sample, {cfg.data.image_size}x{cfg.data.image_size} NCSN++ fp32"
                      f"{' x2 (classifier-free guidance)' if guided else ''}, batch {batch}, "
                      f"{steps} of {NFE} NFE timed after {warmup} warm-up, extrapolated linearly",
            "ms_per_step": per_step * 1e3, "sample_nfe_per_sec": batch / per_step}


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import psld_b200
    cfg_name, _, _, workload_desc = WORKLOADS[args.workload]
    cfg = getattr(psld_b200, cfg_name)()
    batch = args.cpu_batch
    # bound the run: (steps+warmup) CPU steps of ~0.17 s/sample each must end within minutes
    guided = args.workload == "cifar10_cfg"
    per_sample_est = 0.4 if guided else 0.2
    while batch > 1 and (args.steps + args.warmup) * batch * per_sample_est > 240:
        batch //= 2
    r = run_cpu_port(cfg, batch, args.steps, args.warmup, guided=guided)
    line = {"metric": metric_name(args.workload),
            "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": workload_desc, "cpu_batch": batch},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ======================================================================== B200 arm
TIER_DTYPE = {"bf16": "bf16", "fp32": "f32", "bf16x3": "bf16x3"}
TIER_NOTE = {
    "bf16x3": "fp32-tolerance tier: split-bf16 operands, three tcgen05 MMAs per product, fp32 accumulation",
    "bf16": "throughput tier: bf16 operands and activations, fp32 accumulation (~5e-3 trajectory error)",
    "fp32": "true fp32 FFMA on the CUDA cores",
}


def measure_tier(args, precision, ctx):
    """Device-timed steps + per-op roofline + (optionally) the end-to-end run of ONE precision tier."""
    import ctypes as C
    import torch
    import torch.distributed as dist
    from psld_b200 import SSCSSampler, time_grid
    from psld_b200 import _lib as L
    from psld_b200.distributed import gather_samples, max_over_ranks
    from psld_b200.profiling import profile_plan
    from psld_b200.schedule import StepTables

    net, sde, cfg, dev, rank, world, local, pk = (ctx[k] for k in
                                                  ("net", "sde", "cfg", "dev", "rank", "world", "local", "pk"))
    B, H, chw, ts = ctx["B"], ctx["H"], ctx["chw"], ctx["ts"]
    net.set_precision(precision)
    plan = net.plan(B, 1, True)
    lib = L.lib()
    state_dtype = torch.float32 if args.state == "float32" else torch.float64
    state = sde.prior_sampling_device((B, 3, H, H), seed=1 + rank, device=dev).to(state_dtype)
    plan.x_in.copy_(state)
    side = ctx["side"]

    def run_steps(first, count):
        tabs = StepTables(sde, ts[first:first + count + 1], count, "sscs_sde", False, 1e-3,
                          merge_noise=True)
        table = tabs.time_table.to(dev)
        raw = torch.frombuffer(bytearray(C.string_at(C.addressof(tabs.sscs), C.sizeof(tabs.sscs))),
                               dtype=torch.uint8).to(dev)
        counter = torch.zeros(1, dtype=torch.int32, device=dev)
        d = L.SamplerDesc()
        if args.graph:
            d.sscs_dev, d.step_counter = raw.data_ptr(), counter.data_ptr()
        d.sampler, d.n_steps, d.denoise = 0, count, 0
        d.state_dtype = L.dtype_code(state_dtype)
        d.fuse_halves, d.temb_op = 2, plan.temb_op     # one fused pass, one merged draw per step
        d.B, d.chw, d.seed = B, chw, 99 + rank
        d.state, d.net_in, d.eps = state.data_ptr(), plan.x_in.data_ptr(), plan.eps.data_ptr()
        d.time_table = table.data_ptr()
        d.sscs = C.cast(tabs.sscs, C.POINTER(L.SscsCoeffs))
        L.check(lib.psld_sampler_run(plan.op_array, plan.n_ops, C.byref(d),
                                     C.c_void_p(side.cuda_stream)), "sampler_run")
        return table, tabs, raw, counter

    torch.cuda.synchronize(dev)
    with torch.cuda.stream(side):
        keep = run_steps(0, max(args.warmup, 3))
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    clocks = ClockSampler(local).start() if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    if args.profiler_range:             # ncu --profile-from-start off: capture exactly the timed steps
        torch.cuda.cudart().cudaProfilerStart()
    with torch.cuda.stream(side):
        e0.record()                     # events on the stream the kernels are launched on
        keep2 = run_steps(args.warmup, args.steps)
        e1.record()
    torch.cuda.synchronize(dev)
    if args.profiler_range:
        torch.cuda.cudart().cudaProfilerStop()
    if world > 1:
        dist.barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1), dev)
    clk = clocks.stop() if clocks is not None else None
    # copied now: the update roofline below runs the update kernel in place on `state`
    outputs = {"state": state.cpu().numpy()} if args.dump_outputs else {}
    ms_per_step = ms_total / args.steps
    value = B * world / (NFE * ms_per_step * 1e-3)
    # first-half-step launch + per step (program + fused update)
    launches = 1 + args.steps * (plan.launches + 1 + (1 if args.graph else 0))
    finite = bool(torch.isfinite(state).all().item())

    # ---- per-kernel roofline: per-op CUDA-event times give every kernel's SHARE of a step; the
    # achieved rate is the algorithmic work over (share x the graph-replayed step time), so it can
    # never exceed what the driver-checked step time allows
    prof = profile_plan(plan, iters=max(1, args.profile_ops)) if args.profile_ops > 0 else {}
    conv_classes = prof.pop("_conv_classes", {})
    roof = None
    total_ms = sum(v["ms"] for v in prof.values()) if prof else 0.0
    tc_names = [k for k in ("conv_tc", "conv_tc_gn") if k in prof]
    mult = 3 if precision == "bf16x3" else 1       # bf16 MMAs executed per algorithmic product
    if tc_names:
        flops = sum(prof[k]["flops"] for k in tc_names)         # algorithmic, zero padding excluded
        ev_ms = sum(prof[k]["ms"] for k in tc_names)
        nl = sum(prof[k]["n"] for k in tc_names)
        share = ev_ms / total_ms
        ms_in_step = share * ms_per_step
        ach = flops / (ms_in_step * 1e-3) / 1e12
        traffic, tsrc = None, None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp) and B == 256 and args.workload == "cifar10":
            tj = json.load(open(tp)).get(precision, {})
            ks = [tj["kernels"][k] for k in ("conv_tc_kernel", "conv_gn_tc_kernel", "conv_gn_x3_kernel")
                  if k in tj.get("kernels", {})]
            if ks:
                traffic = sum(k["traffic_bytes_per_launch"] * k["launches"] for k in ks) / sum(k["launches"] for k in ks)
                tsrc = tj["source"]
        roof = {"bound": "tensor",
                "kernel": "conv_tc_kernel" + ((" + conv_gn_x3_kernel" if precision == "bf16x3" else " + conv_gn_tc_kernel")
                                             if "conv_tc_gn" in prof else "") +
                          " (tcgen05 implicit-GEMM convolutions, " + TIER_DTYPE[precision] + ")",
                "achieved": ach, "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                "frac": ach / pk["tf_sustained"],
                # bf16x3 executes three bf16 MMAs per algorithmic product (there is no fp32 tensor-core
                # path): `frac` is bounded by 1/3 by construction; the executed rate is what compares
                # with the cuBLAS bf16 peaks (sustained = long power-capped run, burst = short run)
                "executed_mma_per_product": mult, "achieved_executed": ach * mult,
                "frac_executed": ach * mult / pk["tf_sustained"],
                "frac_executed_vs_burst_peak": ach * mult / pk["tf_burst"], "burst_peak": pk["tf_burst"],
                "traffic": traffic, "traffic_unit": "bytes/launch (DRAM read+write, ncu)",
                "traffic_source": tsrc, "algorithmic_flop_per_launch": flops / nl,
                "peak_source": pk["src"] + ", sustained cuBLAS bf16",
                "launches_per_step": nl, "avg_launch_ms": ms_in_step / nl,
                "share_of_step": share, "time_basis": "per-op CUDA-event share x graph-replayed ms_per_step",
                "per_kernel": {k: {"ms": round(prof[k]["ms"], 3), "launches": prof[k]["n"],
                                   "tflops": round(prof[k]["flops"] / (prof[k]["ms"] * 1e-3) / 1e12, 1)}
                               for k in tc_names}}
        tpj = os.path.join(ROOT, "profiles", "tensor_pipe.json")
        if os.path.exists(tpj):        # ncu sm__pipe_tensor_cycles_active captures (committed evidence)
            roof["ncu_tensor_pipe"] = json.load(open(tpj)).get(precision)
    elif "conv_simt" in prof:
        c = prof["conv_simt"]
        ach = c["flops"] / (c["ms"] / total_ms * ms_per_step * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": "conv_simt_kernel (fp32 FFMA)", "achieved": ach,
                "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": ach / pk["tf_sustained"],
                "traffic": None, "peak_source": pk["src"]}

    # ---- end to end through the public API: pinned host prior -> HOST samples
    e2e = None
    if args.e2e_nfe > 0:
        cfg_e = ctx["make_cfg"](batch_size=B, n_samples=B * world, n_discrete_steps=args.e2e_nfe)
        cfg_e.evaluation.sampler["state_dtype"] = args.state
        Se = SSCSSampler(cfg_e, sde, net)
        ts_e, n_e = time_grid(cfg_e)
        host_prior = sde.prior_sampling([B, 3, H, H]).pin_memory()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        out = Se.sample(host_prior, ts_e, n_e, denoise=True, eps=1e-3)
        x = gather_samples(out)                       # single NCCL all-gather of the x half
        host = x.to("cpu", non_blocking=False)
        torch.cuda.synchronize(dev)
        dt = max_over_ranks(time.perf_counter() - t0, dev)
        scale = NFE / float(args.e2e_nfe)
        e2e = {"value": B * world / (dt * scale), "unit": UNIT,
               "h2d_bytes_per_step": int(host_prior.numel() * 4),
               "d2h_bytes_per_step": int(host.numel() * host.element_size()),
               "seconds": dt, "nfe": args.e2e_nfe, "api": "SSCSSampler.sample + gather_samples",
               "finite": bool(torch.isfinite(host).all().item())}
        if args.dump_outputs:
            outputs["samples"] = host.numpy()
    return {"precision": precision, "dtype": TIER_DTYPE[precision], "note": TIER_NOTE[precision],
            "value": value, "ms_per_step": ms_per_step, "e2e": e2e, "roofline": roof, "clocks": clk,
            "gpu_launches": launches, "finite": finite, "engines": dict(plan.engine_count),
            "tensor_frac_of_step": (ctx["flop"] * B / (ms_per_step * 1e-3) / 1e12) / pk["tf_sustained"],
            "per_kernel_ms": {k: round(v["ms"] / total_ms * ms_per_step, 4) for k, v in prof.items()},
            "conv_classes": {k: {"n": v["n"], "ms": round(v["ms"], 4), "tflops": round(v["tflops"], 1)}
                             for k, v in sorted(conv_classes.items(), key=lambda kv: -kv[1]["ms"])},
            "_state": state, "_plan": plan, "_outputs": outputs}


def gpu_eager_baseline(cfg, sde_cfg_B, dev, steps=2):
    """Context, never the target: the reference's algorithm as PLAIN PyTorch-eager CUDA code on the same
    B200 (the oracle port's ``ncsnpp_forward`` + SSCS algebra with ``.cuda()`` tensors: cuDNN / cuBLAS
    through ATen, FIR through the pure-ATen ``upfirdn2d``), fp32, device-timed."""
    import torch
    from oracle import psld_oracle as O
    from oracle.weights import fill_state_dict, noise_bank, prior
    from psld_b200 import NCSNpp
    B = sde_cfg_B
    H = cfg.data.image_size
    shapes = {k: tuple(v.shape) for k, v in NCSNpp(cfg).state_dict().items()}
    sd = {k: v.to(dev) for k, v in fill_state_dict(shapes, 0).items()}
    score = lambda u, t: O.ncsnpp_forward(cfg, sd, u, t.to(u.device))
    ts, n = O.time_grid(cfg)
    u0 = prior((B, 3, H, H), 0.5, 1).to(dev)
    out = {}
    for name, tf32 in (("tf32_convs_torch_default", True), ("strict_fp32", False)):
        torch.backends.cudnn.allow_tf32 = tf32
        torch.backends.cuda.matmul.allow_tf32 = False
        nb = [z.to(dev) for z in noise_bank(2 * (steps + 1), (B, 6, H, H), 2)]
        with torch.no_grad():
            O.sscs_sample(cfg, score, u0, ts, 1, nb, denoise=False)
            torch.cuda.synchronize(dev)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            O.sscs_sample(cfg, score, u0, ts, steps, nb, denoise=False)
            b.record()
            torch.cuda.synchronize(dev)
        ms = a.elapsed_time(b) / steps
        out[name] = {"value": B / (NFE * ms * 1e-3), "unit": UNIT, "ms_per_step": ms}
    torch.backends.cudnn.allow_tf32 = True
    out["what"] = (f"oracle port (plain PyTorch eager, fp32) of NCSN++ forward + SSCS algebra on cuda, batch {B}, "
                   f"{steps} steps after 1 warm-up, extrapolated linearly to {NFE} NFE")
    return out


def main_b200(args):
    import torch
    import torch.distributed as dist
    from psld_b200 import NCSNpp, PSLD, time_grid
    from psld_b200 import _lib as L
    from psld_b200.distributed import env_rank

    rank, world, local = env_rank()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    pk = peaks()
    import psld_b200
    cfg_name, flop_per_sample_nfe, default_batch, workload_desc = WORKLOADS[args.workload]
    make_cfg = getattr(psld_b200, cfg_name)
    scaling = "weak"
    if args.batch_total > 0:             # fixed total batch sharded over the ranks (BASELINE configs[2]/[3])
        if args.batch_total % world:
            raise SystemExit(f"--batch-total {args.batch_total} is not divisible by {world} GPUs")
        args.batch = args.batch_total // world
        scaling = "strong"
    elif args.batch <= 0:
        args.batch = default_batch
    cfg = make_cfg(batch_size=args.batch, n_samples=args.batch * world)
    cfg.evaluation.sampler["state_dtype"] = args.state
    torch.manual_seed(1234)
    net = NCSNpp(cfg).eval().to(dev)   # random-init weights
    guided = args.workload == "cifar10_cfg"
    if guided:                         # two networks, two passes per step (BASELINE configs[4])
        from psld_b200 import ClassifierFreeGuidance
        net = ClassifierFreeGuidance(cond=net, uncond=NCSNpp(cfg).eval().to(dev), weight=CFG_WEIGHT)
    sde = PSLD(cfg)
    B = args.batch
    H = cfg.data.image_size
    ts, n = time_grid(cfg)
    ctx = dict(net=net, sde=sde, cfg=cfg, dev=dev, rank=rank, world=world, local=local, pk=pk, B=B, H=H,
               chw=3 * H * H, ts=ts, side=torch.cuda.Stream(dev), make_cfg=make_cfg, flop=flop_per_sample_nfe)

    main = measure_tier(args, args.precision, ctx)
    lib = L.lib()
    state_dtype = torch.float32 if args.state == "float32" else torch.float64
    # fused phase-space update alone (HBM-bound), timed at this batch
    def _update_roofline(sd):
        st = main["_state"] if sd == state_dtype else main["_state"].to(sd)
        u = time_update(lib, st, main["_plan"], B, 3 * H * H, L.stream_ptr(dev), dev, sd, sde, ts)
        u["peak"] = pk["hbm"]
        u["frac"] = u["achieved"] / pk["hbm"]
        u["state_dtype"] = "float64" if sd == torch.float64 else "float32"
        if "achieved" in u.get("large", {}):
            u["large"]["frac"] = u["large"]["achieved"] / pk["hbm"]
        return u

    upd = _update_roofline(state_dtype)
    other_sd = torch.float32 if state_dtype == torch.float64 else torch.float64
    upd["other_state_dtype"] = _update_roofline(other_sd)      # the throughput / reference-faithful twin

    # ---- the other tensor-core tier, stated separately (north_star: "the bf16 score_fn path stated
    # separately"): same workload, same measurement, its own roofline and end-to-end number
    other = None
    sec = {"bf16x3": "bf16", "bf16": "bf16x3"}.get(args.precision)
    if sec and not args.no_secondary:
        o = measure_tier(args, sec, ctx)
        other = {k: o[k] for k in ("precision", "dtype", "note", "value", "ms_per_step", "e2e", "roofline",
                                   "gpu_launches", "finite", "tensor_frac_of_step", "per_kernel_ms",
                                   "conv_classes", "clocks")}

    cpu = eager = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = run_cpu_port(make_cfg(), args.cpu_batch, args.cpu_steps, 1, guided=guided)
        cpu = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}
    if rank == 0 and world == 1 and not args.no_gpu_eager and not guided:
        try:
            eager = gpu_eager_baseline(make_cfg(), min(B, 64), dev)
        except Exception as e:      # context only: never fail the bench line on it
            eager = {"error": f"{type(e).__name__}: {str(e)[:120]}"}

    if rank == 0:
        line = {
            "metric": metric_name(args.workload),
            "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None,
            "dtype": main["dtype"], "data": "synthetic",
            "config": {
                "workload": workload_desc,
                "batch_per_gpu": B, "batch_total": B * world, "nfe_per_sample": NFE,
                "precision_tier": args.precision + ": " + main["note"],
                "state_dtype": args.state, "noise": "in-kernel Philox4x32-10",
                "step": "one SSCS predictor step = 1 score_fn call + 1 fused update",
                "cuda_graph": bool(args.graph),
                "l2": "activations per step (GBs at B=256) exceed the 126 MB L2; no flush needed",
                "parallelism": f"batch-sharded x{world}, no per-step communication, one final NCCL all-gather",
            },
            "clocks": main["clocks"], "e2e": main["e2e"], "gpu_launches": main["gpu_launches"],
            "roofline": main["roofline"], "roofline_update": upd, "cpu_baseline": cpu,
            "gpu_eager_baseline": eager,
            "tensor_frac_of_step": main["tensor_frac_of_step"],
            "per_kernel_ms": main["per_kernel_ms"],
            "engines": main["engines"], "finite": main["finite"],
            "conv_classes": main["conv_classes"],
        }
        if other is not None:
            line[other["precision"] + "_path"] = other
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, main["_outputs"])
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def time_update(lib, state, plan, B, chw, stream, dev, state_dtype, sde, ts, big_pairs=1 << 24):
    """Fused per-step update (score step + both half-steps, one merged Philox draw) alone, CUDA
    events: at the bench batch (latency-bound: ~25 MB) and at >= 2^24 pairs (bandwidth-bound)."""
    import ctypes as C
    import torch
    from psld_b200 import _lib as L
    from psld_b200.schedule import StepTables
    tabs = StepTables(sde, ts[:3], 2, "sscs_sde", False, 1e-3, merge_noise=True)
    sdt = L.dtype_code(state_dtype)
    stages = L.STAGE_SCORE | L.STAGE_HALF_B
    sb = 8 if state_dtype == torch.float64 else 4
    per_pair = 2 * sb * 2 + 8 + 8          # state in+out, eps in, fp32 net_in out (Philox noise)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def measure(st, xin, eps, Bq, reps=10):
        sp, ip, ep = L.ptr(st), L.ptr(xin), L.ptr(eps)
        total = 0.0
        for r in range(reps + 2):
            flush.zero_()                               # evict L2 between timed launches
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            L.check(lib.psld_sscs_update(sp, sp, sdt, ip, ep, None, None, None, C.byref(tabs.sscs[0]),
                                         stages, 5, r, Bq, chw, stream), "update")
            b.record()
            torch.cuda.synchronize(dev)
            if r >= 2:
                total += a.elapsed_time(b)
        return total / reps

    ms = measure(state, plan.x_in, plan.eps, B)
    out = {"bound": "hbm", "kernel": "sscs_update_kernel (score step + merged half-steps, Philox)",
           "achieved": per_pair * B * chw / (ms * 1e-3) / 1e9, "unit": "GB/s",
           "bytes_per_pair": per_pair, "pairs": B * chw, "avg_launch_ms": ms,
           "l2": "256 MB flush between launches", "traffic": None}
    Bb = max(B, -(-big_pairs // chw))
    try:
        st = torch.randn(Bb, 6, chw // 3, dtype=torch.float32, device=dev).to(state_dtype)
        xin = torch.empty(Bb, 6, chw // 3, dtype=torch.float32, device=dev)
        eps = torch.randn(Bb, 6, chw // 3, dtype=torch.float32, device=dev)
        msb = measure(st, xin, eps, Bb, reps=5)
        out["large"] = {"pairs": Bb * chw, "avg_launch_ms": msb,
                        "achieved": per_pair * Bb * chw / (msb * 1e-3) / 1e9}
    except RuntimeError as e:   # pragma: no cover
        out["large"] = {"error": str(e)[:80]}
    return out


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        main_reference(a)
    else:
        main_b200(a)
