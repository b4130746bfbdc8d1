"""Device-timed SSCS step of the 256x256 NCSN++ (nf=128, ch_mult [1,1,2,2,2,2,2], 2 blocks, attention
at 16, fir, Fourier features, output_skip + input_skip + sum) in both tensor-core tiers.

Reports, per tier: the SSCS step time (CUDA events around a run of the native sampler loop), the
per-kernel time of one forward by family (psld_b200.profiling), the conv-family TFLOP/s from
algorithmic FLOPs, and the forward time with and without the 256-pixel-wide conv_tc tiles (the
variant routes every convolution with 256-wide output rows to the CUDA cores, as the library did
before it had those tiles).  The card's name and power limit are read in the same run.

    python scripts/bench_highres.py [--batch 32] [--steps 10] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from oracle.weights import fill_state_dict, prior  # noqa: E402
from psld_b200 import NCSNpp, PSLD, SSCSSampler, make_config, time_grid  # noqa: E402
from psld_b200.profiling import profile_plan  # noqa: E402
from psld_b200.program import Plan  # noqa: E402


def config(batch, steps):
    return make_config(image_size=256, score_fn=dict(
        nf=128, ch_mult=[1, 1, 2, 2, 2, 2, 2], num_res_blocks=2, attn_resolutions=[16], dropout=0.0,
        fir=True, progressive="output_skip", progressive_input="input_skip", progressive_combine="sum",
        embedding_type="fourier"), evaluation=dict(sampler="sscs_sde", n_discrete_steps=steps + 1,
                                                   batch_size=batch, n_samples=batch))


class Ow128Plan(Plan):
    """The same program with conv_tc limited to output rows of at most 128 pixels."""

    def op_conv(self, x1, x2, w, bias, **kw):
        if not kw.get("in_nchw") and kw.get("affine") is None and x1.shape[2] > 128 and kw.get("stride", 1) == 1:
            kw["allow_tc"] = False
        return super().op_conv(x1, x2, w, bias, **kw)

    def _ext_fusable(self, b, e1, e2, cout):
        return b.shape[2] <= 128 and super()._ext_fusable(b, e1, e2, cout)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:          # the tool may be missing: say so rather than guess
        q = f"unavailable ({type(e).__name__})"
    return {"name": name, "power_limit_and_max_sm_clock": q}


def time_forward(plan, iters):
    for _ in range(2):
        plan.run()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        plan.run()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--steps", type=int, default=10, help="timed SSCS steps (plus one warm-up run)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    B = args.batch
    cfg = config(B, args.steps)
    net = NCSNpp(cfg).eval()
    net.load_state_dict(fill_state_dict({k: tuple(v.shape) for k, v in net.state_dict().items()}, 0))
    net = net.cuda()
    ts, n = time_grid(cfg)
    u0 = prior((B, 3, 256, 256), 0.5, 1).cuda()      # [B, 6, H, W] phase-space prior draw
    res = {"workload": f"NCSN++ 256x256 output_skip+input_skip, SSCS, B={B}", "card": card(), "tiers": {}}
    for tier in ("bf16x3", "bf16"):
        net.set_precision(tier)
        S = SSCSSampler(cfg, PSLD(cfg), net)
        S.sample(u0.clone(), ts.cuda(), n, denoise=False, eps=cfg.evaluation.eval_eps)      # warm-up, plan build
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = S.sample(u0.clone(), ts.cuda(), n, denoise=False, eps=cfg.evaluation.eval_eps)
        b.record()
        torch.cuda.synchronize()
        step_ms = a.elapsed_time(b) / n
        plan = net.plan(B, 1, True)
        prof = profile_plan(plan, iters=3, warmup=1)
        prof.pop("_conv_classes")
        conv_ms = sum(v["ms"] for k, v in prof.items() if k.startswith("conv"))
        conv_flops = sum(v["flops"] for k, v in prof.items() if k.startswith("conv"))
        fwd_ms = time_forward(plan, 5)
        with torch.no_grad():
            p128 = Ow128Plan(net, B, 1, True)
        fwd128_ms = time_forward(p128, 3)
        prof128 = profile_plan(p128, iters=1, warmup=1)
        prof128.pop("_conv_classes")
        res["tiers"][tier] = {
            "sscs_step_ms": round(step_ms, 3), "steps_timed": n, "finite": bool(torch.isfinite(out).all()),
            "forward_ms": round(fwd_ms, 3),
            "per_kernel_ms": {k: round(v["ms"], 3) for k, v in sorted(prof.items())},
            "launches": {k: v["n"] for k, v in sorted(prof.items())},
            "engines": plan.engine_count,
            "conv_tflops": round(conv_flops / (conv_ms * 1e-3) / 1e12, 1),
            "conv_gflop_per_forward": round(conv_flops / 1e9, 1),
            "ow128_only": {"forward_ms": round(fwd128_ms, 3), "engines": p128.engine_count,
                           "per_kernel_ms": {k: round(v["ms"], 3) for k, v in sorted(prof128.items())}},
        }
        p128.release()
        del p128, S
        net.invalidate()
        torch.cuda.empty_cache()
    res["card"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
