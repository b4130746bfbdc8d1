"""Device-timed attention over 1024 and 4096 tokens, and the SSCS step of a 64x64 net with attention at
64, 32 and 16, in both tensor-core tiers.

Reports, per tier:
  * the attention op with its fused output projection (PSLD_OP_ATTN, PROJ = 1) at HW = 1024, C = 256
    and HW = 4096, C = 128, batch 64: time per op (CUDA events over repeated launches) and TFLOP/s
    from algorithmic FLOPs, 4 N HW^2 C for the attention plus 2 N HW C^2 for the projection;
  * the same HW = 1024 attention on the CUDA-core engine (PROJ = 0, 4 N HW^2 C), timed alternately
    with the tensor-core op in the same process.  Before the key-streaming kernel this was the only
    engine for 1024 tokens;
  * the SSCS step time of the CelebA-64 NCSN++ with attn_resolutions = [64, 32, 16] (CUDA events
    around a run of the native sampler loop).
The working set of each op (q|k|v, residual, output: 100 to 400 MB) is larger than the 126 MB L2.
The card's name and power limit are read in the same run.

    python scripts/bench_attention.py [--batch 64] [--reps 20] [--steps 10] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from oracle.weights import fill_state_dict, prior  # noqa: E402
from psld_b200 import NCSNpp, PSLD, SSCSSampler, celeba64_config, time_grid  # noqa: E402
from psld_b200 import _lib as L  # noqa: E402
from bench_highres import card  # noqa: E402


class AttnOp:
    """One PSLD_OP_ATTN record on random device buffers, prepared for the given engine."""

    def __init__(self, N, HW, C, fmt, engine, proj, seed=0):
        g = torch.Generator(device="cuda")
        g.manual_seed(seed)
        m = 2 if fmt == L.BF16S else 1
        rnd = lambda *s: torch.randn(*s, generator=g, device="cuda").to(torch.bfloat16)
        self.keep = [rnd(N, HW, 3 * C * m), torch.empty(N, HW, C * m, dtype=torch.bfloat16, device="cuda")]
        op = L.Op()
        op.kind, op.engine = L.OP_ATTN, engine
        op.i[L.ATTN_N], op.i[L.ATTN_HW], op.i[L.ATTN_C], op.i[L.ATTN_DTYPE] = N, HW, C, fmt
        op.f[0] = float(C ** -0.5)
        op.inp[0], op.out[0] = self.keep[0].data_ptr(), self.keep[1].data_ptr()
        if proj:
            w = rnd(m * C, C) * (C ** -0.5)
            b = torch.zeros(C, device="cuda")
            x = rnd(N, HW, C * m)
            st = torch.zeros(N, C // 4, 2, dtype=torch.float64, device="cuda")
            self.keep += [w, b, x, st]
            op.i[L.ATTN_PROJ] = 1
            op.f[1] = 0.7071
            op.inp[1], op.inp[2], op.inp[3], op.out[1] = w.data_ptr(), b.data_ptr(), x.data_ptr(), st.data_ptr()
        self.op, self.lib = op, L.lib()
        if engine == L.ENGINE_TC:
            L.check(self.lib.psld_op_prepare(ctypes.byref(op)), "psld_op_prepare(attn)")
        self.flops = 4.0 * N * HW * HW * C + (2.0 * N * HW * C * C if proj else 0.0)

    def run(self, reps):
        s = L.stream_ptr()
        for _ in range(reps):
            L.check(self.lib.psld_op_run(ctypes.byref(self.op), s), "psld_op_run(attn)")

    def time_ms(self, reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        self.run(reps)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    def release(self):
        self.lib.psld_op_release(ctypes.byref(self.op))


def _entry(ms_list, flops):
    ms = min(ms_list)
    return {"ms": round(ms, 4), "ms_all_rounds": [round(v, 4) for v in ms_list],
            "tflops": round(flops / (ms * 1e-3) / 1e12, 1), "gflop": round(flops / 1e9, 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--reps", type=int, default=20, help="launches per timed window")
    ap.add_argument("--rounds", type=int, default=3, help="alternating timed windows per op")
    ap.add_argument("--steps", type=int, default=10, help="timed SSCS steps of the network")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    B = args.batch
    res = {"workload": f"attention op B={B}; CelebA-64 NCSN++ attn [64,32,16] SSCS B={B}", "card": card(),
           "tiers": {}}
    for tier, fmt in (("bf16x3", L.BF16S), ("bf16", L.BF16)):
        ops = {"hw1024_c256_tc_proj": AttnOp(B, 1024, 256, fmt, L.ENGINE_TC, True),
               "hw1024_c256_simt": AttnOp(B, 1024, 256, fmt, L.ENGINE_SIMT, False),
               "hw4096_c128_tc_proj": AttnOp(B, 4096, 128, fmt, L.ENGINE_TC, True)}
        for o in ops.values():
            o.run(2)                                   # warm-up: module load, first launches
        torch.cuda.synchronize()
        times = {k: [] for k in ops}
        for _ in range(args.rounds):                  # alternate the engines within one process
            for k, o in ops.items():
                times[k].append(o.time_ms(args.reps if "simt" not in k else max(2, args.reps // 4)))
        t = {k: _entry(v, ops[k].flops) for k, v in times.items()}
        t["hw1024_c256_tc_vs_simt_speedup"] = round(t["hw1024_c256_simt"]["ms"] / t["hw1024_c256_tc_proj"]["ms"], 1)
        for o in ops.values():
            o.release()
        del ops
        torch.cuda.empty_cache()
        res["tiers"][tier] = {"attention_op": t}

    cfg = celeba64_config(n_discrete_steps=args.steps + 1, batch_size=B, n_samples=B)
    cfg.model.score_fn.update(attn_resolutions=[64, 32, 16])
    net = NCSNpp(cfg).eval()
    net.load_state_dict(fill_state_dict({k: tuple(v.shape) for k, v in net.state_dict().items()}, 0))
    net = net.cuda()
    ts, n = time_grid(cfg)
    u0 = prior((B, 3, 64, 64), 0.5, 1).cuda()
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
        plan = net.plan(B, 1, True)
        res["tiers"][tier]["attn64_net_sscs"] = {
            "sscs_step_ms": round(a.elapsed_time(b) / n, 3), "steps_timed": n,
            "finite": bool(torch.isfinite(out).all()), "engines": plan.engine_count}
        del S
        net.invalidate()
        torch.cuda.empty_cache()
    res["card_after"] = card()
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
