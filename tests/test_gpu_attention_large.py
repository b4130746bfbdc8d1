"""GPU: attention at 32x32 maps and larger.

  * the key-streaming tensor-core attention (attn_stream_tc.cu) in both tensor-core tiers at HW = 512,
    1024, 4096 (and 16384 at N = 1), every C in {64, 128, 192, 256}, with and without the fused
    projection, N = 1, odd, and several waves of CTAs, against the fp64 reference of tests/emulate.py
    with the checker of test_gpu_program_ops.py; q is scaled x4 (steep rows whose maximum jumps from
    tile to tile) and key channel 0 ramps with the key index, so the row maximum of the even queries
    sits in the last key tiles and the online rescale runs;
  * the CUDA-core attention over more keys than one shared-memory score row holds (1600, 4096
    tokens) in all three activation formats, and bitwise equality with stored outputs of the
    single-pass kernel for shapes that fit one row;
  * a seeded sweep over the newly accepted tensor-core shapes (each case passes or is rejected with
    PSLD_EUNSUPPORTED, as the planner's mirror predicts);
  * a 64x64 net with attention at 64, 32 and 16: forward vs the fp64 oracle in all three tiers with the
    CelebA-64 forward gates, no CUDA-core attention in the tensor-core tiers, every distinct op of its
    programs through the checker, a 20-NFE SSCS trajectory vs the oracle sampler and CUDA-graph replay
    vs the host loop.

Regenerate tests/golden/attn_simt_single_pass.npz with the build whose outputs it pins:
    python tests/test_gpu_attention_large.py --write-golden tests/golden/attn_simt_single_pass.npz
"""
import ctypes
import math
import os
import sys

import numpy as np
import pytest
import torch

import test_gpu_program_ops as T
from _net import make_net, sampler_inputs
from _ops import max_rel, rel_l2
from oracle import psld_oracle as O
from psld_b200 import celeba64_config, time_grid
from psld_b200 import _lib as L
from psld_b200.program import Plan, build_plan
from test_gpu_sampler import _run

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "attn_simt_single_pass.npz")
TIERS = {"bf16x3": L.BF16S, "bf16": L.BF16}
FWD_GATES = {"fp32": 2e-5, "bf16x3": 5e-5, "bf16": 2e-2}     # CelebA-64 forward (test_gpu_network.py)


# ------------------------------------------------------------------------------------- op records
def attn_op(N, HW, C, fmt, proj=False, engine=L.ENGINE_TC):
    fake = iter(range(0x10000, 0x10000 + 64 * 16, 64))
    op = L.Op()
    op.kind, op.engine = L.OP_ATTN, engine
    op.i[L.ATTN_N], op.i[L.ATTN_HW], op.i[L.ATTN_C], op.i[L.ATTN_DTYPE] = N, HW, C, fmt
    op.f[0] = float(C ** -0.5)
    op.inp[0], op.out[0] = next(fake), next(fake)
    if proj:
        op.i[L.ATTN_PROJ] = 1
        op.f[1] = 0.7071
        op.inp[1], op.inp[2], op.inp[3], op.out[1] = next(fake), next(fake), next(fake), next(fake)
    return op


def steep_qkv(v, C):
    """q x4; key channel 0 = 3 sqrt(C) * key index / (HW - 1); q channel 0 = 4 on even queries, which
    adds a logit ramp of 0..12 over the keys, so their largest key sits in the last tiles."""
    v = v.clone()
    HW = v.shape[1]
    v[..., :C] *= 4.0
    v[..., C] = torch.linspace(0.0, 3.0 * math.sqrt(C), HW, dtype=v.dtype, device=v.device)
    v[:, 0::2, 0] = 4.0
    return v


@pytest.fixture
def steep_inputs(monkeypatch):
    """check_op of test_gpu_program_ops with the q|k|v input of an attention op passed through
    steep_qkv.  Yields a setter for the current op."""
    cur = {}
    encode = T.encode

    def enc(v, sp):
        if cur and sp.shape == cur["shape"] and sp.role == "act":
            v = steep_qkv(v, cur["C"])
        return encode(v, sp)

    def use(op):
        cur["shape"] = (op.i[L.ATTN_N], op.i[L.ATTN_HW], 3 * op.i[L.ATTN_C])
        cur["C"] = op.i[L.ATTN_C]

    monkeypatch.setattr(T, "encode", enc)
    return use


@pytest.fixture
def steep_gates(monkeypatch):
    """Gates of test_gpu_program_ops.py for the steep inputs.  Logits there reach about 100 instead of
    about 10, and the absolute error of a logit grows with its size: with fp32 rounding in the
    CUDA-core kernels, and with the dropped lo*lo product of the split-bf16 tensor-core operands.
    The error does not grow with the number of keys (512 to 16384 measure alike), and the single-pass
    kernels show it too: on these inputs the single-pass CUDA-core kernel at 1024 tokens measures
    elem 5.4e-5 in split bf16, and attn_tc at 256 tokens in bf16x3 max 1.4e-4, elem 5.8e-4.  Worst
    per-sample values measured on a B200 (1000 W power limit), gates at most 2x measured:
      fp32           l2 4.1e-6  max 1.5e-5  elem 8.7e-5
      bf16x3 memory  l2 4.7e-6  max 1.3e-5  elem 5.9e-5
      bf16x3 attn    l2 1.8e-5  max 1.4e-4  elem 8.0e-4   (stat 4.3e-6)
    The bf16 classes keep their gates (measured bf16 attn: l2 1.8e-3, max 3.8e-3, elem 1.0e-2)."""
    g = dict(T.GATES)
    g["fp32"] = (8e-6, 3e-5, 0.0, 1.7e-4, None)
    g["bf16x3 memory"] = (1e-5, 3e-5, T.SP, 1.1e-4, None)
    g["bf16x3 attn"] = (2e-5, 2.8e-4, T.SP, 1.6e-3, 3e-5)
    monkeypatch.setattr(T, "GATES", g)


def _check(op, fmt, seed, use):
    use(op)
    res = T.check_op(op, fmt, seed)
    assert res is not None, f"{T.describe(op)} N={op.i[L.ATTN_N]} rejected by psld_op_prepare"
    cls, w, fails = res
    print(f"{T.describe(op):40s} N={op.i[L.ATTN_N]:<4d} proj={op.i[L.ATTN_PROJ]} {cls:13s} l2 {w['l2']:.2e} "
          f"max {w['max']:.2e} elem {w['elem']:.2e} stat {w['stat']:.2e}{'  FAIL' if fails else ''}")
    return [f"{T.describe(op)} N={op.i[L.ATTN_N]} proj={op.i[L.ATTN_PROJ]}: {m}" for m in fails]


def _waves_n(HW):
    """Batch that launches about three waves of one-CTA-per-SM query tiles on 148 SMs."""
    return max(1, (3 * 148 * 128) // HW) | 1


# ------------------------------------------------------------------------------------- tensor cores
@pytest.mark.parametrize("HW", [256, 512, 1024, 4096])      # 256: attn_tc, the all-keys kernel
@pytest.mark.parametrize("tier", ["bf16x3", "bf16"])
def test_stream_attention_vs_fp64_reference(tier, HW, steep_inputs, steep_gates):
    fmt = TIERS[tier]
    ns = (1, 5, _waves_n(HW))
    failures, k = [], 0
    for C in (64, 128, 192, 256):
        for proj in (False, True):
            op = attn_op(ns[k % 3], HW, C, fmt, proj)
            failures += _check(op, fmt, 100 + k, steep_inputs)
            k += 1
            torch.cuda.empty_cache()
    assert not failures, "\n".join(failures[:40])


@pytest.mark.parametrize("tier", ["bf16x3", "bf16"])
def test_stream_attention_16384_tokens(tier, steep_inputs, steep_gates):
    fmt = TIERS[tier]
    failures = _check(attn_op(1, 16384, 128, fmt, True), fmt, 7, steep_inputs)
    torch.cuda.empty_cache()
    assert not failures, "\n".join(failures)


def _sweep_cases(fmt, n=30, seed=4096):
    """Seeded attention records over the shapes the tensor-core engine now takes (HW % 128 == 0 from
    512, C in {64, 128, 192, 256}) and their neighbours it rejects (HW = 384, 576, C = 320)."""
    r = np.random.default_rng(seed + fmt)
    cases = []
    for _ in range(n):
        HW = int(r.choice([384, 512, 576, 640, 768, 1024, 1152, 1536, 2048, 2304, 3072, 4096]))
        C = int(r.choice([64, 128, 192, 256, 256, 320]))
        N = int(r.choice([1, 2, 3, 5, 7, 37]))
        N = max(1, min(N, 40_000 // HW))
        cases.append(attn_op(N, HW, C, fmt, HW % 128 == 0 and r.random() < 0.6))
    return cases


@pytest.mark.parametrize("tier", ["bf16x3", "bf16"])
def test_stream_attention_sweep(tier, steep_inputs, steep_gates):
    fmt = TIERS[tier]
    failures, run = [], 0
    for c, op in enumerate(_sweep_cases(fmt)):
        steep_inputs(op)
        res = T.check_op(op, fmt, seed=3000 + c)
        assert (res is None) == (not Plan._attn_tc_eligible(op.i[L.ATTN_HW], op.i[L.ATTN_C])), T.describe(op)
        if res is None:
            print(f"sweep {tier} #{c:2d} {T.describe(op):40s} N={op.i[L.ATTN_N]}: PSLD_EUNSUPPORTED")
            continue
        run += 1
        cls, w, fails = res
        print(f"sweep {tier} #{c:2d} {T.describe(op):40s} N={op.i[L.ATTN_N]:<3d} proj={op.i[L.ATTN_PROJ]} "
              f"l2 {w['l2']:.2e} max {w['max']:.2e} elem {w['elem']:.2e}{'  FAIL' if fails else ''}")
        failures += [f"#{c} {T.describe(op)} N={op.i[L.ATTN_N]}: {m}" for m in fails]
    assert run >= 15 and not failures, "\n".join(failures[:40])


# ------------------------------------------------------------------------------------- CUDA cores
@pytest.mark.parametrize("fmt", [L.F32, L.BF16, L.BF16S], ids=["fp32", "bf16", "bf16x3"])
@pytest.mark.parametrize("HW,C,N", [(1024, 128, 3), (1600, 320, 2), (4096, 128, 2)])
def test_simt_attention_any_hw_vs_fp64_reference(fmt, HW, C, N, steep_inputs, steep_gates):
    failures = _check(attn_op(N, HW, C, fmt, engine=L.ENGINE_SIMT), fmt, 11, steep_inputs)
    assert not failures, "\n".join(failures)


# (format, HW, C, N): shapes whose score rows fit shared memory run the single-pass kernel
SINGLE_PASS = [(L.F32, 256, 64, 1), (L.F32, 100, 320, 1), (L.BF16, 256, 64, 1), (L.BF16S, 256, 64, 1)]


def _simt_single_pass_outputs():
    """Output bytes of the CUDA-core attention on seeded q|k|v (numpy PCG64), one per SINGLE_PASS case."""
    lib = L.lib()
    out = {}
    for c, (fmt, HW, C, N) in enumerate(SINGLE_PASS):
        v = torch.from_numpy(np.random.default_rng(77 + c).standard_normal((N, HW, 3 * C)) * 1.3).cuda()
        sp_in = T.Spec((N, HW, 3 * C), fmt, "act", None)
        sp_out = T.Spec((N, HW, C), fmt, "out", None)
        qkv = T.encode(v, sp_in).contiguous()
        y = torch.zeros(T.nbytes(sp_out), dtype=torch.uint8, device="cuda")
        op = attn_op(N, HW, C, fmt, engine=L.ENGINE_SIMT)
        op.inp[0], op.out[0] = qkv.data_ptr(), y.data_ptr()
        L.check(lib.psld_op_run(ctypes.byref(op), L.stream_ptr()), "psld_op_run(attn simt)")
        torch.cuda.synchronize()
        out[f"case{c}"] = y.cpu().numpy()
    return out


def test_simt_single_pass_bitwise_unchanged():
    g = np.load(GOLDEN)
    for k, y in _simt_single_pass_outputs().items():
        assert np.array_equal(y, g[k]), k


# ------------------------------------------------------------------------------------- 64x64 network
def attn64_config(**ev):
    cfg = celeba64_config(**ev)
    cfg.model.score_fn.update(attn_resolutions=[64, 32, 16], init_scale=1.0)
    return cfg


_NET = {}


def _net(tier):
    if "net" not in _NET:
        _NET["net"] = make_net(attn64_config(), tier)
    net, sd = _NET["net"]
    net.set_precision(tier)
    return net, sd


def _oracle64(cfg, sd, x, t):
    sd64 = {k: v.detach().to("cuda", torch.float64) for k, v in sd.items()}
    with torch.no_grad():
        return O.ncsnpp_forward(cfg, sd64, x.to("cuda", torch.float64), t.to("cuda", torch.float64))


def test_attn64_forward_vs_oracle_fp64():
    r = np.random.default_rng(5)
    B = 3
    x = torch.from_numpy(r.standard_normal((B, 6, 64, 64)).astype(np.float32))
    t = torch.from_numpy(r.uniform(0.05, 0.95, B).astype(np.float32))
    ref = None
    for tier, gate in FWD_GATES.items():
        net, sd = _net(tier)
        if ref is None:
            ref = _oracle64(net.full_config, sd, x, t)
        plan = net.plan(B, B, False)
        attn = [op for op in plan.op_array if op.kind == L.OP_ATTN]
        assert {op.i[L.ATTN_HW] for op in attn} == {64, 256, 1024, 4096}
        if tier != "fp32":
            assert all(op.engine == L.ENGINE_TC for op in attn), plan.engine_count
        y = net(x.cuda(), t.cuda()).double()
        torch.cuda.synchronize()
        e2, em = rel_l2(y, ref), max_rel(y, ref)
        print(f"64x64 attn [64,32,16] {tier}: rel-L2 {e2:.2e} max {em:.2e} {plan.engine_count}")
        assert torch.isfinite(y).all() and e2 <= gate, (tier, e2)


def test_attn64_program_ops_vs_fp64_reference():
    seen, failures, worst = set(), [], {}
    for tier in ("bf16x3", "bf16", "fp32"):
        net, _ = _net(tier)
        plan = build_plan(net, 2, 1, True)
        keep = {t.data_ptr(): t for t in plan.keep}
        for op in list(plan.op_array):
            sig = T._signature(op)
            if sig in seen:
                continue
            seen.add(sig)
            res = T.check_op(op, T._fmt(plan), seed=len(seen), weights=keep.__getitem__, B=plan.B)
            if res is None:
                failures.append(f"{tier}: {T.describe(op)} rejected by psld_op_prepare")
                continue
            cls, w, fails = res
            T._merge(worst, cls, w)
            print(f"attn64 {tier:7s} {T.describe(op):52s} {cls:13s} l2 {w['l2']:.2e} max {w['max']:.2e}"
                  f"{'  FAIL' if fails else ''}")
            failures += [f"{tier}: {T.describe(op)}: {m}" for m in fails]
        del plan, keep
        torch.cuda.empty_cache()
    T._report([f"64x64 attn [64,32,16]: {len(seen)} distinct op signatures"], worst)
    assert not failures, "\n".join(failures[:40])


class _Oracle64ScoreFn:
    """The oracle forward in float64 on the device (returns fp32 on the host, like OracleScoreFn)."""

    def __init__(self, cfg, sd):
        self.cfg = cfg
        self.sd = {k: v.detach().to("cuda", torch.float64) for k, v in sd.items()}

    def __call__(self, u, t):
        with torch.no_grad():
            y = O.ncsnpp_forward(self.cfg, self.sd, u.to("cuda", torch.float64), t.to("cuda", torch.float64))
        return y.float().cpu()


def test_attn64_sscs_trajectory_vs_oracle():
    cfg = attn64_config(sampler="sscs_sde", n_discrete_steps=20)
    B = 2
    _, n = time_grid(cfg)
    u0, nb = sampler_inputs(cfg, B, n, "sscs_sde")
    net, sd = make_net(cfg, "bf16x3")
    ref = O.sscs_sample(cfg, _Oracle64ScoreFn(cfg, sd), u0, O.time_grid(cfg)[0], n, nb)
    out, _, _ = _run(cfg, net, u0, nb, record=False)
    e2, em = rel_l2(out.cpu(), ref), max_rel(out.cpu(), ref)
    print(f"64x64 attn [64,32,16] SSCS {n}+1 NFE bf16x3: rel-L2 {e2:.2e} max {em:.2e}")
    assert e2 <= 1e-4 and em <= 1e-4, (e2, em)


def test_attn64_graph_replay_equals_host_loop():
    cfg = attn64_config(sampler="sscs_sde", n_discrete_steps=9)
    for tier in ("bf16", "bf16x3"):
        net, _ = make_net(cfg, tier)
        u0, _ = sampler_inputs(cfg, 3, 8, "sscs_sde")
        a, _, _ = _run(cfg, net, u0, None, record=False, graph=False)
        b, _, _ = _run(cfg, net, u0, None, record=False, graph=True)
        assert torch.isfinite(a).all() and torch.equal(a, b), tier


if __name__ == "__main__" and "--write-golden" in sys.argv:
    path = sys.argv[sys.argv.index("--write-golden") + 1]
    np.savez(path, **_simt_single_pass_outputs())
    print("wrote", path)
