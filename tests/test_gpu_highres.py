"""GPU: NCSN++ with the output-skip / input-skip pyramids (progressive=output_skip,
progressive_input=input_skip, combine=sum) and the 256-pixel-wide tensor-core convolutions.

  * forward of tiny / mid nets vs the reference forward of tests/_pyramid.py in float64 on the device, every pyramid combination,
    fir on / off, Fourier / positional embedding, all three precision tiers;
  * the 128x128 and 256x256 configurations of the score-SDE family at B = 2: no convolution on the
    CUDA cores in either tensor-core tier, and every distinct op of their programs vs the fp64
    reference of tests/emulate.py (+ the head residual, tests/_pyramid.py) with the checker of test_gpu_program_ops.py;
  * a seeded sweep of OW = 256 conv_tc records (and NCHW heads with a residual);
  * a 20-NFE SSCS trajectory vs the oracle sampler, and CUDA-graph replay vs the host loop.
"""
import numpy as np
import pytest
import torch

import _pyramid
import emulate
import test_gpu_program_ops as T
from _net import make_net, sampler_inputs
from _ops import max_rel, rel_l2
from oracle import psld_oracle as O
from psld_b200 import PSLD, SSCSSampler, make_config, mid_config, time_grid, tiny_config
from psld_b200 import _lib as L
from psld_b200.program import Plan, build_plan
from test_gpu_sampler import _run

pytestmark = pytest.mark.gpu

GATES = {"fp32": 1e-5, "bf16x3": 1e-4, "bf16": 3e-2}
COMBOS = [("input_skip", "none"), ("none", "output_skip"), ("input_skip", "output_skip")]


def _pyramid_cfg(base, pin, prog, fir=True, emb="fourier", **ev):
    cfg = base(**ev)
    cfg.model.score_fn.update(progressive_input=pin, progressive=prog, progressive_combine="sum", fir=fir,
                              embedding_type=emb, init_scale=1.0)
    return cfg


def highres_config(size):
    """The 128x128 / 256x256 NCSN++ of the score-SDE family (fir, Fourier features, output_skip +
    input_skip + sum) on the PSLD state (6 channels)."""
    ch_mult = {128: [1, 2, 2, 2, 4], 256: [1, 1, 2, 2, 2, 2, 2]}[size]
    return make_config(image_size=size, score_fn=dict(
        nf=128, ch_mult=ch_mult, num_res_blocks=2, attn_resolutions=[16], dropout=0.0, fir=True,
        progressive="output_skip", progressive_input="input_skip", progressive_combine="sum",
        embedding_type="fourier", init_scale=1.0), evaluation=dict(batch_size=2, n_samples=2))


def _oracle64(cfg, sd, x, t):
    sd64 = {k: v.detach().to("cuda", torch.float64) for k, v in sd.items()}
    with torch.no_grad():
        return _pyramid.ncsnpp_forward(cfg, sd64, x.to("cuda", torch.float64), t.to("cuda", torch.float64))


def _inputs(B, H, seed=0):
    r = np.random.default_rng(seed)
    x = torch.from_numpy(r.standard_normal((B, 6, H, H)).astype(np.float32))
    t = torch.from_numpy(r.uniform(0.05, 0.95, B).astype(np.float32))
    return x, t


@pytest.mark.parametrize("emb", ["fourier", "positional"])
@pytest.mark.parametrize("fir", [True, False])
@pytest.mark.parametrize("pin,prog", COMBOS)
@pytest.mark.parametrize("base", ["tiny", "mid"])
def test_pyramid_forward_vs_oracle_fp64(base, pin, prog, fir, emb):
    cfg = _pyramid_cfg({"tiny": tiny_config, "mid": mid_config}[base], pin, prog, fir, emb)
    net, sd = make_net(cfg, "fp32")
    x, t = _inputs(2, cfg.data.image_size)
    ref = _oracle64(cfg, sd, x, t)
    for tier, gate in GATES.items():
        net.set_precision(tier)
        y = net(x.cuda(), t.cuda()).double()
        torch.cuda.synchronize()
        e2, em = rel_l2(y, ref), max_rel(y, ref)
        print(f"{base} {pin}/{prog} fir={fir} {emb} {tier}: rel-L2 {e2:.2e} max {em:.2e} {net.plan(2, 2, False).engine_count}")
        assert e2 <= gate and em <= gate, (tier, e2, em)


_BIG = {}


def _big_net(size, tier):
    if size not in _BIG:
        _BIG[size] = make_net(highres_config(size), "bf16x3")
    net, sd = _BIG[size]
    net.set_precision(tier)
    return net, sd


@pytest.mark.parametrize("size", [128, 256])
def test_highres_nets_run_on_tensor_cores(size):
    """Full-size configurations at B = 2: no SIMT convolution in either tensor-core tier, and the
    forward agrees with the fp64 oracle."""
    x, t = _inputs(2, size, seed=1)
    ref = None
    for tier in ("bf16x3", "bf16"):
        net, sd = _big_net(size, tier)
        plan = net.plan(2, 2, False)
        print(f"{size}x{size} {tier}: {plan.n_ops} ops, engines {plan.engine_count}")
        # bf16x3: maps of fewer than 32 pixels (the 4x4 level of the 256x256 net) keep the CUDA-core
        # conv, the split-bf16 tensor-core output needs H*W % 32 == 0; everything else is tcgen05
        simt = [op for op in plan.op_array if op.kind == L.OP_CONV and op.engine == L.ENGINE_SIMT]
        assert all(tier == "bf16x3" and op.i[L.CONV_OH] * op.i[L.CONV_OW] < 32 for op in simt), \
            [T.describe(op) for op in simt]
        y = net(x.cuda(), t.cuda()).double()
        if ref is None:
            ref = _oracle64(net.full_config, sd, x, t)
        e2 = rel_l2(y, ref)
        print(f"  rel-L2 vs fp64 oracle {e2:.2e}")
        assert torch.isfinite(y).all() and e2 <= GATES[tier], e2
    _BIG.pop(size, None)
    torch.cuda.empty_cache()


def _head_slot_specs(op):
    """test_gpu_program_ops.slot_specs, plus the fp32 NCHW residual of the network head: [N, V, OH, OW]
    over the V valid output channels (include/psld_b200.h)."""
    s = _slot_specs(op)
    i = op.i
    if op.kind == L.OP_CONV and i[L.CONV_OUT_LAYOUT] == L.NCHW and ("in", 2) in s:
        tc = op.engine in (L.ENGINE_TC, L.ENGINE_TC_GN)
        valid = int(op.f[1]) if tc else i[L.CONV_COUT]
        s["in", 2] = T.Spec((i[L.CONV_N], valid, i[L.CONV_OH], i[L.CONV_OW]), L.F32, "act", None)
    return s


_slot_specs = T.slot_specs


@pytest.fixture
def head_residual_specs(monkeypatch):
    """The checker of test_gpu_program_ops with the NCHW-head residual in its slot layout and reference."""
    monkeypatch.setattr(T, "slot_specs", _head_slot_specs)
    monkeypatch.setattr(T, "reference_op", _pyramid.reference_op)
    monkeypatch.setattr(emulate, "reference_op", _pyramid.reference_op)


@pytest.fixture
def long_contraction_gates(monkeypatch):
    """These nets contract over up to twice the CIFAR-10 lengths (1024-channel conv inputs, K = 9216;
    attention over 512 channels), so the fp32 / split-bf16 accumulation error per op grows by up to
    sqrt(2): the gates of the fp32-tolerance classes are 1.5x those of test_gpu_program_ops.py
    (measured on a B200: conv 8x8 1024->512 rel-L2 2.1e-5, attention c512 elementwise 1.01e-5)."""
    g = dict(T.GATES)
    for cls in ("fp32", "bf16x3 conv", "bf16x3 attn", "bf16x3 memory"):
        l2, mx, a, b, st = g[cls]
        g[cls] = (1.5 * l2, 1.5 * mx, a, 1.5 * b, None if st is None else 1.5 * st)
    monkeypatch.setattr(T, "GATES", g)


@pytest.mark.parametrize("size", [128, 256])
def test_highres_program_ops_vs_fp64_reference(size, head_residual_specs, long_contraction_gates):
    seen, failures, worst = set(), [], {}
    for tier in ("bf16x3", "bf16"):
        net, _ = _big_net(size, tier)
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
            print(f"{size} {tier:7s} {T.describe(op):52s} {cls:13s} l2 {w['l2']:.2e} max {w['max']:.2e}"
                  f"{'  FAIL' if fails else ''}")
            failures += [f"{tier}: {T.describe(op)}: {m}" for m in fails]
        del plan, keep
    _BIG.pop(size, None)
    torch.cuda.empty_cache()
    T._report([f"{size}x{size}: {len(seen)} distinct op signatures"], worst)
    assert not failures, "\n".join(failures[:40])


def _ow256_cases(fmt, n=16, seed=256):
    """Seeded conv_tc records with 256-pixel-wide output rows: 3x3 / 1x1, one or two sources, +temb,
    +residual, the fused 1x1 shortcut, statistics, and the fp32 NCHW head with its residual."""
    r = np.random.default_rng(seed + fmt)
    fake = iter(range(0x10000, 0x10000 + 64 * 1000, 64))
    cases = []
    for c in range(n):
        op = L.Op()
        op.kind, op.engine = L.OP_CONV, L.ENGINE_TC
        i = op.i
        head = c % 4 == 3
        N = int(r.choice([1, 2, 3, 5]))
        OW = 256
        OH = int(r.choice([1, 2, 4, 16, 64, 256]))
        ks = 3 if head else int(r.choice([1, 3]))
        C1 = 64 * int(r.integers(1, 4))
        C2 = 0 if head else 64 * int(r.integers(0, 3))
        cout = 32 if head else 32 * int(r.choice([1, 2, 3, 4, 8]))
        if OH * OW * N > 300_000:
            N = max(1, 300_000 // (OH * OW))
        i[L.CONV_N], i[L.CONV_H], i[L.CONV_W], i[L.CONV_C1], i[L.CONV_C2] = N, OH, OW, C1, C2
        i[L.CONV_COUT], i[L.CONV_KS], i[L.CONV_STRIDE], i[L.CONV_PAD] = cout, ks, 1, ks // 2
        i[L.CONV_OH], i[L.CONV_OW] = OH, OW
        i[L.CONV_IN_DTYPE] = i[L.CONV_OUT_DTYPE] = i[L.CONV_RES_DTYPE] = fmt
        op.f[0], op.f[1] = float(r.choice([1.0, 0.7071])), float(cout)
        op.inp[0], op.inp[4], op.out[0] = next(fake), next(fake), next(fake)
        if C2:
            op.inp[1] = next(fake)
        if r.random() < 0.7:
            op.inp[5] = next(fake)
        if head or r.random() < 0.5:
            op.inp[2] = next(fake)
        if head:
            i[L.CONV_OUT_LAYOUT], i[L.CONV_OUT_DTYPE], i[L.CONV_RES_DTYPE] = L.NCHW, L.F32, L.F32
            op.f[0], op.f[1] = 1.0, float(int(r.choice([3, 6])))
        else:
            if r.random() < 0.5:
                op.inp[3] = next(fake)
                i[L.CONV_TEMB_OFF] = 32 * int(r.integers(0, 3))
                i[L.CONV_TEMB_BSTRIDE] = 0 if r.random() < 0.5 else i[L.CONV_TEMB_OFF] + cout + 32
            if ks == 3 and r.random() < 0.4:
                i[L.CONV_EXT_C1] = 64 * int(r.integers(1, 3))
                op.inp[8] = next(fake)
                if r.random() < 0.5:
                    i[L.CONV_EXT_C2] = 64
                    op.inp[9] = next(fake)
            if r.random() < 0.7:
                op.out[1] = next(fake)
        cases.append(op)
    return cases


@pytest.mark.parametrize("tier", ["bf16x3", "bf16"])
def test_ow256_conv_tc_sweep_vs_fp64_reference(tier, head_residual_specs):
    fmt = L.BF16S if tier == "bf16x3" else L.BF16
    failures, n_run = [], 0
    for c, op in enumerate(_ow256_cases(fmt)):
        res = T.check_op(op, fmt, seed=5000 + c)
        assert (res is None) == (Plan._tc_eligible(op) != L.OK), T.describe(op)
        if res is None:
            print(f"{T.describe(op):60s} N={op.i[L.CONV_N]}: PSLD_EUNSUPPORTED")
            continue
        n_run += 1
        cls, w, fails = res
        print(f"{T.describe(op):60s} N={op.i[L.CONV_N]:<3d} l2 {w['l2']:.2e} max {w['max']:.2e} "
              f"stat {w['stat']:.2e}{'  FAIL' if fails else ''}")
        failures += [f"{T.describe(op)}: {m}" for m in fails]
    assert n_run >= 12 and not failures, "\n".join(failures[:40])


def test_pyramid_sscs_trajectory_vs_oracle():
    cfg = _pyramid_cfg(tiny_config, "input_skip", "output_skip", sampler="sscs_sde", n_discrete_steps=20)
    ts, n = time_grid(cfg)
    B = 3
    u0, nb = sampler_inputs(cfg, B, n, "sscs_sde")
    net, sd = make_net(cfg, "fp32")
    ref = O.sscs_sample(cfg, _pyramid.ScoreFn(cfg, sd), u0, O.time_grid(cfg)[0], n, nb)
    for tier, gate in (("fp32", 1e-5), ("bf16x3", 1e-4)):
        net.set_precision(tier)
        S = SSCSSampler(cfg, PSLD(cfg), net)
        S.noise = torch.stack(nb).cuda()
        out = S.sample(u0.cuda(), ts.cuda(), n, denoise=True, eps=cfg.evaluation.eval_eps)
        torch.cuda.synchronize()
        e2, em = rel_l2(out.cpu(), ref), max_rel(out.cpu(), ref)
        print(f"SSCS {n}+1 NFE {tier}: rel-L2 {e2:.2e} max {em:.2e}")
        assert e2 <= gate and em <= gate, (tier, e2, em)


def test_pyramid_graph_replay_equals_host_loop():
    cfg = _pyramid_cfg(tiny_config, "input_skip", "output_skip", sampler="sscs_sde", n_discrete_steps=9)
    net, _ = make_net(cfg, "bf16")
    u0, _ = sampler_inputs(cfg, 3, 8, "sscs_sde")
    a, _, _ = _run(cfg, net, u0, None, record=False, graph=False)
    b, _, _ = _run(cfg, net, u0, None, record=False, graph=True)
    assert torch.isfinite(a).all() and torch.equal(a, b)
