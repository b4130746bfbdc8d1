"""CPU: module tree and op programs of NCSN++ with the output-skip / input-skip pyramids
(progressive=output_skip, progressive_input=input_skip, combine=sum), and the promise that the
programs of the existing networks did not change when those were added."""
import hashlib

import numpy as np
import pytest
import torch

import _pyramid
import emulate
from emulate import run_plan
from oracle.weights import fill_state_dict
from psld_b200 import NCSNpp, celeba64_config, cifar10_config, make_config, mid_config, tiny_config
from psld_b200 import _lib as L
from psld_b200.program import Plan, build_plan


def _cfg(base, pin, prog, **sf):
    cfg = base()
    cfg.model.score_fn.update(progressive_input=pin, progressive=prog, progressive_combine="sum", **sf)
    return cfg


def highres_config(size):
    ch_mult = {128: [1, 2, 2, 2, 4], 256: [1, 1, 2, 2, 2, 2, 2]}[size]
    return make_config(image_size=size, score_fn=dict(
        nf=128, ch_mult=ch_mult, num_res_blocks=2, attn_resolutions=[16], fir=True,
        progressive="output_skip", progressive_input="input_skip", progressive_combine="sum",
        embedding_type="fourier"))


def _expected_tree(cfg):
    """(kind, channels) of every all_modules entry in the order of Song's ncsnpp.py __init__."""
    sf = cfg.model.score_fn
    nf, nres = sf.nf, len(sf.ch_mult)
    res = [cfg.data.image_size // 2 ** i for i in range(nres)]
    pin, prog = sf.progressive_input, sf.progressive
    out = [("fourier", None), ("dense", None), ("dense", None), ("conv3", (sf.in_ch, nf))]
    hs, c = [nf], nf
    for lvl in range(nres):
        for _ in range(sf.num_res_blocks):
            out.append(("rb", (c, nf * sf.ch_mult[lvl])))
            c = nf * sf.ch_mult[lvl]
            if res[lvl] in sf.attn_resolutions:
                out.append(("attn", c))
            hs.append(c)
        if lvl != nres - 1:
            out.append(("rb_down", (c, c)))
            if pin == "input_skip":
                out.append(("combine", (sf.in_ch, c)))
            hs.append(c)
    out += [("rb", (c, c)), ("attn", c), ("rb", (c, c))]
    for lvl in reversed(range(nres)):
        for _ in range(sf.num_res_blocks + 1):
            out.append(("rb", (c + hs.pop(), nf * sf.ch_mult[lvl])))
            c = nf * sf.ch_mult[lvl]
        if res[lvl] in sf.attn_resolutions:
            out.append(("attn", c))
        if prog == "output_skip":
            out += [("gn", c), ("conv3", (c, sf.out_ch))]
        if lvl != 0:
            out.append(("rb_up", (c, c)))
    if prog != "output_skip":
        out += [("gn", c), ("conv3", (c, sf.out_ch))]
    return out


def _kind(m):
    n = type(m).__name__
    if n == "ResnetBlockBigGANpp":
        return ("rb_up" if m.up else "rb_down" if m.down else "rb"), (m.in_ch, m.out_ch)
    if n == "AttnBlockpp":
        return "attn", m.channels
    if n == "Combine":
        return "combine", (m.Conv_0.in_channels, m.Conv_0.out_channels)
    if n == "GroupNorm":
        return "gn", m.num_channels
    if n == "Conv2d":
        return "conv3", (m.in_channels, m.out_channels)
    if n == "Linear":
        return "dense", None
    return {"GaussianFourierProjection": "fourier"}.get(n, n), None


@pytest.mark.parametrize("pin,prog", [("input_skip", "none"), ("none", "output_skip"),
                                      ("input_skip", "output_skip"), ("residual", "output_skip")])
@pytest.mark.parametrize("base", [tiny_config, mid_config])
def test_module_tree_order_names_shapes(base, pin, prog):
    cfg = _cfg(base, pin, prog)
    net = NCSNpp(cfg)
    if pin == "residual":           # the residual pyramid keeps its own (tested) module list
        assert [_kind(m)[0] for m in net.all_modules].count("gn") == len(cfg.model.score_fn.ch_mult)
        return
    assert [_kind(m) for m in net.all_modules] == _expected_tree(cfg)
    sd = net.state_dict()
    for i, m in enumerate(net.all_modules):
        if type(m).__name__ == "Combine":       # Conv_0 = ddpm_conv1x1(input channels, h channels)
            C = m.Conv_0.out_channels
            assert tuple(sd[f"all_modules.{i}.Conv_0.weight"].shape) == (C, 6, 1, 1)
            assert tuple(sd[f"all_modules.{i}.Conv_0.bias"].shape) == (C,)
            assert not any(k.startswith(f"all_modules.{i}.") and ".Conv_0." not in k for k in sd)
    last = net.all_modules[-1]
    assert isinstance(last, torch.nn.Conv2d) and last.out_channels == 6


def test_full_size_parameter_counts():
    got = {s: sum(p.numel() for p in NCSNpp(highres_config(s)).parameters()) for s in (128, 256)}
    assert got == {128: 86170782, 256: 65623338}, got
    assert len(NCSNpp(highres_config(256)).state_dict()) == 645


def test_rejected_configurations():
    cfg = _cfg(tiny_config, "input_skip", "output_skip")
    cfg.model.score_fn.progressive_combine = "cat"
    with pytest.raises(NotImplementedError, match="progressive_combine=sum"):
        NCSNpp(cfg)
    with pytest.raises(NotImplementedError, match="progressive must be"):
        NCSNpp(_cfg(tiny_config, "none", "residual"))


@pytest.mark.parametrize("fir", [True, False])
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-5), ("bf16x3", 1e-4), ("bf16", 3e-2)])
def test_pyramid_program_vs_reference(precision, tol, fir, monkeypatch):
    """The op program of output_skip + input_skip interpreted on the host (tests/emulate.py) gives the
    reference forward of tests/_pyramid.py; the NCHW-head residual routes as the library does."""
    monkeypatch.setattr(emulate, "reference_op", _pyramid.reference_op)
    cfg = _cfg(mid_config, "input_skip", "output_skip", fir=fir)
    net = NCSNpp(cfg).eval()
    net.precision = precision
    sd = fill_state_dict({k: tuple(v.shape) for k, v in net.state_dict().items()}, 0)
    net.load_state_dict(sd)
    r = np.random.default_rng(0)
    x = torch.from_numpy(r.standard_normal((2, 6, 32, 32)).astype(np.float32))
    t = torch.tensor([0.6, 0.05])
    y = _pyramid.ncsnpp_forward(cfg, sd, x, t)
    plan = build_plan(net, 2, 2, False, dry=True)
    out = run_plan(plan, x, t)
    assert float((out - y).norm() / y.norm()) <= tol
    if precision != "fp32":
        assert plan.engine_count["simt"] == 0, plan.engine_count
    heads = [op for op in plan.ops if op.kind == L.OP_CONV and op.i[L.CONV_OUT_LAYOUT] == L.NCHW]
    assert len(heads) == 2 and not heads[0].inp[2] and heads[1].inp[2]
    assert heads[1].i[L.CONV_RES_DTYPE] == L.F32


def test_tc_eligibility_of_wide_rows():
    op = L.Op()
    i = op.i
    i[L.CONV_N], i[L.CONV_H], i[L.CONV_W], i[L.CONV_C1], i[L.CONV_COUT] = 2, 256, 256, 128, 128
    i[L.CONV_KS], i[L.CONV_STRIDE], i[L.CONV_PAD], i[L.CONV_OH], i[L.CONV_OW] = 3, 1, 1, 256, 256
    i[L.CONV_IN_DTYPE] = i[L.CONV_OUT_DTYPE] = i[L.CONV_RES_DTYPE] = L.BF16
    assert Plan._tc_eligible(op) == L.OK
    i[L.CONV_W] = i[L.CONV_OW] = 512
    assert Plan._tc_eligible(op) == L.EUNSUPPORTED
    i[L.CONV_W], i[L.CONV_OW], i[L.CONV_H], i[L.CONV_OH] = 513, 256, 513, 256     # stride 2: rows <= 128
    i[L.CONV_STRIDE], i[L.CONV_PAD] = 2, 0
    assert Plan._tc_eligible(op) == L.EUNSUPPORTED
    i[L.CONV_W], i[L.CONV_OW], i[L.CONV_H], i[L.CONV_OH] = 256, 256, 256, 256     # NCHW head + residual
    i[L.CONV_STRIDE], i[L.CONV_PAD], i[L.CONV_OUT_LAYOUT], i[L.CONV_OUT_DTYPE] = 1, 1, L.NCHW, L.F32
    op.inp[2] = 0x1000
    assert Plan._tc_eligible(op) == L.EUNSUPPORTED          # residual must be fp32
    i[L.CONV_RES_DTYPE] = L.F32
    assert Plan._tc_eligible(op) == L.OK


# Digests of the op programs of the existing networks at their benchmark batches (one shared time
# row), computed at the commit before the pyramids and 256-wide tiles were added: every op's kind,
# engine, i[] and f[], and the bytes of every packed parameter it reads.
PARENT_DIGESTS = {
    ("tiny", "fp32"): "8db894e8454aa1d7d50c60291927b064",
    ("tiny", "bf16"): "65c3728f7436b46ff09807eced7f82dd",
    ("tiny", "bf16x3"): "9954089fbeddb683efc4de584b6546ed",
    ("mid", "fp32"): "735421e3ca38e3b6ee80b1a429398c9c",
    ("mid", "bf16"): "9936132d1b902c4b466a429ec69e2f07",
    ("mid", "bf16x3"): "d3c54d47b65fe71d1c7dcd2636dbd89b",
    ("cifar10", "fp32"): "3605fd9c8328d2b802d92620b87a9946",
    ("cifar10", "bf16"): "ea3cbd3783663a5bf3b21f71ad126ed8",
    ("cifar10", "bf16x3"): "e8940afffe3484e6b553e6fb2e8a7400",
    ("celeba64", "fp32"): "4d4155ae0db060738c8eb995f5e008bc",
    ("celeba64", "bf16"): "36652bd80dbad4cacf51f741de7c4d8c",
    ("celeba64", "bf16x3"): "bc845a947256ced79c5591133b40e26c",
}
_CONFIGS = {"tiny": tiny_config, "mid": mid_config, "cifar10": cifar10_config, "celeba64": celeba64_config}
_WEIGHT_SLOTS = {L.OP_CONV: (4, 5), L.OP_ATTN: (1, 2), L.OP_GN: (2, 3), L.OP_TEMB: (1, 2, 3, 4, 5, 6, 7)}


def program_digest(cfg, precision):
    net = NCSNpp(cfg).eval()
    net.precision = precision
    net.load_state_dict(fill_state_dict({k: tuple(v.shape) for k, v in net.state_dict().items()}, 0))
    plan = build_plan(net, int(cfg.evaluation.batch_size), 1, False, dry=True)
    T = {}
    for t in plan.keep:
        T.setdefault(t.data_ptr(), t)
    h = hashlib.sha256()
    for op in plan.ops:
        h.update(np.asarray([op.kind, op.engine, *op.i], np.int64).tobytes())
        h.update(np.asarray(list(op.f), np.float32).tobytes())
        for s in _WEIGHT_SLOTS.get(op.kind, ()):
            if op.inp[s]:
                h.update(T[op.inp[s]].detach().contiguous().view(-1).view(torch.uint8).numpy().tobytes())
    return h.hexdigest()[:32]


@pytest.mark.parametrize("name,precision", sorted(PARENT_DIGESTS))
def test_existing_programs_unchanged(name, precision):
    assert program_digest(_CONFIGS[name](), precision) == PARENT_DIGESTS[name, precision]


@pytest.mark.parametrize("emb", ["fourier", "positional"])
def test_pyramid_reference_equals_oracle_without_pyramids(emb):
    """tests/_pyramid.ncsnpp_forward is the oracle's forward where the oracle applies (residual input
    pyramid, single output head)."""
    from oracle import psld_oracle as O
    cfg = tiny_config()
    cfg.model.score_fn.embedding_type = emb
    net = NCSNpp(cfg)
    sd = fill_state_dict({k: tuple(v.shape) for k, v in net.state_dict().items()}, 3)
    r = np.random.default_rng(1)
    x = torch.from_numpy(r.standard_normal((2, 6, 32, 32)).astype(np.float32))
    t = torch.tensor([0.4, 0.9])
    assert torch.equal(_pyramid.ncsnpp_forward(cfg, sd, x, t), O.ncsnpp_forward(cfg, sd, x, t))
