"""Every distinct op of the benchmarked programs, at the batches the benchmark runs, against the fp64
reference semantics of ``tests/emulate.py::reference_op``.

The kernel tests (test_gpu_kernels.py, test_gpu_x3.py) pick shapes by hand at batches of 1 to 41,
and the network tests compare whole forwards with one rel-L2 over the tensor.  Here each op record
of a real plan (CIFAR-10 at B = 1, 3, 128, 256, CelebA-64 at B = 1, 64, classifier-free guidance at
B = 128, fp32 CUDA-core engines at B = 256, one forward plan with per-sample time rows) is copied,
pointed at test-owned buffers and run alone, so the launch geometry (pair / single CTA, persistent
rounds, tail N-split, images per tile) is exactly the one the benchmark launches.  A seeded sweep
over the C ABI's stated tensor-core eligibility covers the shapes the planner does not emit.

Every buffer has a guard band of random bytes on each side, and the buffer start keeps the 512-byte
alignment of a fresh torch allocation.  Checks, per sample (so one bad image or tile is not diluted
by the rest of the batch):
  * rel-L2 and max-abs / max|ref| against the fp64 reference of the same decoded inputs;
  * an elementwise bound |y - ref| <= a |ref| + b rms(ref), so one wrong row or pixel fails;
  * every element the op must write is finite, every element it must leave alone still holds its
    prefill, guard bands and input buffers are unchanged byte for byte;
  * GroupNorm statistics accumulators end at (random base) + fp64 sums of the reference output.
"""
from __future__ import annotations

import ctypes as C
import math
import time
from collections import namedtuple

import numpy as np
import pytest
import torch

from _net import make_net
from _ops import to_split
from emulate import reference_op
from psld_b200 import _lib as L
from psld_b200 import celeba64_config, cifar10_config
from psld_b200.guidance import GuidedPlan
from psld_b200.program import Plan, build_plan

pytestmark = pytest.mark.gpu

DEV = "cuda"
GUARD = 4096                      # bytes on each side of every buffer (a multiple of 512)
W2 = "w2"                         # split-bf16 weight planes [2][rows, K] (logical [rows, K])

Spec = namedtuple("Spec", "shape fmt role src")      # src: input slot a statistics input describes

# ---------------------------------------------------------------------------------------------- gates
# (rel-L2, max-abs/max|ref|, a, b, statistics) per sample; the elementwise bound is
# |y - ref| <= a |ref| + b rms(ref).  a = 2^-8 covers the one bf16 rounding of a bf16 output, 2^-16 the
# split rounding of a split-bf16 one.  Worst per-sample values measured on a B200 (1000 W power limit)
# over the programs and the sweep are in the comments, in the same order; gates that were widened are
# at most 2x the measured value.
BF, SP = 2.0 ** -8, 2.0 ** -16
GATES = {
    # fp32 tier: CUDA-core fp32 engines, fp32 summation order (test_gpu_kernels.py: 3e-6)
    "fp32":            (3e-6, 3e-5, 0.0, 4e-5, None),       # 1.1e-6 4.0e-6 1.9e-5
    # split-bf16 tensor-core tier (test_gpu_x3.py: 2e-5 rel-L2, 3e-5 max, statistics 3e-5)
    "bf16x3 conv":     (2e-5, 3e-5, SP, 1.2e-4, 3e-5),      # 1.2e-5 2.2e-5 6.0e-5 1.8e-5
    "bf16x3 attn":     (2e-5, 3e-5, SP, 1.2e-4, 3e-5),      # 5.8e-6 1.5e-5 5.9e-5 9.6e-7
    "bf16x3 memory":   (1e-5, 3e-5, SP, 1e-5, None),        # 2.6e-6 7.6e-6 1.8e-7
    # bf16 conv_tc: operands are exact bf16 values and the output is rounded once
    "bf16 conv_tc":    (4e-3, 2 * BF, BF, 2.0 ** -12, 2e-4),   # 1.8e-3 3.9e-3 1.1e-5 6.3e-6
    # bf16 GroupNorm-on-load conv and attention: tanh-form SiLU before the bf16 rounding of A, bf16 P
    "bf16 conv_gn":    (6e-3, 2 * BF, BF, 4e-3, 5e-3),      # 1.7e-3 3.9e-3 2.0e-3 2.1e-5
    "bf16 attn":       (8e-3, 8e-3, BF, 1.2e-2, 1e-2),      # 1.9e-3 4.0e-3 6.0e-3 1.5e-4
    "bf16 memory":     (6e-3, 2 * BF, BF, 2.0 ** -12, None),   # 1.7e-3 3.9e-3 9.9e-6
    # format-free fp32 ops of every tier
    "temb":            (3e-6, 3e-5, 0.0, 3e-5, None),       # 1.8e-7 2.1e-7 7.8e-7
    "gn affine":       (3e-6, 3e-5, 0.0, 3e-5, None),       # 3.9e-8 7.0e-8 1.2e-7
    # (1 + w) a - w b rounds once to fp32; where the two terms cancel that rounding is large against
    # the result's rms, hence b above 2^-24
    "axpby":           (3e-7, 3e-7, 0.0, 9e-7, None),       # 4.0e-8 8.8e-8 4.4e-7
    "zero":            (0.0, 0.0, 0.0, 0.0, None),
}


def op_class(op):
    k, e = op.kind, op.engine
    if k == L.OP_ZERO:
        return "zero"
    if k == L.OP_AXPBY:
        return "axpby"
    if k == L.OP_TEMB:
        return "temb"
    if k == L.OP_GN and op.i[L.GN_AFFINE_ONLY]:
        return "gn affine"
    dt = {L.OP_LAYOUT: op.i[L.LAYOUT_DTYPE], L.OP_GN: op.i[L.GN_IN_DTYPE], L.OP_FIR: op.i[L.FIR_DTYPE],
          L.OP_CONV: op.i[L.CONV_IN_DTYPE], L.OP_ATTN: op.i[L.ATTN_DTYPE]}[k]
    if k == L.OP_CONV and op.i[L.CONV_IN_LAYOUT] == L.NCHW:
        dt = op.i[L.CONV_OUT_DTYPE]
    if dt == L.F32:
        return "fp32"
    tier = {L.BF16: "bf16", L.BF16S: "bf16x3"}[dt]
    if k == L.OP_CONV and e == L.ENGINE_TC:
        return "bf16x3 conv" if dt == L.BF16S else "bf16 conv_tc"
    if k == L.OP_CONV and e == L.ENGINE_TC_GN:
        return "bf16x3 conv" if dt == L.BF16S else "bf16 conv_gn"
    if k == L.OP_ATTN and e == L.ENGINE_TC:
        return tier + " attn"
    return tier + " memory"


# ------------------------------------------------------------------------------------- slot layout
def slot_specs(op):
    """{("in"|"out", slot): Spec} of every non-NULL pointer, as include/psld_b200.h documents it.
    role: act (random input), w (parameter: copied from the plan), time, stat_in (fp64 sums of the
    input slot ``src``), out, stat_out (accumulated statistics), scratch."""
    i, k = op.i, op.kind
    s = {}
    if k == L.OP_ZERO:
        s["out", 0] = Spec(((i[0] | (i[1] << 31)) // 8,), L.F64, "out", None)
    elif k == L.OP_AXPBY:
        n = i[0] | (i[1] << 31)
        s["in", 0] = s["in", 1] = Spec((n,), L.F32, "act", None)
        s["out", 0] = Spec((n,), L.F32, "out", None)
    elif k == L.OP_LAYOUT:
        N, Cc, HW, dt = i[L.LAYOUT_N], i[L.LAYOUT_C], i[L.LAYOUT_HW], i[L.LAYOUT_DTYPE]
        if i[L.LAYOUT_DIR] == 0:
            s["in", 0] = Spec((N, Cc, HW), L.F32, "act", None)
            s["out", 0] = Spec((N, HW, i[L.LAYOUT_CPAD] or Cc), dt, "out", None)
        else:
            s["in", 0] = Spec((N, HW, Cc), dt, "act", None)
            s["out", 0] = Spec((N, Cc, HW), L.F32, "out", None)
    elif k == L.OP_TEMB:
        nt, nf, tot = i[L.TEMB_NT], i[L.TEMB_NF], i[L.TEMB_TOTALC]
        E = 2 * nf if i[L.TEMB_EMB] == 0 else nf
        s["in", 0] = Spec((nt,), L.F32, "time", None)
        for j, shp in ((1, (nf,)), (2, (4 * nf, E)), (3, (4 * nf,)), (4, (4 * nf, 4 * nf)), (5, (4 * nf,)),
                       (6, (tot, 4 * nf)), (7, (tot,))):
            s["in", j] = Spec(shp, L.F32, "w", None)
        s["out", 0] = Spec((nt, tot), L.F32, "out", None)
        s["out", 1] = Spec((nt, E + 8 * nf), L.F32, "scratch", None)
        if op.out[2]:
            raise AssertionError("TEMB with a device step counter is not covered")
    elif k == L.OP_GN:
        N, HW, C1, C2, G = i[L.GN_N], i[L.GN_HW], i[L.GN_C1], i[L.GN_C2], i[L.GN_G]
        s["in", 0] = Spec((N, HW, C1), i[L.GN_IN_DTYPE], "act", None)
        s["in", 1] = Spec((N, HW, C2), i[L.GN_IN_DTYPE], "act", None)
        s["in", 2] = s["in", 3] = Spec((C1 + C2,), L.F32, "w", None)
        s["in", 4] = Spec((N, C1 // 4, 2), L.F64, "stat_in", 0)
        s["in", 5] = Spec((N, C2 // 4, 2), L.F64, "stat_in", 1)
        s["out", 0] = Spec((N, C1 + C2, 2), L.F32, "out", None) if i[L.GN_AFFINE_ONLY] else \
            Spec((N, HW, C1 + C2), i[L.GN_OUT_DTYPE], "out", None)
        s["out", 1] = Spec((N * i[L.GN_NCHUNK] * G * 2,), L.F64, "scratch", None)
    elif k == L.OP_FIR:
        N, H, W, Cc = i[L.FIR_N], i[L.FIR_H], i[L.FIR_W], i[L.FIR_C]
        up, down, KH = i[L.FIR_UP], i[L.FIR_DOWN], i[L.FIR_KH]
        OH = (H * up + i[L.FIR_PAD0] + i[L.FIR_PAD1] - KH) // down + 1
        OW = (W * up + i[L.FIR_PAD0] + i[L.FIR_PAD1] - KH) // down + 1
        s["in", 0] = Spec((N, H, W, Cc), i[L.FIR_DTYPE], "act", None)
        s["out", 0] = Spec((N, OH, OW, Cc), i[L.FIR_DTYPE], "out", None)
    elif k == L.OP_CONV:
        N, H, W, C1, C2 = i[L.CONV_N], i[L.CONV_H], i[L.CONV_W], i[L.CONV_C1], i[L.CONV_C2]
        cout, ks, OH, OW = i[L.CONV_COUT], i[L.CONV_KS], i[L.CONV_OH], i[L.CONV_OW]
        dt, tc = i[L.CONV_IN_DTYPE], op.engine in (L.ENGINE_TC, L.ENGINE_TC_GN)
        e1, e2 = (i[L.CONV_EXT_C1], i[L.CONV_EXT_C2]) if tc else (0, 0)
        s["in", 0] = Spec((N, H, W, C1), dt, "act", None)
        s["in", 1] = Spec((N, H, W, C2), dt, "act", None)
        s["in", 2] = Spec((N, OH, OW, cout), i[L.CONV_RES_DTYPE], "act", None)
        bs = i[L.CONV_TEMB_BSTRIDE]
        s["in", 3] = Spec((N, bs) if bs else (1, i[L.CONV_TEMB_OFF] + cout), L.F32, "act", None)
        K = ks * ks * (C1 + C2)
        if tc:
            s["in", 4] = Spec((cout, K + e1 + e2), W2 if dt == L.BF16S else L.BF16, "w", None)
        else:
            s["in", 4] = Spec((K, cout), L.F32, "w", None)
        s["in", 5] = Spec((cout,), L.F32, "w", None)
        s["in", 6] = Spec((N, C1 + C2, 2), L.F32, "affine", None)
        s["in", 8] = Spec((N, OH, OW, e1), dt, "act", None)
        s["in", 9] = Spec((N, OH, OW, e2), dt, "act", None)
        if i[L.CONV_OUT_LAYOUT] == L.NCHW:
            valid = int(op.f[1]) if tc else cout
            s["out", 0] = Spec((N, valid, OH, OW), L.F32, "out", None)
        else:
            s["out", 0] = Spec((N, OH, OW, cout), i[L.CONV_OUT_DTYPE], "out", None)
        s["out", 1] = Spec((N, cout // 4, 2), L.F64, "stat_out", None)
    elif k == L.OP_ATTN:
        N, HW, Cc, dt = i[L.ATTN_N], i[L.ATTN_HW], i[L.ATTN_C], i[L.ATTN_DTYPE]
        s["in", 0] = Spec((N, HW, 3 * Cc), dt, "act", None)
        s["in", 1] = Spec((Cc, Cc), W2 if dt == L.BF16S else L.BF16, "w", None)
        s["in", 2] = Spec((Cc,), L.F32, "w", None)
        s["in", 3] = Spec((N, HW, Cc), dt, "act", None)
        s["out", 0] = Spec((N, HW, Cc), dt, "out", None)
        s["out", 1] = Spec((N, Cc // 4, 2), L.F64, "stat_out", None)
    else:
        raise AssertionError(f"op kind {k} has no reference: add it to tests/emulate.py and here")
    if op.engine not in (L.ENGINE_SIMT, L.ENGINE_TC, L.ENGINE_TC_GN) or \
            (op.engine != L.ENGINE_SIMT and k not in (L.OP_CONV, L.OP_ATTN)) or \
            (op.engine == L.ENGINE_TC_GN and k != L.OP_CONV):
        raise AssertionError(f"op kind {k} engine {op.engine} has no reference")
    ptr = {"in": op.inp, "out": op.out}
    return {key: sp for key, sp in s.items() if ptr[key[0]][key[1]]}


def storage(buf, sp):
    """Typed view of a buffer's payload for a slot spec."""
    shape, fmt = sp.shape, sp.fmt
    if fmt == L.BF16S:
        return buf.view(torch.bfloat16).view(*shape[:-1], 2 * shape[-1])
    if fmt == W2:
        return buf.view(torch.bfloat16).view(2 * shape[0], *shape[1:])
    dt = {L.F32: torch.float32, L.F64: torch.float64, L.BF16: torch.bfloat16}[fmt]
    return buf.view(dt).view(shape)


def nbytes(sp):
    n = math.prod(sp.shape)
    return n * {L.F32: 4, L.F64: 8, L.BF16: 2, L.BF16S: 4, W2: 4}[sp.fmt]


def encode(v, sp):
    """Logical values -> storage tensor of the slot's format."""
    if sp.fmt == L.BF16S:
        return to_split(v.float()).as_subclass(torch.Tensor).view(torch.bfloat16)
    if sp.fmt == W2:
        hi = v.float().to(torch.bfloat16)
        return torch.cat([hi, (v.float() - hi.float()).to(torch.bfloat16)], 0)
    return v.to({L.F32: torch.float32, L.F64: torch.float64, L.BF16: torch.bfloat16}[sp.fmt])


def decode(st, sp):
    """Storage tensor -> logical values in float64."""
    if sp.fmt == L.BF16S:
        c = sp.shape[-1]
        return st[..., :c].double() + st[..., c:].double()
    if sp.fmt == W2:
        r = sp.shape[0]
        return st[:r].double() + st[r:].double()
    return st.double()


def written_mask(sp, idx):
    m = torch.zeros(sp.shape, dtype=torch.bool, device=DEV)
    m[idx] = True
    return torch.cat([m, m], -1) if sp.fmt == L.BF16S else m


def _bits(t):
    return t.view({1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}[t.element_size()])


def _signature(op):
    return (op.kind, op.engine, tuple(op.i), tuple(np.float32(list(op.f)).view(np.uint32).tolist()),
            tuple(bool(p) for p in op.inp), tuple(bool(p) for p in op.out))


def describe(op):
    i, k = op.i, op.kind
    name = {1: "LAYOUT", 2: "TEMB", 3: "GN", 4: "FIR", 5: "CONV", 6: "ATTN", 7: "ZERO", 8: "AXPBY"}[k]
    if k == L.OP_CONV:
        return (f"{name} e{op.engine} {i[L.CONV_H]}x{i[L.CONV_W]} {i[L.CONV_C1]}+{i[L.CONV_C2]}"
                f"(+{i[L.CONV_EXT_C1] + i[L.CONV_EXT_C2]})->{i[L.CONV_COUT]} k{i[L.CONV_KS]}s{i[L.CONV_STRIDE]}"
                f"{' nchw' if i[L.CONV_OUT_LAYOUT] == L.NCHW else ''}{' st' if op.out[1] else ''}")
    if k == L.OP_GN:
        return (f"{name} hw{i[L.GN_HW]} {i[L.GN_C1]}+{i[L.GN_C2]} g{i[L.GN_G]}"
                f"{' aff' if i[L.GN_AFFINE_ONLY] else ''}{' mg' if op.inp[4] else ''}")
    if k == L.OP_ATTN:
        return f"{name} e{op.engine} hw{i[L.ATTN_HW]} c{i[L.ATTN_C]}{' proj' if i[L.ATTN_PROJ] else ''}"
    if k == L.OP_FIR:
        return f"{name} {i[L.FIR_H]}x{i[L.FIR_W]}x{i[L.FIR_C]} up{i[L.FIR_UP]} down{i[L.FIR_DOWN]}"
    return name


# ------------------------------------------------------------------------------------- one op
def check_op(src_op, fmt, seed, weights=None, B=None):
    """Runs a copy of ``src_op`` on fresh guarded buffers and compares it with reference_op in fp64.
    ``weights(ptr)`` returns the plan tensor behind a parameter pointer (None: random parameters).
    Returns None when psld_op_prepare rejects the op with PSLD_EUNSUPPORTED, else
    (class, per-metric worst values, list of failure messages)."""
    op = L.Op.from_buffer_copy(src_op)
    op.aux = None
    specs = slot_specs(op)
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    ptrs = {}                                  # original pointer -> [buffer, payload bytes, first spec]
    for (io, j), sp in specs.items():
        p = (op.inp if io == "in" else op.out)[j]
        e = ptrs.setdefault(p, [None, 0, sp, io])
        assert e[3] == io, "a pointer is both read and written by one op"
        e[1] = max(e[1], nbytes(sp))
    for p, e in ptrs.items():
        buf = torch.empty(2 * GUARD + e[1], dtype=torch.uint8, device=DEV)
        buf.random_(0, 256, generator=g)       # guard bands: random bytes
        e[0] = buf
    payload = lambda p: ptrs[p][0][GUARD:GUARD + ptrs[p][1]]
    vals = {}                                  # pointer -> logical fp64 value of an input
    for (io, j), sp in sorted(specs.items(), key=lambda kv: kv[1].role == "stat_in"):
        p = (op.inp if io == "in" else op.out)[j]
        st = storage(payload(p), sp)
        if sp.role == "w" and weights is not None:
            w = weights(p)
            assert w.numel() * w.element_size() == nbytes(sp), (describe(op), io, j, w.shape, sp)
            payload(p).copy_(w.reshape(-1).view(torch.uint8))
        elif sp.role in ("act", "w", "time", "affine"):
            v = torch.randn(sp.shape, generator=g, device=DEV, dtype=torch.float64)
            if sp.role == "time":
                v = torch.rand(sp.shape, generator=g, device=DEV, dtype=torch.float64) * 0.99 + 0.01
                if op.i[L.TEMB_LOGGED]:
                    v = v.log()
            elif sp.role == "affine":       # (scale, shift) of a GroupNorm applied on load
                v = v * torch.tensor([0.3, 0.2], device=DEV, dtype=torch.float64) + \
                    torch.tensor([1.0, 0.0], device=DEV, dtype=torch.float64)
            elif sp.role == "w":
                v = v / math.sqrt(sp.shape[-1] if len(sp.shape) > 1 else 100.0)
            else:
                v = v * 1.3 + 0.2
            st.copy_(encode(v, sp))
        elif sp.role == "stat_in":
            sp_src = specs["in", sp.src]
            x = decode(storage(payload(op.inp[sp.src]), sp_src), sp_src)
            x = x.reshape(x.shape[0], -1, x.shape[-1] // 4, 4)
            st.copy_(torch.stack([x.sum((1, 3)), (x * x).sum((1, 3))], -1))
        else:                                  # outputs, scratch: NaN prefill
            st.copy_(torch.full(st.shape, float("nan"), dtype=st.dtype, device=DEV))
        if io == "in" and p not in vals:
            vals[p] = decode(storage(payload(p), sp), sp)
    get = lambda p: None if not p else vals[p]
    ref = reference_op(op, get, fmt)
    # statistics accumulators start from a random base of the size of what is added
    base = {}
    for slot, (idx, v, acc) in ref.items():
        if acc:
            sp = specs["out", slot]
            scale = float(v.abs().max()) + 1.0
            b = (torch.rand(sp.shape, generator=g, device=DEV, dtype=torch.float64) + 0.5) * scale
            storage(payload(op.out[slot]), sp).copy_(b)
            base[slot] = b
    before = {p: e[0].clone() for p, e in ptrs.items()}
    orig_out = list(op.out)
    repoint(op, {p: e[0].data_ptr() + GUARD for p, e in ptrs.items()})
    lib = L.lib()
    rc = lib.psld_op_prepare(C.byref(op))
    if rc == L.EUNSUPPORTED:
        return None
    L.check(rc, f"psld_op_prepare({describe(op)})")
    try:
        L.check(lib.psld_op_run(C.byref(op), L.stream_ptr()), f"psld_op_run({describe(op)})")
        torch.cuda.synchronize()
    finally:
        lib.psld_op_release(C.byref(op))
    cls = op_class(op)
    l2g, mxg, a, b, stg = GATES[cls]
    fails, worst = [], {"l2": 0.0, "max": 0.0, "elem": 0.0, "stat": 0.0}
    for p, e in ptrs.items():
        buf, n = e[0], e[1]
        old = before[p]
        if e[3] == "in":
            if not torch.equal(buf, old):
                fails.append(f"input buffer changed ({e[2]})")
        elif not (torch.equal(buf[:GUARD], old[:GUARD]) and torch.equal(buf[GUARD + n:], old[GUARD + n:])):
            fails.append(f"guard band of an output overwritten ({e[2]})")
    for slot, (idx, v, acc) in ref.items():
        sp = specs["out", slot]
        p = orig_out[slot]
        st = storage(payload(p), sp)
        st_old = storage(before[p][GUARD:GUARD + ptrs[p][1]], sp)
        m = written_mask(sp, idx)
        if not torch.equal(_bits(st)[~m], _bits(st_old)[~m]):
            fails.append(f"out[{slot}]: elements outside the written region changed")
        y = decode(st, sp)[idx]
        r = v.to(y.device).reshape(y.shape)
        if acc:
            d = (y - base[slot][idx] - r).reshape(r.shape[0], -1)
            e = (d.abs().amax(1) / r.reshape(r.shape[0], -1).abs().amax(1).clamp_min(1e-300)).max().item()
            worst["stat"] = max(worst["stat"], e)
            if not e <= (stg if stg is not None else 0.0):
                fails.append(f"out[{slot}] statistics: {e:.3e} > {stg}")
            continue
        if not torch.isfinite(y).all():
            fails.append(f"out[{slot}]: {int((~torch.isfinite(y)).sum())} written elements are not finite")
            continue
        S = B if (op.kind == L.OP_AXPBY and B and r.numel() % B == 0) else (1 if r.dim() == 1 else r.shape[0])
        d, rr = (y - r).reshape(S, -1), r.reshape(S, -1)
        nr = rr.norm(dim=1)
        zero = nr == 0
        if bool(zero.any()) and float(d[zero].abs().max()) != 0.0:
            fails.append(f"out[{slot}]: nonzero where the reference is exactly zero")
        nr = nr.clamp_min(1e-300)
        l2 = (d.norm(dim=1) / nr).masked_fill(zero, 0.0)
        mx = (d.abs().amax(1) / rr.abs().amax(1).clamp_min(1e-300)).masked_fill(zero, 0.0)
        rms = nr / math.sqrt(rr.shape[1])
        el = ((d.abs() - a * rr.abs()).amax(1) / rms).masked_fill(zero, 0.0)
        for key, val, gate in (("l2", l2, l2g), ("max", mx, mxg), ("elem", el, b)):
            w_, s_ = val.max(0)
            worst[key] = max(worst[key], float(w_))
            if not float(w_) <= gate:
                fails.append(f"out[{slot}] {key} {float(w_):.3e} > {gate:.1e} (sample {int(s_)} of {S})")
    return cls, worst, fails


def repoint(op, new):
    for arr in (op.inp, op.out):
        for j in range(L.OP_NP):
            if arr[j]:
                arr[j] = new[arr[j]]


# ------------------------------------------------------------------------------------- programs
def _full(c):
    c.model.score_fn.init_scale = 1.0
    return c


_NETS = {}


def _net(name, precision, seed=0):
    key = (name, seed)
    if key not in _NETS:
        cfg = _full({"cifar10": cifar10_config, "celeba64": celeba64_config}[name]())
        _NETS[key] = make_net(cfg, precision, seed=seed)[0]
    net = _NETS[key]
    net.set_precision(precision)
    return net


def _plans():
    """(label, plan factory) of every program the benchmark runs, plus the fp32 CUDA-core engines at
    the bench batch and one forward plan with per-sample time rows."""
    out = []
    for prec in ("bf16x3", "bf16"):
        for B in (1, 3, 128, 256):
            out.append((f"cifar10 {prec} B={B}", lambda p=prec, B=B: build_plan(_net("cifar10", p), B, 1, True)))
    out.append(("cifar10 bf16x3 cfg-guidance B=128", lambda: GuidedPlan(
        build_plan(_net("cifar10", "bf16x3"), 128, 1, True),
        build_plan(_net("cifar10", "bf16x3", seed=1), 128, 1, True), 1.5)))
    for prec in ("bf16x3", "bf16"):
        for B in (1, 64):
            out.append((f"celeba64 {prec} B={B}", lambda p=prec, B=B: build_plan(_net("celeba64", p), B, 1, True)))
    out.append(("cifar10 fp32 B=256", lambda: build_plan(_net("cifar10", "fp32"), 256, 1, True)))
    out.append(("cifar10 bf16x3 forward B=3 nt=3", lambda: build_plan(_net("cifar10", "bf16x3"), 3, 3, False)))
    return out


def _fmt(plan):
    return L.BF16 if plan.bf16 else (L.BF16S if plan.x3 else L.F32)


def _report(rows, worst_by_class):
    print()
    for r in rows:
        print(r)
    print("worst per-sample error per op class (rel-L2 | max-abs/max|ref| | elementwise/rms | statistics):")
    for cls, w in sorted(worst_by_class.items()):
        print(f"  {cls:15s} {w['l2']:.3e} | {w['max']:.3e} | {w['elem']:.3e} | {w['stat']:.3e}")


def _merge(worst_by_class, cls, w):
    acc = worst_by_class.setdefault(cls, {"l2": 0.0, "max": 0.0, "elem": 0.0, "stat": 0.0})
    for k_, v in w.items():
        acc[k_] = max(acc[k_], v)


def test_program_ops_vs_fp64_reference():
    t0 = time.time()
    seen, failures, rows, worst_by_class = set(), [], [], {}
    for label, make in _plans():
        plan = make()
        keep = {t.data_ptr(): t for t in plan.keep}
        ops = plan.ops if isinstance(plan, GuidedPlan) else list(plan.op_array)
        new = 0
        for op in ops:
            sig = _signature(op)
            if sig in seen:
                continue
            seen.add(sig)
            new += 1
            res = check_op(op, _fmt(plan), seed=len(seen), weights=keep.__getitem__, B=plan.B)
            if res is None:
                failures.append(f"{label}: {describe(op)} rejected by psld_op_prepare")
                continue
            cls, w, fails = res
            _merge(worst_by_class, cls, w)
            print(f"{label:34s} {describe(op):52s} B={plan.B:<4d} {cls:13s} l2 {w['l2']:.2e} max {w['max']:.2e} "
                  f"elem {w['elem']:.2e} stat {w['stat']:.2e}{'  FAIL' if fails else ''}")
            failures += [f"{label}: {describe(op)}: {m}" for m in fails]
        rows.append(f"{label:34s} {new:4d} new distinct op signatures ({len(ops)} ops)")
        del plan, keep, ops
        torch.cuda.empty_cache()
    _report(rows, worst_by_class)
    print(f"{len(seen)} distinct signatures in {time.time() - t0:.1f} s")
    assert not failures, "\n".join(failures[:40])


# ------------------------------------------------------------------------------------- shape sweep
def _pow2(lo, hi, r):
    return 1 << int(r.integers(int(math.log2(lo)), int(math.log2(hi)) + 1))


def _sweep_cases(fmt, n=30, seed=2024):
    """Seeded op records drawn from the C ABI's stated tensor-core eligibility (include/psld_b200.h,
    prepare_conv_tc / prepare_conv_gn_tc / prepare_attn_tc): conv_tc with OW, OH powers of two,
    4 <= OW <= 128, OH down to 1, Cin % 64 == 0 over one or two sources, Cout % 32 == 0, 1x1 / 3x3,
    stride 2, fused shortcut; GroupNorm-on-load with W = 32, H >= 4 or W = 16, H >= 8 and odd N;
    attention over 64, 128, 256 tokens.  Batches span images per tile > N, single tiles, one and
    several persistent waves and the N-split of a partial last wave."""
    r = np.random.default_rng(seed + fmt)
    fake = iter(range(0x10000, 0x10000 + 64 * 1000, 64))
    cases = []
    for c in range(n):
        op = L.Op()
        kind = ["conv_tc"] * 6 + ["conv_gn"] * 3 + ["attn"]
        kind = kind[int(r.integers(len(kind)))]
        N = int(r.choice([1, 2, 3, 5, 7, 37, 61, 129, 150, 257]))
        if kind == "attn":
            HW, Cc = int(r.choice([64, 128, 256])), int(r.choice([64, 128, 192, 256]))
            op.kind, op.engine = L.OP_ATTN, L.ENGINE_TC
            op.i[L.ATTN_N], op.i[L.ATTN_HW], op.i[L.ATTN_C], op.i[L.ATTN_DTYPE] = N, HW, Cc, fmt
            op.f[0] = float(Cc ** -0.5)
            op.inp[0], op.out[0] = next(fake), next(fake)
            if HW % 128 == 0 and r.random() < 0.6:
                op.i[L.ATTN_PROJ] = 1
                op.f[1] = 0.7071
                op.inp[1], op.inp[2], op.inp[3], op.out[1] = next(fake), next(fake), next(fake), next(fake)
            cases.append(op)
            continue
        op.kind = L.OP_CONV
        i = op.i
        if kind == "conv_gn":
            op.engine = L.ENGINE_TC_GN
            W = int(r.choice([16, 32]))
            H = _pow2(4 if W == 32 else 8, 64, r)
            OH, OW, ks, stride, pad = H, W, 3, 1, 1
            C1 = 64 * int(r.integers(1, 5))
            C2 = 64 * int(r.integers(0, 3))
            cout = 64 * int(r.choice([1, 2, 4, 8]))
            N = N | 1                             # odd tile counts: the last pair is half empty
        else:
            op.engine = L.ENGINE_TC
            OW = _pow2(4, 128, r)
            OH = int(r.choice([1, 2])) if r.random() < 0.25 else _pow2(4, 128, r)
            if OW * OH > 8192:
                OH = max(1, 8192 // OW)
            ks = int(r.choice([1, 3]))
            stride = 2 if (ks == 3 and r.random() < 0.25) else 1
            C1 = 64 * int(r.integers(1, 5))
            C2 = 64 * int(r.integers(0, 3)) if stride == 1 else 0
            cout = 32 * int(r.choice([1, 2, 3, 4, 6, 8, 12, 16]))
            if stride == 2:
                H, W, pad = 2 * OH + 1, 2 * OW + 1, 0
            else:
                H, W, pad = OH, OW, ks // 2
        if OH * OW * N > 400_000:
            N = max(1, 400_000 // (OH * OW))
        i[L.CONV_N], i[L.CONV_H], i[L.CONV_W], i[L.CONV_C1], i[L.CONV_C2] = N, H, W, C1, C2
        i[L.CONV_COUT], i[L.CONV_KS], i[L.CONV_STRIDE], i[L.CONV_PAD] = cout, ks, stride, pad
        i[L.CONV_OH], i[L.CONV_OW] = OH, OW
        i[L.CONV_IN_DTYPE] = i[L.CONV_OUT_DTYPE] = i[L.CONV_RES_DTYPE] = fmt
        op.f[0], op.f[1] = float(r.choice([1.0, 0.7071])), float(cout)
        op.inp[0], op.inp[4], op.out[0] = next(fake), next(fake), next(fake)
        if C2:
            op.inp[1] = next(fake)
        if r.random() < 0.7:
            op.inp[5] = next(fake)
        if r.random() < 0.5:
            op.inp[2] = next(fake)
        if r.random() < 0.5:
            op.inp[3] = next(fake)
            i[L.CONV_TEMB_OFF] = 32 * int(r.integers(0, 3))
            i[L.CONV_TEMB_BSTRIDE] = 0 if r.random() < 0.5 else i[L.CONV_TEMB_OFF] + cout + 32
        if kind == "conv_gn":
            op.inp[6] = next(fake)
            i[L.CONV_GN_SILU] = int(r.random() < 0.7)
        if stride == 1 and ks == 3 and r.random() < 0.35:     # fused 1x1 shortcut over cat(e1, e2)
            i[L.CONV_EXT_C1] = 64 * int(r.integers(1, 4))
            op.inp[8] = next(fake)
            if r.random() < 0.5:
                i[L.CONV_EXT_C2] = 64 * int(r.integers(1, 3))
                op.inp[9] = next(fake)
        if (OH * OW) % 32 == 0 and r.random() < 0.7:
            op.out[1] = next(fake)
        cases.append(op)
    return cases


@pytest.mark.parametrize("tier", ["bf16x3", "bf16"])
def test_tc_shape_sweep_vs_fp64_reference(tier):
    fmt = L.BF16S if tier == "bf16x3" else L.BF16
    failures, rejected, worst_by_class = [], [], {}
    for c, op in enumerate(_sweep_cases(fmt)):
        res = check_op(op, fmt, seed=1000 + c)
        if op.kind == L.OP_CONV and op.engine == L.ENGINE_TC:      # the planner's host mirror agrees
            assert (res is None) == (Plan._tc_eligible(op) != L.OK), describe(op)
        if res is None:
            rejected.append(describe(op) + f" N={op.i[0]}")
            print(f"sweep {tier} #{c:2d} {describe(op):52s} N={op.i[0]:<4d} rejected (PSLD_EUNSUPPORTED)")
            continue
        cls, w, fails = res
        _merge(worst_by_class, cls, w)
        print(f"sweep {tier} #{c:2d} {describe(op):52s} N={op.i[0]:<4d} {cls:13s} l2 {w['l2']:.2e} "
              f"max {w['max']:.2e} elem {w['elem']:.2e} stat {w['stat']:.2e}{'  FAIL' if fails else ''}")
        failures += [f"#{c} {describe(op)} N={op.i[0]}: {m}" for m in fails]
    _report([f"{tier} sweep: {len(rejected)} of 30 rejected: {rejected}"], worst_by_class)
    assert not failures, "\n".join(failures[:40])
