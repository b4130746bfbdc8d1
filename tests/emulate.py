"""TEST INFRASTRUCTURE — reference semantics of every ``psld_op`` kind.

``reference_op`` restates one op record as the header ``include/psld_b200.h`` documents it, in
plain torch arithmetic, on whatever device and floating dtype its inputs come in.
``tests/test_gpu_program_ops.py`` runs it in float64 on the GPU and compares every distinct op of
the benchmarked programs with the CUDA kernel.  ``run_plan`` executes a *dry* plan
(``psld_b200.program.build_plan(..., dry=True)``, host tensors) op by op in fp32, which validates
the HOST logic (layer order, weight packing, buffer wiring, epilogue flags, temb offsets) without a
GPU.  Nothing in ``psld_b200`` imports this module.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from oracle.psld_oracle import upfirdn2d  # noqa: E402
from psld_b200 import _lib as L  # noqa: E402

ALL = (Ellipsis,)


def _f(t):
    return t.to(torch.float32)


def _act_round(x, fmt):
    """Rounding of an intermediate the kernels store as an activation-format tensor core operand:
    bf16 plans round it to bf16, split-bf16 (16 significand bits) and fp32 plans keep it."""
    return x.to(torch.bfloat16).to(x.dtype) if fmt == L.BF16 else x


def _tc_weight(w, rows, fmt):
    """Tensor-core weight [rows, K]; split-bf16 planes [2][rows, K] are merged to hi + lo."""
    if fmt == L.BF16S and w.shape[0] == 2 * rows:
        w = w[:rows] + w[rows:]
    return w.reshape(rows, -1)


def _mg_sums(y_nhwc):
    """(sum, sum of squares) per sample x 4 channels of [N, ..., C]: the GroupNorm micro-group statistics."""
    v = y_nhwc.reshape(y_nhwc.shape[0], -1, y_nhwc.shape[-1] // 4, 4)
    return torch.stack([v.sum((1, 3)), (v * v).sum((1, 3))], -1)


def reference_op(op, get, fmt):
    """Reference result of one op record.

    ``get(ptr)`` returns the logical tensor behind a pointer (split-bf16 storage already decoded to
    its values, weight planes merged or not) or None for NULL; ``fmt`` is the activation format of
    the program (``L.F32``, ``L.BF16`` or ``L.BF16S``), which decides where the tensor-core kernels
    round intermediates.  Arithmetic runs in the dtype of the op's main input.

    Returns ``{out slot: (index, value, accumulate)}``: the op writes ``value`` (reshaped) into
    ``out[slot][index]`` and leaves every other element of that buffer alone, or adds it there when
    ``accumulate`` is set (GroupNorm statistics).  Values are unrounded: storing them in the output
    format is the caller's business."""
    i, f = op.i, op.f
    k = op.kind
    if k == L.OP_ZERO:
        if not op.out[0]:
            return {}
        n = (i[0] | (i[1] << 31)) // 8
        return {0: ((slice(0, n),), torch.zeros(n, dtype=torch.float64), False)}
    if k == L.OP_LAYOUT:
        N, Cc, HW = i[L.LAYOUT_N], i[L.LAYOUT_C], i[L.LAYOUT_HW]
        src = get(op.inp[0])
        if i[L.LAYOUT_DIR] == 1:
            return {0: (ALL, src.reshape(N, HW, Cc).permute(0, 2, 1), False)}
        cpad = i[L.LAYOUT_CPAD] or Cc
        cw = i[L.LAYOUT_CWRITE] or cpad
        y = src.new_zeros(N, HW, cw)
        y[..., :Cc] = src.reshape(N, Cc, HW).permute(0, 2, 1)
        return {0: ((Ellipsis, slice(0, cw)), y, False)}
    if k == L.OP_AXPBY:
        n = i[0] | (i[1] << 31)
        xa, ya = get(op.inp[0]).reshape(-1), get(op.inp[1])
        assert xa.numel() == n and (ya is None or ya.numel() == n)
        y = f[0] * xa if ya is None else f[0] * xa + f[1] * ya.reshape(-1)
        return {0: (ALL, y, False)}
    if k == L.OP_TEMB:
        assert not op.out[2], "step-counter time rows are not modelled"
        nt, nf = i[L.TEMB_NT], i[L.TEMB_NF]
        tt = get(op.inp[0]).reshape(-1)[:nt]
        dt = get(op.inp[2]).dtype
        t32 = _f(tt)
        # the embedding argument is formed in fp32 in the reference model (layerspp.py:40-41,
        # layers.py:500-514) and in the kernel; sin / cos and the MLP run in the compute dtype
        if i[L.TEMB_EMB] == 0:
            lt = t32 if i[L.TEMB_LOGGED] else torch.log(t32)
            xp = ((lt[:, None] * _f(get(op.inp[1]).reshape(-1))[None, :]) * 2) * np.float32(np.pi)
        else:
            half = nf // 2
            e = torch.exp(torch.arange(half, dtype=torch.float32, device=tt.device)
                          * -np.float32(np.log(np.float32(10000.0)) / np.float32(half - 1)))
            xp = t32[:, None] * e[None, :]
        xp = xp.to(dt)
        emb = torch.cat([torch.sin(xp), torch.cos(xp)], -1)
        if emb.shape[1] < nf:
            emb = F.pad(emb, (0, nf - emb.shape[1]))
        h = F.linear(emb, get(op.inp[2]), get(op.inp[3]))
        h = F.linear(F.silu(h), get(op.inp[4]), get(op.inp[5]))
        return {0: (ALL, F.linear(F.silu(h), get(op.inp[6]), get(op.inp[7])), False)}
    if k == L.OP_GN:
        N, HW, C1, C2, G = i[L.GN_N], i[L.GN_HW], i[L.GN_C1], i[L.GN_C2], i[L.GN_G]
        x1, x2 = get(op.inp[0]).reshape(N, HW, C1), get(op.inp[1])
        x2 = None if x2 is None else x2.reshape(N, HW, C2)
        xx = x1 if x2 is None else torch.cat([x1, x2], -1)
        Cc = C1 + C2
        if op.inp[4]:      # producer-side micro-group statistics must describe exactly x1 / x2
            for src, p in ((x1, op.inp[4]), (x2, op.inp[5])):
                if src is None:
                    continue
                st, ref = get(p), _mg_sums(src.double())
                assert st is not None and st.numel() == ref.numel(), (p, ref.shape)
                # bf16 plans: the producer summed unrounded fp32 values, tolerate the rounding
                st = st.reshape(ref.shape).double()
                assert float((st - ref).abs().max()) <= 2e-2 * float(ref.abs().max()) + 1e-3
        v = xx.reshape(N, HW, G, Cc // G)
        mean = v.mean((1, 3))
        var = ((v - mean[:, None, :, None]) ** 2).mean((1, 3))
        rstd = 1.0 / torch.sqrt(var + f[0])
        cpg = Cc // G
        gamma, beta = get(op.inp[2]).reshape(Cc), get(op.inp[3]).reshape(Cc)
        sc = rstd.repeat_interleave(cpg, 1) * gamma[None]            # [N, C]
        sh = beta[None] - mean.repeat_interleave(cpg, 1) * sc
        if i[L.GN_AFFINE_ONLY]:
            return {0: (ALL, torch.stack([sc, sh], -1), False)}
        y = xx * sc[:, None, :] + sh[:, None, :]
        if i[L.GN_SILU]:
            y = F.silu(y)
        return {0: (ALL, y, False)}
    if k == L.OP_FIR:
        N, H, W, Cc = i[L.FIR_N], i[L.FIR_H], i[L.FIR_W], i[L.FIR_C]
        KH = i[L.FIR_KH]
        ca = i[L.FIR_CACT] or Cc
        taps = np.asarray([f[j] for j in range(KH * KH)], np.float32).reshape(KH, KH)
        xx = get(op.inp[0]).reshape(N, H, W, Cc)[..., :ca].permute(0, 3, 1, 2)
        y = upfirdn2d(xx, taps, up=i[L.FIR_UP], down=i[L.FIR_DOWN], pad=(i[L.FIR_PAD0], i[L.FIR_PAD1]))
        return {0: ((Ellipsis, slice(0, ca)), y.permute(0, 2, 3, 1), False)}
    if k == L.OP_CONV:
        N, H, W = i[L.CONV_N], i[L.CONV_H], i[L.CONV_W]
        C1, C2, cout, ks = i[L.CONV_C1], i[L.CONV_C2], i[L.CONV_COUT], i[L.CONV_KS]
        OH, OW = i[L.CONV_OH], i[L.CONV_OW]
        Cin = C1 + C2
        tc = op.engine in (L.ENGINE_TC, L.ENGINE_TC_GN)
        assert i[L.CONV_IN_LAYOUT] == L.NHWC
        x1, x2 = get(op.inp[0]).reshape(N, H, W, C1), get(op.inp[1])
        xx = x1 if x2 is None else torch.cat([x1, x2.reshape(N, H, W, C2)], -1)
        if op.engine == L.ENGINE_TC_GN:      # GroupNorm(+SiLU) applied on load
            aff = get(op.inp[6]).reshape(N, Cin, 2)
            xx = xx * aff[:, None, None, :, 0] + aff[:, None, None, :, 1]
            if i[L.CONV_GN_SILU]:
                xx = F.silu(xx)
            xx = _act_round(xx, fmt)
        ne = i[L.CONV_EXT_C1] + i[L.CONV_EXT_C2] if tc else 0
        w = get(op.inp[4])
        w_ext = None
        if tc:
            w = _tc_weight(w, cout, fmt)
            if ne:      # fused 1x1 shortcut (K-extension)
                w_ext = w[:, ks * ks * Cin:].reshape(cout, ne, 1, 1)
            w = w[:, : ks * ks * Cin].reshape(cout, ks, ks, Cin).permute(0, 3, 1, 2)
        else:
            w = w.reshape(ks, ks, Cin, cout).permute(3, 2, 0, 1)
        bias = get(op.inp[5])
        y = F.conv2d(xx.permute(0, 3, 1, 2), w, None if bias is None else bias.reshape(cout),
                     stride=i[L.CONV_STRIDE], padding=i[L.CONV_PAD])
        assert y.shape[2] == OH and y.shape[3] == OW
        if w_ext is not None:
            e1, e2 = get(op.inp[8]), get(op.inp[9])
            e1 = e1.reshape(N, OH, OW, i[L.CONV_EXT_C1])
            x_ext = e1 if e2 is None else torch.cat([e1, e2.reshape(N, OH, OW, i[L.CONV_EXT_C2])], -1)
            y = y + F.conv2d(x_ext.permute(0, 3, 1, 2), w_ext)
        if op.inp[3]:
            tp = get(op.inp[3]).reshape(-1)
            off, bs = i[L.CONV_TEMB_OFF], i[L.CONV_TEMB_BSTRIDE]
            rows = tp[off:off + cout].expand(N, -1) if bs == 0 else tp.reshape(-1, bs)[:N, off:off + cout]
            y = y + rows[:, :, None, None]
        if op.inp[2]:
            y = y + get(op.inp[2]).reshape(N, OH, OW, cout).permute(0, 3, 1, 2)
        y = y * f[0]
        res = {}
        if op.out[1]:      # accumulated: the program zeroes the arena first
            res[1] = (ALL, _mg_sums(y.permute(0, 2, 3, 1)), True)
        if i[L.CONV_OUT_LAYOUT] == L.NCHW:
            valid = int(f[1]) if tc else cout
            res[0] = (ALL, y[:, :valid], False)
        else:
            res[0] = (ALL, y.permute(0, 2, 3, 1), False)
        return res
    if k == L.OP_ATTN:
        N, HW, Cc = i[L.ATTN_N], i[L.ATTN_HW], i[L.ATTN_C]
        qkv = get(op.inp[0]).reshape(N, HW, 3 * Cc)
        q, kk, v = qkv[..., :Cc], qkv[..., Cc:2 * Cc], qkv[..., 2 * Cc:]
        w = torch.softmax(torch.einsum("bqc,bkc->bqk", q, kk) * f[0], dim=-1)
        o = torch.einsum("bqk,bkc->bqc", w, v)
        if not i[L.ATTN_PROJ]:
            return {0: (ALL, o, False)}
        # fused NIN_3 + skip connection (+ statistics of the result)
        assert op.engine == L.ENGINE_TC and HW % 128 == 0
        b3 = get(op.inp[2])
        y = F.linear(_act_round(o, fmt), _tc_weight(get(op.inp[1]), Cc, fmt),
                     None if b3 is None else b3.reshape(Cc))
        y = (y + get(op.inp[3]).reshape(N, HW, Cc)) * f[1]
        res = {0: (ALL, y, False)}
        if op.out[1]:
            res[1] = (ALL, _mg_sums(y), True)
        return res
    raise AssertionError(f"no reference for op kind {op.kind}")


def run_plan(plan, x, t):
    """x: [B,in_ch,H,W] f32, t: [nt] f32 (tau, or log tau for a ``logged`` plan) -> eps."""
    T = {k.data_ptr(): k for k in plan.keep}
    get = lambda p: None if not p else _f(T[p])
    fmt = L.BF16 if plan.bf16 else (L.BF16S if plan.x3 else L.F32)
    plan.x_in.copy_(x)
    plan.time_buf.copy_(t)
    for op in plan.ops:
        if op.kind == L.OP_ZERO:
            if op.out[0]:
                ch = next(c for c in plan.stat_chunks if c.data_ptr() == op.out[0])
                nbytes = op.i[0] | (op.i[1] << 31)
                assert nbytes % 8 == 0 and nbytes // 8 <= ch.numel()
                ch[: nbytes // 8].zero_()
            continue
        for slot, (idx, v, acc) in reference_op(op, get, fmt).items():
            dst = T[op.out[slot]][idx]
            v = v.reshape(dst.shape)
            dst.add_(v) if acc else dst.copy_(v)
    return plan.eps.clone()
