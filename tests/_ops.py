"""Test helpers: build single ``psld_op`` records and run them through the C ABI."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from psld_b200 import _lib as L


class Split(torch.Tensor):
    """Marker subclass: a float32-typed tensor whose BYTES are split bf16 ([C hi | C lo] per pixel
    row, include/psld_b200.h PSLD_BF16S); its logical shape is the float32 shape."""


def to_split(x):
    """fp32 [..., C] -> split-bf16 storage (returned as a float32-typed ``Split`` of the same shape)."""
    x = x.to(torch.float32)
    hi = x.to(torch.bfloat16)
    lo = (x - hi.to(torch.float32)).to(torch.bfloat16)
    return torch.cat([hi, lo], -1).contiguous().view(torch.float32).as_subclass(Split)


def from_split(t):
    """split-bf16 storage -> fp32 values (hi + lo)."""
    b = t.as_subclass(torch.Tensor).contiguous().view(torch.bfloat16)
    Cc = b.shape[-1] // 2
    return b[..., :Cc].to(torch.float32) + b[..., Cc:].to(torch.float32)


def split_like(shape, device):
    return torch.full(shape, float("nan"), dtype=torch.float32, device=device).as_subclass(Split)


def val(t):
    """Logical fp32/fp64-able values of a tensor in any activation format."""
    return from_split(t) if isinstance(t, Split) else t.as_subclass(torch.Tensor)


def code(t):
    return L.BF16S if isinstance(t, Split) else L.dtype_code(t.dtype)


def run_op(op, prepare=False):
    lib = L.lib()
    if prepare:
        L.check(lib.psld_op_prepare(C.byref(op)), "prepare")
    try:
        L.check(lib.psld_op_run(C.byref(op), L.stream_ptr()), "run")
        torch.cuda.synchronize()
    finally:
        if prepare:
            lib.psld_op_release(C.byref(op))


def conv_op(x1, x2, w_oihw, bias, *, stride=1, pad=None, residual=None, temb=None, temb_off=0,
            temb_bstride=0, scale=1.0, engine=L.ENGINE_SIMT, out_nchw_f32=False, out=None,
            mg_stats=False, affine=None, gn_silu=True, ext=None):
    """x*: NHWC tensors on cuda.  Returns (op, out, keepalive)."""
    N, H, W, C1 = x1.shape
    C2 = x2.shape[-1] if x2 is not None else 0
    Cout, Cin, ks, _ = w_oihw.shape
    assert Cin == C1 + C2
    pad = ks // 2 if pad is None else pad
    OH = (H + 2 * pad - ks) // stride + 1
    OW = (W + 2 * pad - ks) // stride + 1
    dev = x1.device
    keep = []
    op = L.Op()
    op.kind, op.engine = L.OP_CONV, engine
    i = op.i
    i[L.CONV_N], i[L.CONV_H], i[L.CONV_W], i[L.CONV_C1], i[L.CONV_C2] = N, H, W, C1, C2
    i[L.CONV_COUT], i[L.CONV_KS], i[L.CONV_STRIDE], i[L.CONV_PAD] = Cout, ks, stride, pad
    i[L.CONV_OH], i[L.CONV_OW] = OH, OW
    i[L.CONV_IN_LAYOUT] = L.NHWC
    i[L.CONV_OUT_LAYOUT] = L.NCHW if out_nchw_f32 else L.NHWC
    i[L.CONV_IN_DTYPE] = code(x1)
    i[L.CONV_OUT_DTYPE] = L.F32 if out_nchw_f32 else code(x1)
    i[L.CONV_RES_DTYPE] = code(x1)
    i[L.CONV_TEMB_OFF], i[L.CONV_TEMB_BSTRIDE] = temb_off, temb_bstride
    op.f[0] = scale
    cout_k = Cout
    w = w_oihw.to(dev, torch.float32)
    b = bias.to(dev, torch.float32).contiguous() if bias is not None else None
    if engine in (L.ENGINE_TC, L.ENGINE_TC_GN):
        if out_nchw_f32 and Cout % 32:
            cout_k = -(-Cout // (64 if engine == L.ENGINE_TC_GN else 32)) * (64 if engine == L.ENGINE_TC_GN else 32)
        wt = w.permute(0, 2, 3, 1).reshape(Cout, -1)
        if cout_k != Cout:
            wt = torch.cat([wt, wt.new_zeros(cout_k - Cout, wt.shape[1])], 0)
            if b is not None:
                b = torch.cat([b, b.new_zeros(cout_k - Cout)])
        if ext is not None:      # (e1, e2, w_ext [Cout, E, 1, 1]): fused 1x1 shortcut
            e1, e2, we = ext
            wt = torch.cat([wt, we.to(dev, torch.float32).reshape(Cout, -1)], 1)
            op.inp[8] = e1.data_ptr()
            op.inp[9] = e2.data_ptr() if e2 is not None else None
            i[L.CONV_EXT_C1] = e1.shape[-1]
            i[L.CONV_EXT_C2] = e2.shape[-1] if e2 is not None else 0
            keep += [e1, e2]
        if isinstance(x1, Split):      # weight planes [2][Cout, K]
            hi = wt.to(torch.bfloat16)
            wt = torch.cat([hi.to(torch.float32), wt - hi.to(torch.float32)], 0)
        wp = wt.to(torch.bfloat16).contiguous()
        i[L.CONV_COUT] = cout_k
        op.f[1] = float(Cout)
    else:
        wp = w.permute(2, 3, 1, 0).reshape(-1, Cout).contiguous()
    keep += [wp, b]
    if out is None:
        if out_nchw_f32:
            out = torch.full((N, Cout, OH, OW), float("nan"), dtype=torch.float32, device=dev)
        else:
            out = torch.full((N, OH, OW, Cout), float("nan"), dtype=x1.dtype, device=dev)
            if isinstance(x1, Split):
                out = out.as_subclass(Split)
    op.inp[0] = x1.data_ptr()
    op.inp[1] = x2.data_ptr() if x2 is not None else None
    op.inp[2] = residual.data_ptr() if residual is not None else None
    op.inp[3] = temb.data_ptr() if temb is not None else None
    op.inp[4] = wp.data_ptr()
    op.inp[5] = b.data_ptr() if b is not None else None
    op.out[0] = out.data_ptr()
    if affine is not None:
        op.inp[6] = affine.data_ptr()
        i[L.CONV_GN_SILU] = int(gn_silu)
        keep.append(affine)
    if mg_stats:
        mg = torch.zeros((N, Cout // 4, 2), dtype=torch.float64, device=dev)    # accumulated: zero first
        op.out[1] = mg.data_ptr()
        keep.append(mg)
    return op, out, keep


def conv_ref(x1, x2, w_oihw, bias, *, stride=1, pad=None, residual=None, temb=None, temb_off=0,
             temb_bstride=0, scale=1.0):
    """CPU fp32/fp64 reference of the op semantics (inputs NHWC, any device)."""
    import torch.nn.functional as F
    ks = w_oihw.shape[-1]
    pad = ks // 2 if pad is None else pad
    x1, x2, residual = val(x1), (val(x2) if x2 is not None else None), (val(residual) if residual is not None else None)
    xx = x1.double().cpu() if x2 is None else torch.cat([x1.double().cpu(), x2.double().cpu()], -1)
    y = F.conv2d(xx.permute(0, 3, 1, 2), w_oihw.double().cpu(),
                 bias.double().cpu() if bias is not None else None, stride=stride, padding=pad)
    Cout = w_oihw.shape[0]
    if temb is not None:
        tp = temb.double().cpu()
        rows = tp.reshape(-1)[temb_off:temb_off + Cout][None].expand(y.shape[0], -1) if temb_bstride == 0 \
            else tp[:, temb_off:temb_off + Cout]
        y = y + rows[:, :, None, None]
    if residual is not None:
        y = y + residual.double().cpu().permute(0, 3, 1, 2)
    return (y * scale)     # NCHW float64


def mg_ref(y_nhwc):
    """Per-sample micro-group statistics [N, C/4, 2] of an NHWC tensor (fp64)."""
    v = y_nhwc.double().cpu().reshape(y_nhwc.shape[0], -1, y_nhwc.shape[-1] // 4, 4)
    return torch.stack([v.sum((1, 3)), (v * v).sum((1, 3))], -1)


def gn_op(x1, x2, gamma, beta, G, silu, eps=1e-6, nchunk=4, out_dtype=None, mg1=None, mg2=None):
    N = x1.shape[0]
    HW = int(np.prod(x1.shape[1:-1]))
    C1 = x1.shape[-1]
    C2 = x2.shape[-1] if x2 is not None else 0
    out = torch.full((*x1.shape[:-1], C1 + C2), float("nan"), dtype=out_dtype or x1.dtype, device=x1.device)
    if isinstance(x1, Split):
        out = out.as_subclass(Split)
    scratch = torch.zeros(N * nchunk * G * 2 + 16, dtype=torch.float64, device=x1.device)
    op = L.Op()
    op.kind = L.OP_GN
    i = op.i
    i[L.GN_N], i[L.GN_HW], i[L.GN_C1], i[L.GN_C2], i[L.GN_G] = N, HW, C1, C2, G
    i[L.GN_SILU], i[L.GN_IN_DTYPE], i[L.GN_OUT_DTYPE], i[L.GN_NCHUNK] = int(silu), code(x1), code(out), nchunk
    op.f[0] = eps
    op.inp[0] = x1.data_ptr()
    op.inp[1] = x2.data_ptr() if x2 is not None else None
    op.inp[2], op.inp[3] = gamma.data_ptr(), beta.data_ptr()
    op.inp[4] = mg1.data_ptr() if mg1 is not None else None
    op.inp[5] = mg2.data_ptr() if mg2 is not None else None
    op.out[0], op.out[1] = out.data_ptr(), scratch.data_ptr()
    return op, out, [scratch]


def fir_op(x, taps, up, down, pad0, pad1):
    N, H, W, Cc = x.shape
    KH = taps.shape[0]
    OH = (H * up + pad0 + pad1 - KH) // down + 1
    OW = (W * up + pad0 + pad1 - KH) // down + 1
    out = torch.full((N, OH, OW, Cc), float("nan"), dtype=x.dtype, device=x.device)
    if isinstance(x, Split):
        out = out.as_subclass(Split)
    op = L.Op()
    op.kind = L.OP_FIR
    i = op.i
    i[L.FIR_N], i[L.FIR_H], i[L.FIR_W], i[L.FIR_C] = N, H, W, Cc
    i[L.FIR_UP], i[L.FIR_DOWN], i[L.FIR_PAD0], i[L.FIR_PAD1] = up, down, pad0, pad1
    i[L.FIR_KH], i[L.FIR_DTYPE] = KH, code(x)
    for j, v in enumerate(np.asarray(taps, np.float32).reshape(-1)):
        op.f[j] = float(v)
    op.inp[0], op.out[0] = x.data_ptr(), out.data_ptr()
    return op, out


def attn_op(qkv, Cc, engine=L.ENGINE_SIMT, proj=None):
    """proj = (w3 [out, in] f32, bias f32, x NHWC, scale): fused output projection + skip.
    Returns (op, out) or (op, out, keep) when proj is given (keep[-1] = statistics accumulator)."""
    N = qkv.shape[0]
    HW = int(np.prod(qkv.shape[1:-1]))
    out = torch.full((*qkv.shape[:-1], Cc), float("nan"), dtype=qkv.dtype, device=qkv.device)
    if isinstance(qkv, Split):
        out = out.as_subclass(Split)
    op = L.Op()
    op.kind, op.engine = L.OP_ATTN, engine
    op.i[L.ATTN_N], op.i[L.ATTN_HW], op.i[L.ATTN_C], op.i[L.ATTN_DTYPE] = N, HW, Cc, code(qkv)
    op.f[0] = float(int(Cc) ** (-0.5))
    op.inp[0], op.out[0] = qkv.data_ptr(), out.data_ptr()
    if proj is None:
        return op, out
    w3, b3, x, scale = proj
    w3 = w3.to(qkv.device, torch.float32)
    if isinstance(qkv, Split):          # weight planes [2][C out, C in]
        hi = w3.to(torch.bfloat16)
        w3 = torch.cat([hi.to(torch.float32), w3 - hi.to(torch.float32)], 0)
    wp = w3.to(torch.bfloat16).contiguous()
    bp = b3.to(qkv.device, torch.float32).contiguous()
    mg = torch.zeros((N, Cc // 4, 2), dtype=torch.float64, device=qkv.device)
    op.i[L.ATTN_PROJ] = 1
    op.f[1] = scale
    op.inp[1], op.inp[2], op.inp[3] = wp.data_ptr(), bp.data_ptr(), x.data_ptr()
    op.out[1] = mg.data_ptr()
    return op, out, [wp, bp, x, mg]


def rel_l2(a, b):
    a, b = val(a).double().cpu(), val(b).double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


def per_sample_rel_l2(a, b):
    """rel-L2 of every sample (leading dimension) separately, as a float64 tensor."""
    a, b = val(a).double(), val(b).double().to(val(a).device)
    d = (a - b).reshape(a.shape[0], -1).norm(dim=1)
    return (d / b.reshape(b.shape[0], -1).norm(dim=1).clamp_min(1e-300)).cpu()


def max_rel(a, b):
    a, b = val(a).double().cpu(), val(b).double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))
