"""TEST INFRASTRUCTURE — reference semantics of the NCSN++ pyramids and of the NCHW-head residual.

``ncsnpp_forward`` is Song's ``NCSNpp.forward`` (ncsnpp.py:287-438, layerspp.py ``Combine`` /
``Upsample`` / ``Downsample``) for ``progressive in {none, output_skip}``, ``progressive_input in
{none, residual, input_skip}`` with ``progressive_combine=sum``, in plain ATen ops on whatever device
and dtype its inputs come in; it is built from the blocks of ``oracle/psld_oracle.py`` and agrees with
that oracle's ``ncsnpp_forward`` where both apply.

``reference_op`` extends ``emulate.reference_op`` by the fp32 NCHW residual of the network head
(``include/psld_b200.h``: added to the valid output channels before the scale).  Tests install it with
``monkeypatch`` in place of ``emulate.reference_op`` (``run_plan``) and of the copy that
``test_gpu_program_ops`` imported (``check_op``).
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn.functional as F

import emulate
from oracle.psld_oracle import (_gn, attnblock, conv_downsample_2d, downsample_2d, resblock,
                                upsample_2d)
from psld_b200 import _lib as L

_reference_op = emulate.reference_op


def ncsnpp_forward(config, sd, x, time_cond):
    sf = config.model.score_fn
    nf, ch_mult, nrb = sf.nf, list(sf.ch_mult), sf.num_res_blocks
    nres = len(ch_mult)
    attn_res = list(sf.attn_resolutions)
    prog, pin = sf.progressive.lower(), sf.progressive_input.lower()
    assert sf.resblock_type.lower() == "biggan" and prog in ("none", "output_skip")
    assert pin in ("none", "residual", "input_skip")
    assert pin != "input_skip" or sf.get("progressive_combine", "sum").lower() == "sum"

    def pyr_down(v):                    # layerspp.Downsample(with_conv=False)
        return downsample_2d(v, sf.fir_kernel) if sf.fir else F.avg_pool2d(v, 2)

    def pyr_up(v):                      # layerspp.Upsample(with_conv=False)
        return upsample_2d(v, sf.fir_kernel) if sf.fir else F.interpolate(v, scale_factor=2, mode="nearest")

    key = lambda i: f"all_modules.{i}"
    i = 0
    if sf.embedding_type.lower() == "fourier":                     # layerspp.py:40
        W = sd[key(i) + ".W"]; i += 1
        xp = torch.log(time_cond)[:, None] * W[None, :] * 2 * np.pi
        temb = torch.cat([torch.sin(xp), torch.cos(xp)], dim=-1)
    else:                               # layers.py:500-514: the argument is formed in fp32
        half = nf // 2
        e = torch.exp(torch.arange(half, dtype=torch.float32, device=x.device) * -(math.log(10000) / (half - 1)))
        e = (time_cond.float()[:, None] * e[None, :]).to(x.dtype)
        temb = torch.cat([torch.sin(e), torch.cos(e)], dim=1)
    temb = F.linear(temb, sd[key(i) + ".weight"], sd[key(i) + ".bias"]); i += 1
    temb = F.linear(F.silu(temb), sd[key(i) + ".weight"], sd[key(i) + ".bias"]); i += 1
    pyr = x if pin != "none" else None
    hs = [F.conv2d(x, sd[key(i) + ".weight"], sd[key(i) + ".bias"], padding=1)]; i += 1
    for lvl in range(nres):
        for _ in range(nrb):
            h = resblock(sd, key(i), hs[-1], temb, sf); i += 1
            if h.shape[-1] in attn_res:
                h = attnblock(sd, key(i), h, sf.skip_rescale); i += 1
            hs.append(h)
        if lvl != nres - 1:
            h = resblock(sd, key(i), hs[-1], temb, sf, down=True); i += 1
            if pin == "input_skip":                                # Combine(method="sum")
                pyr = pyr_down(pyr)
                p = key(i) + ".Conv_0"; i += 1
                h = F.conv2d(pyr, sd[p + ".weight"], sd[p + ".bias"]) + h
            elif pin == "residual":                                # ncsnpp.py:350-357
                p = key(i) + ".Conv2d_0"; i += 1
                pyr = conv_downsample_2d(pyr, sd[p + ".weight"], sf.fir_kernel) + sd[p + ".bias"].reshape(1, -1, 1, 1)
                pyr = (pyr + h) / np.sqrt(2.0) if sf.skip_rescale else pyr + h
                h = pyr
            hs.append(h)
    h = hs[-1]
    h = resblock(sd, key(i), h, temb, sf); i += 1
    h = attnblock(sd, key(i), h, sf.skip_rescale); i += 1
    h = resblock(sd, key(i), h, temb, sf); i += 1
    out_pyr = None
    for lvl in reversed(range(nres)):
        for _ in range(nrb + 1):
            h = resblock(sd, key(i), torch.cat([h, hs.pop()], dim=1), temb, sf); i += 1
        if h.shape[-1] in attn_res:
            h = attnblock(sd, key(i), h, sf.skip_rescale); i += 1
        if prog == "output_skip":                                  # ncsnpp.py:405-418
            ph = F.silu(_gn(sd, key(i), h)); i += 1
            ph = F.conv2d(ph, sd[key(i) + ".weight"], sd[key(i) + ".bias"], padding=1); i += 1
            out_pyr = ph if out_pyr is None else pyr_up(out_pyr) + ph
        if lvl != 0:
            h = resblock(sd, key(i), h, temb, sf, up=True); i += 1
    assert not hs
    if prog == "output_skip":
        h = out_pyr
    else:
        h = F.silu(_gn(sd, key(i), h)); i += 1
        h = F.conv2d(h, sd[key(i) + ".weight"], sd[key(i) + ".bias"], padding=1); i += 1
    assert i == 1 + max(int(k.split(".")[1]) for k in sd), i
    return h


class ScoreFn:
    """score_fn(u, t) -> eps backed by ``ncsnpp_forward`` (fp32 on the CPU, like oracle.OracleScoreFn)."""

    def __init__(self, config, sd):
        self.config = config
        self.sd = {k: v.detach().to(torch.float32).cpu() for k, v in sd.items()}

    def __call__(self, u, t):
        with torch.no_grad():
            return ncsnpp_forward(self.config, self.sd, u, t)


def reference_op(op, get, fmt):
    """``emulate.reference_op`` plus the fp32 NCHW residual of an NCHW-output convolution."""
    i = op.i
    if not (op.kind == L.OP_CONV and i[L.CONV_OUT_LAYOUT] == L.NCHW and op.inp[2]):
        return _reference_op(op, get, fmt)
    assert i[L.CONV_RES_DTYPE] == L.F32
    bare = L.Op.from_buffer_copy(op)
    bare.inp[2] = None
    out = _reference_op(bare, get, fmt)
    idx, y, acc = out[0]
    N, V, OH, OW = y.shape
    out[0] = (idx, y + op.f[0] * get(op.inp[2]).reshape(N, V, OH, OW).to(y.dtype), acc)
    return out
