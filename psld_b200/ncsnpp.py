"""NCSN++ score network on hand-written sm_100a kernels, drop-in for the reference module.

Contract kept (SURVEY.md §8b; reference ``main/models/score_fn/song_sde/ncsnpp.py:35-438``):
``cls(config)``; ``__call__(u: f32[B,in_ch,H,W], t: f32[B]) -> f32[B,out_ch,H,W]`` with ``t``
the forward diffusion time; parameters live under ``all_modules.<i>.<Sub>.<param>`` with the
reference's names and shapes, so Lightning checkpoints (``ema_score_fn.all_modules.*``) load
with ``load_state_dict``; the module survives ``deepcopy``/``eval``/``parameters``.

What is different is *how* it runs: the module tree below only HOLDS parameters.  The forward
is compiled once per (batch, #time rows) into a flat "program" of ``psld_op`` records
(``include/psld_b200.h``) with pre-packed weights and pre-allocated NHWC activation buffers,
and replayed by the native executor ``psld_program_run`` — there is no per-layer Python or
PyTorch dispatch on the hot path and no eager fallback.

Supported configuration space (the BASELINE configs, the shipped sampling scripts and the
high-resolution NCSN++ configurations of the score-SDE family): ``resblock_type=biggan``,
``progressive in {none,output_skip}``, ``progressive_input in {none,residual,input_skip}``,
``progressive_combine=sum``, ``embedding_type in {fourier,positional}``, ``fir in {True,False}``
(``progressive_input=residual`` needs ``fir=True``), ``nonlinearity=swish``, and any
``attn_resolutions``.  Attention runs on the tensor cores (``bf16``, ``bf16x3``) at C = 64..256
(multiple of 64) over 64, 128 or 256 tokens (all keys in one accumulator) or any multiple of 128
tokens from 512 (32x32 maps and larger: keys streamed with an online softmax); other shapes and
the ``fp32`` tier run it on the CUDA cores, which stream keys in chunks when a score row does not
fit in shared memory, so every map size runs.
"""
from __future__ import annotations

import ctypes as C
import math
import os

import numpy as np
import torch
import torch.nn as nn

from . import _lib as L

_SQRT1_2 = float(1.0 / np.sqrt(2.0))

# Precision tiers of the contractions (convolutions, NIN, attention):
#   "bf16x3"  split-bf16 operands, three tcgen05 MMAs per product (a_hi w_hi + a_hi w_lo + a_lo w_hi),
#             fp32 accumulation, split-bf16 activations: fp32-tolerance results on the tensor cores
#   "bf16"    bf16 operands and activations, fp32 accumulation (throughput tier, ~1e-2 per forward)
#   "fp32"    true fp32 FFMA on the CUDA cores (reference-faithful arithmetic)
PRECISIONS = ("fp32", "bf16", "bf16x3")


# ----------------------------------------------------------------------------------------
# Parameter containers (names/shapes = reference state-dict contract)
# ----------------------------------------------------------------------------------------
def _vs_uniform(shape, scale=1.0, in_axis=1, out_axis=0):
    """DDPM 'default_init': variance scaling, fan_avg, uniform (reference layers.py:39-76)."""
    scale = 1e-10 if scale == 0 else scale
    rf = float(np.prod(shape)) / shape[in_axis] / shape[out_axis]
    fan_avg = (shape[in_axis] + shape[out_axis]) * rf / 2.0
    bound = math.sqrt(3.0 * scale / fan_avg)
    return (torch.rand(*shape) * 2.0 - 1.0) * bound


def _conv(cin, cout, k, init_scale=1.0):
    m = nn.Conv2d(cin, cout, kernel_size=k, stride=1, padding=k // 2)
    m.weight.data = _vs_uniform(tuple(m.weight.shape), init_scale)
    nn.init.zeros_(m.bias)
    return m


def _dense(cin, cout):
    m = nn.Linear(cin, cout)
    m.weight.data = _vs_uniform(tuple(m.weight.shape))
    nn.init.zeros_(m.bias)
    return m


def _gn(c):
    return nn.GroupNorm(num_groups=min(c // 4, 32), num_channels=c, eps=1e-6)


class GaussianFourierProjection(nn.Module):
    """Holds the fixed frequencies ``W`` (reference layerspp.py:32-41)."""

    def __init__(self, embedding_size, scale):
        super().__init__()
        self.W = nn.Parameter(torch.randn(embedding_size) * scale, requires_grad=False)


class NIN(nn.Module):
    """``y = x W + b`` over channels, ``W[in, out]`` (reference layers.py:531-540)."""

    def __init__(self, in_dim, num_units, init_scale=0.1):
        super().__init__()
        self.W = nn.Parameter(_vs_uniform((in_dim, num_units), init_scale))
        self.b = nn.Parameter(torch.zeros(num_units))


class ResnetBlockBigGANpp(nn.Module):
    """Parameters of the BigGAN residual block (reference layerspp.py:212-240)."""

    def __init__(self, in_ch, out_ch=None, temb_dim=None, up=False, down=False, dropout=0.1,
                 init_scale=0.0):
        super().__init__()
        out_ch = out_ch if out_ch else in_ch
        self.GroupNorm_0 = _gn(in_ch)
        self.Conv_0 = _conv(in_ch, out_ch, 3)
        if temb_dim is not None:
            self.Dense_0 = _dense(temb_dim, out_ch)
        self.GroupNorm_1 = _gn(out_ch)
        self.Dropout_0 = nn.Dropout(dropout)     # inactive: sampling runs in eval mode
        self.Conv_1 = _conv(out_ch, out_ch, 3, init_scale)
        if in_ch != out_ch or up or down:
            self.Conv_2 = _conv(in_ch, out_ch, 1)
        self.in_ch, self.out_ch, self.up, self.down = in_ch, out_ch, up, down


class AttnBlockpp(nn.Module):
    """Parameters of the attention block (reference layerspp.py:62-73)."""

    def __init__(self, channels, init_scale=0.0):
        super().__init__()
        self.GroupNorm_0 = _gn(channels)
        self.NIN_0 = NIN(channels, channels)
        self.NIN_1 = NIN(channels, channels)
        self.NIN_2 = NIN(channels, channels)
        self.NIN_3 = NIN(channels, channels, init_scale=init_scale)
        self.channels = channels


class _FirConv(nn.Module):
    def __init__(self, in_ch, out_ch):
        super().__init__()
        self.weight = nn.Parameter(_vs_uniform((out_ch, in_ch, 3, 3)))
        self.bias = nn.Parameter(torch.zeros(out_ch))


class PyramidDownsample(nn.Module):
    """FIR-filtered stride-2 3x3 conv of the input pyramid (reference layerspp.py:129-163 with
    ``fir=True, with_conv=True`` -> up_or_down_sampling.Conv2d(down=True), :23-56,144-178)."""

    def __init__(self, in_ch, out_ch):
        super().__init__()
        self.Conv2d_0 = _FirConv(in_ch, out_ch)
        self.in_ch, self.out_ch = in_ch, out_ch


class Combine(nn.Module):
    """Merges the input pyramid into the down path: ``Conv_0(pyr) + h`` (reference layerspp.py:
    Combine with ``method='sum'``; ``Conv_0`` = ddpm_conv1x1)."""

    def __init__(self, dim1, dim2):
        super().__init__()
        self.Conv_0 = _conv(dim1, dim2, 1)


# ----------------------------------------------------------------------------------------
# The network
# ----------------------------------------------------------------------------------------
class NCSNpp(nn.Module):
    """NCSN++ (B200-native).  Registry name ``ncsnpp_b200`` (and optionally ``ncsnpp``)."""

    def __init__(self, config):
        super().__init__()
        self.full_config = config
        self.config = config.model
        sf = config.model.score_fn
        if str(sf.nonlinearity).lower() != "swish":
            raise NotImplementedError("psld_b200 NCSNpp: only nonlinearity=swish (SiLU)")
        if str(sf.resblock_type).lower() != "biggan":
            raise NotImplementedError("psld_b200 NCSNpp: only resblock_type=biggan")
        self.progressive = str(sf.progressive).lower()
        if self.progressive not in ("none", "output_skip"):
            raise NotImplementedError("psld_b200 NCSNpp: progressive must be none|output_skip")
        self.progressive_input = str(sf.progressive_input).lower()
        if self.progressive_input not in ("none", "residual", "input_skip"):
            raise NotImplementedError("psld_b200 NCSNpp: progressive_input must be none|residual|input_skip")
        combine = str(getattr(sf, "progressive_combine", "sum")).lower()
        if self.progressive_input == "input_skip" and combine != "sum":
            # cat would widen every skip tensor by the pyramid's channels: convolutions writing into a
            # channel slice of a wider buffer, which no known configuration needs
            raise NotImplementedError("psld_b200 NCSNpp: input_skip needs progressive_combine=sum")
        self.embedding_type = str(sf.embedding_type).lower()
        assert self.embedding_type in ["fourier", "positional"]
        self.nf = nf = int(sf.nf)
        self.ch_mult = [int(c) for c in sf.ch_mult]
        self.num_res_blocks = int(sf.num_res_blocks)
        self.attn_resolutions = [int(a) for a in sf.attn_resolutions]
        self.num_resolutions = len(self.ch_mult)
        self.image_size = int(config.data.image_size)
        self.all_resolutions = [self.image_size // (2 ** i) for i in range(self.num_resolutions)]
        self.noise_cond = bool(sf.noise_cond)
        self.fir = bool(sf.fir)
        self.fir_kernel = [float(v) for v in sf.fir_kernel]
        self.skip_rescale = bool(sf.skip_rescale)
        self.in_ch, self.out_ch = int(sf.in_ch), int(sf.out_ch)
        if self.progressive_input == "residual" and not self.fir:
            raise NotImplementedError("progressive_input=residual needs fir=True")
        init_scale = float(sf.init_scale)
        dropout = float(sf.dropout)
        prec = getattr(sf, "precision", None) if not isinstance(sf, dict) else sf.get("precision")
        # default = the fp32-tolerance tensor-core tier: swapping the registry names must not change
        # the numerics beyond fp32 tolerance; "bf16" (3x faster, ~5e-3 trajectory error) is opt-in
        self.precision = str(prec or os.environ.get("PSLD_B200_PRECISION", "bf16x3")).lower()
        assert self.precision in PRECISIONS, self.precision

        mods = []
        if self.embedding_type == "fourier":
            assert config.training.continuous, "Fourier features are only used for continuous training."
            mods.append(GaussianFourierProjection(nf, float(sf.fourier_scale)))
            embed_dim = 2 * nf
        else:
            embed_dim = nf
        temb_dim = None
        if self.noise_cond:
            mods.append(_dense(embed_dim, nf * 4))
            mods.append(_dense(nf * 4, nf * 4))
            temb_dim = nf * 4

        def RB(**kw):
            return ResnetBlockBigGANpp(temb_dim=temb_dim, dropout=dropout, init_scale=init_scale, **kw)

        pyr_ch = self.in_ch
        mods.append(_conv(self.in_ch, nf, 3))
        hs_c = [nf]
        in_ch = nf
        for lvl in range(self.num_resolutions):
            for _ in range(self.num_res_blocks):
                out_ch = nf * self.ch_mult[lvl]
                mods.append(RB(in_ch=in_ch, out_ch=out_ch))
                in_ch = out_ch
                if self.all_resolutions[lvl] in self.attn_resolutions:
                    mods.append(AttnBlockpp(in_ch, init_scale))
                hs_c.append(in_ch)
            if lvl != self.num_resolutions - 1:
                mods.append(RB(in_ch=in_ch, down=True))
                if self.progressive_input == "input_skip":
                    mods.append(Combine(pyr_ch, in_ch))       # pyr_ch stays in_ch of the network
                elif self.progressive_input == "residual":
                    mods.append(PyramidDownsample(pyr_ch, in_ch))
                    pyr_ch = in_ch
                hs_c.append(in_ch)
        in_ch = hs_c[-1]
        mods.append(RB(in_ch=in_ch))
        mods.append(AttnBlockpp(in_ch, init_scale))
        mods.append(RB(in_ch=in_ch))
        for lvl in reversed(range(self.num_resolutions)):
            for _ in range(self.num_res_blocks + 1):
                out_ch = nf * self.ch_mult[lvl]
                mods.append(RB(in_ch=in_ch + hs_c.pop(), out_ch=out_ch))
                in_ch = out_ch
            if self.all_resolutions[lvl] in self.attn_resolutions:
                mods.append(AttnBlockpp(in_ch, init_scale))
            if self.progressive == "output_skip":      # this level's output head
                mods.append(_gn(in_ch))
                mods.append(_conv(in_ch, self.out_ch, 3, init_scale))
            if lvl != 0:
                mods.append(RB(in_ch=in_ch, up=True))
        assert not hs_c
        if self.progressive != "output_skip":
            mods.append(_gn(in_ch))
            mods.append(_conv(in_ch, self.out_ch, 3, init_scale))
        self.all_modules = nn.ModuleList(mods)
        self._plans = {}

    # -- plan cache invalidation -----------------------------------------------------
    def _drop_plans(self):
        for p in self.__dict__.get("_plans", {}).values():
            p.release()
        self.__dict__["_plans"] = {}

    def load_state_dict(self, *a, **kw):
        r = super().load_state_dict(*a, **kw)
        self._drop_plans()
        return r

    def _apply(self, fn, *a, **kw):
        r = super()._apply(fn, *a, **kw)
        self._drop_plans()
        return r

    def __deepcopy__(self, memo):
        new = type(self)(self.full_config)
        new.precision = self.precision
        new.load_state_dict(self.state_dict())
        dev = next(self.parameters()).device
        new.to(dev)
        new.train(self.training)
        for p, q in zip(new.parameters(), self.parameters()):
            p.requires_grad = q.requires_grad
        return new

    def set_precision(self, precision: str):
        assert precision in PRECISIONS, precision
        if precision != self.precision:
            self.precision = precision
            self._drop_plans()
        return self

    # -- public call surface -----------------------------------------------------------
    def _fingerprint(self):
        """Cheap identity of the live parameter values: (storage pointer, in-place version counter)
        of every parameter.  Plans hold RE-PACKED copies of the weights (bf16 K-major, concatenated
        Dense_0, fused biases); an in-place update (``p.data.copy_``, an EMA step, an optimizer
        step, ``nn.init``) bumps ``_version`` and a re-assignment changes the pointer, so a stale
        plan is detected and rebuilt instead of silently running with old weights."""
        return tuple((p.data_ptr(), p._version) for p in self.parameters())

    def invalidate(self):
        """Drop every compiled plan (they are rebuilt, with re-packed weights, on next use)."""
        self._drop_plans()

    def plan(self, batch: int, nt: int, logged: bool):
        key = (int(batch), int(nt), bool(logged), self.precision)
        p = self._plans.get(key)
        fp = self._fingerprint()
        if p is not None and p.fingerprint != fp:
            p.release()
            p = None
        if p is None:
            from .program import build_plan
            p = build_plan(self, batch, nt, logged)
            p.fingerprint = fp
            self._plans[key] = p
        return p

    def forward(self, x, time_cond):
        """score_fn(u, t) -> eps (reference ``NCSNpp.forward``, ncsnpp.py:287-438)."""
        if not x.is_cuda:
            raise RuntimeError("psld_b200.NCSNpp runs on CUDA (sm_100a) only; there is no CPU path")
        if x.dim() != 4 or x.shape[1] != self.in_ch:
            raise ValueError(f"expected [B,{self.in_ch},H,W] input, got {tuple(x.shape)}")
        B = x.shape[0]
        p = self.plan(B, B, False)
        with torch.no_grad():
            p.x_in.copy_(x.to(torch.float32))
            p.time_buf.copy_(time_cond.to(torch.float32).reshape(-1).expand(B))
        p.run()
        return p.eps.clone()
