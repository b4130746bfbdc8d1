"""Compiles an :class:`psld_b200.ncsnpp.NCSNpp` into a flat program of ``psld_op`` records.

One plan = one (batch, #time rows, precision) instantiation of the reference forward
(``main/models/score_fn/song_sde/ncsnpp.py:287-438``): weights re-packed into the kernel
layouts, every activation buffer pre-allocated (NHWC, fp32 or bf16), and the layer sequence
unrolled into ops the native executor replays (``psld_program_run`` / ``psld_sampler_run``).

Fusions relative to the reference's eager graph (SURVEY.md §3.2, §7.3-4):
  * ``torch.cat([h, skip])`` is never materialised: GroupNorm and the 1x1 shortcut read two
    sources;
  * bias, ``Dense_0(SiLU(temb))`` add, shortcut add and the ``1/sqrt(2)`` rescale live in the
    convolution epilogue;
  * q, k, v NIN projections are one GEMM with a [C, 3C] weight;
  * the 2-layer temb MLP and all per-block ``Dense_0`` projections are computed once per call
    (and for ONE time row when the whole batch shares t, as it does during sampling);
  * (bf16 plans) GroupNorm statistics are accumulated by the producing convolution's epilogue and
    ``act(GroupNorm(.))`` is applied on load inside the consuming 3x3 convolution where the shape
    allows (GroupNorm_0 -> Conv_0, and GroupNorm_1 -> Conv_1 of identity-shortcut blocks);
  * (bf16 plans) the 1x1 ``Conv_2`` shortcut is appended to ``Conv_1`` as extra K-blocks, and the
    attention block's output projection + skip connection run inside the attention kernel.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib as L

_SQRT1_2 = float(1.0 / np.sqrt(2.0))


def _fir_taps(k1d, gain):
    """``_setup_kernel`` (reference up_or_down_sampling.py:181-188) * gain, as float32."""
    k = np.asarray(k1d, dtype=np.float32)
    if k.ndim == 1:
        k = np.outer(k, k)
    k /= np.sum(k)
    return (k * gain).astype(np.float32)


class Plan:
    def __init__(self, net, B, nt, logged, dry=False):
        self.lib = L.lib()
        self.net = net
        self.B, self.nt, self.logged = int(B), int(nt), bool(logged)
        self.dev = next(net.parameters()).device
        # dry = structural build on host tensors (tests of the builder logic only): the ops are
        # never launched and TC eligibility is decided by the same rules as psld_op_prepare.
        self.dry = bool(dry)
        if self.dev.type != "cuda" and not self.dry:
            raise RuntimeError("psld_b200: parameters must be on a CUDA device (no CPU path)")
        self.bf16 = net.precision == "bf16"
        # "bf16x3": split-bf16 activations / weights (value = hi + lo, [C hi | C lo] pixel rows = 4
        # bytes per element, so the buffers are ALLOCATED as float32 of the logical shape) and
        # three tcgen05 MMA groups per k-block: fp32-tolerance results on the tensor cores
        self.x3 = net.precision == "bf16x3"
        self.tc = self.bf16 or self.x3
        self.adt = torch.bfloat16 if self.bf16 else torch.float32
        self.acode = L.BF16 if self.bf16 else (L.BF16S if self.x3 else L.F32)
        self.keep = []          # tensors referenced by raw pointers
        self.ops = []
        self.pool = {}
        self.engine_count = {"tc": 0, "simt": 0}
        self.cin_valid = {}     # op index -> real input channels of convs over a zero-padded input
        self.mg = {}            # data_ptr of an activation -> its GroupNorm statistics accumulator
        self.stat_chunks = []   # f64 arenas the accumulators are carved from (zeroed by OP_ZERO)
        self.stat_used = []
        self.temb_op = -1
        self._build()
        self.n_ops = len(self.ops)
        self.op_array = (L.Op * self.n_ops)(*self.ops)
        self.launches = self.lib.psld_program_launches(self.op_array, self.n_ops)

    # ---------------------------------------------------------------- helpers
    def _new(self, *shape, dtype=None):
        t = torch.empty(*shape, dtype=dtype or self.adt, device=self.dev)
        self.keep.append(t)
        return t

    def _acquire(self, *shape):
        key = tuple(shape)
        lst = self.pool.setdefault(key, [])
        if lst:
            return lst.pop()
        return self._new(*shape)

    def _release_affine(self, t):
        self.pool.setdefault(("aff",) + tuple(t.shape), []).append(t)

    def _gn_fusable(self, x1, x2, cout):
        """Host mirror of prepare_conv_gn_tc (csrc/conv_gn_tc.cu): can act(GroupNorm(x)) -> conv3x3
        run as ONE kernel that normalises its input tile in shared memory?"""
        if not self.tc:
            return False
        N, H, W, C1 = x1.shape
        C2 = x2.shape[-1] if x2 is not None else 0
        if C1 % 64 or C2 % 64 or cout % 64 or (cout > 256 and cout % 256):
            return False
        if not ((W == 32 and H >= 4) or (W == 16 and H >= 8)) or (H & (H - 1)):
            return False
        return N * (H // (128 // W)) >= 2

    def _ext_fusable(self, b, e1, e2, cout):
        """Can Conv_2 (1x1 shortcut over e = cat(e1, e2)) ride along Conv_1's MMA stream?"""
        if not self.tc:
            return False
        N, H, W, Cb = b.shape
        E1 = e1.shape[-1]
        E2 = e2.shape[-1] if e2 is not None else 0
        pow2 = lambda v: v > 0 and (v & (v - 1)) == 0
        if self.x3 and (H * W) % 32:        # split-bf16 output goes through the staged epilogue only
            return False
        return (Cb % 64 == 0 and E1 % 64 == 0 and E2 % 64 == 0 and cout % 32 == 0 and pow2(W)
                and pow2(H) and 4 <= W <= 256 and tuple(e1.shape[:3]) == (N, H, W))

    def _release(self, t):
        self.pool.setdefault(tuple(t.shape), []).append(t)
        self.mg.pop(t.data_ptr(), None)     # accumulators are never reused within a step

    _STAT_CHUNK = 1 << 22       # doubles per arena (32 MB)
    _STAT_SLOTS = 4             # OP_ZERO placeholders at the top of the program

    def _mg_buffer(self, n, cout):
        """f64 [n, cout/4, 2] accumulator (sum, sumsq per sample x 4 channels), carved from an
        arena that one OP_ZERO clears at the top of every program run."""
        need = n * (cout // 4) * 2
        if not self.stat_chunks or self.stat_used[-1] + need > self.stat_chunks[-1].numel():
            if len(self.stat_chunks) == self._STAT_SLOTS:
                raise RuntimeError("psld_b200: GroupNorm statistics arena exhausted")
            # arena size grows with the batch (~18 K doubles per sample for the CIFAR-10 net): at most
            # _STAT_SLOTS arenas may be needed, whatever the batch
            chunk = max(self._STAT_CHUNK, 1 << int(self.B * 6000).bit_length())
            self.stat_chunks.append(self._new(max(chunk, need), dtype=torch.float64))
            self.stat_used.append(0)
        off = self.stat_used[-1]
        self.stat_used[-1] = off + need
        view = self.stat_chunks[-1].narrow(0, off, need).view(n, cout // 4, 2)
        self.keep.append(view)
        return view

    def _finish_stat_arenas(self, zero_ops):
        for k, idx in enumerate(zero_ops):
            op = self.ops[idx]
            if k < len(self.stat_chunks):
                nbytes = self.stat_used[k] * 8
                op.out[0] = self.stat_chunks[k].data_ptr()
                op.i[0], op.i[1] = nbytes & 0x7FFFFFFF, nbytes >> 31

    def _w(self, t, dtype=torch.float32):
        t = t.detach().to(device=self.dev, dtype=dtype).contiguous()
        self.keep.append(t)
        return t

    def _w_bf16(self, w):
        """fp32 weight [rows, K] as a tensor-core operand: bf16, or for split-bf16 plans the planes
        [2][rows, K] with hi = rn(w), lo = rn(w - hi)."""
        if self.x3:
            hi = w.to(torch.bfloat16)
            w = torch.cat([hi, (w - hi.to(torch.float32)).to(torch.bfloat16)], 0)
        return self._w(w, torch.bfloat16)

    def _pack_tc_conv(self, op, w, b32, ext, cout_pad):
        """Weight and bias of a tensor-core convolution: w [Cout, Cin, ks, ks] becomes [cout_pad, K]
        (K = taps x channels, channels fastest) with zero rows beyond Cout.  A fused 1x1 shortcut
        ``ext = (e1, e2, w_sc, b_sc)`` is appended along K: its input becomes a second A source
        (centre tap) and its bias joins the conv bias."""
        Cout = w.shape[0]
        wt = w.permute(0, 2, 3, 1).reshape(Cout, -1)
        if ext is not None:
            e1, e2, we, be = ext
            wt = torch.cat([wt, we.detach().to(self.dev, torch.float32).reshape(Cout, -1)], 1)
            op.inp[8] = e1.data_ptr()
            op.inp[9] = e2.data_ptr() if e2 is not None else None
            op.i[L.CONV_EXT_C1] = e1.shape[-1]
            op.i[L.CONV_EXT_C2] = e2.shape[-1] if e2 is not None else 0
            if be is not None:
                b32 = self._w((b32 if b32 is not None else 0) + be.detach().to(self.dev, torch.float32))
        if cout_pad != Cout:
            wt = torch.cat([wt, wt.new_zeros(cout_pad - Cout, wt.shape[1])], 0)
            if b32 is not None:
                b32 = self._w(torch.cat([b32, b32.new_zeros(cout_pad - Cout)]))
        op.i[L.CONV_COUT] = cout_pad
        op.inp[4] = self._w_bf16(wt).data_ptr()
        op.inp[5] = b32.data_ptr() if b32 is not None else None

    def _op(self, kind, engine=L.ENGINE_SIMT):
        op = L.Op()
        op.kind = kind
        op.engine = engine
        return op

    def _push(self, op):
        self.ops.append(op)
        return len(self.ops) - 1

    # ---------------------------------------------------------------- op builders
    def op_layout(self, src, dst, N, Cc, HW, direction, cpad=0, cwrite=0):
        op = self._op(L.OP_LAYOUT)
        op.i[L.LAYOUT_N], op.i[L.LAYOUT_C], op.i[L.LAYOUT_HW] = N, Cc, HW
        op.i[L.LAYOUT_DIR], op.i[L.LAYOUT_DTYPE], op.i[L.LAYOUT_CPAD] = direction, self.acode, cpad
        op.i[L.LAYOUT_CWRITE] = cwrite
        op.inp[0], op.out[0] = src.data_ptr(), dst.data_ptr()
        self._push(op)

    def op_gn(self, x1, x2, gn_mod, silu, HW, affine_only=False):
        """GroupNorm(+SiLU) over cat(x1, x2) -> new [B, HW.., C1+C2] buffer; with ``affine_only``
        only the per-(sample, channel) (scale, shift) pair [B, C, 2] fp32 is produced, for a
        convolution that normalises its input on load (PSLD_ENGINE_TC_GN)."""
        C1 = x1.shape[-1]
        C2 = x2.shape[-1] if x2 is not None else 0
        Cc = C1 + C2
        G = gn_mod.num_groups
        assert gn_mod.num_channels == Cc, (gn_mod.num_channels, Cc)
        if affine_only:
            key = ("aff", self.B, Cc, 2)
            lst = self.pool.setdefault(key, [])
            y = lst.pop() if lst else self._new(self.B, Cc, 2, dtype=torch.float32)
        else:
            y = self._acquire(*x1.shape[:-1], Cc)
        # stats pass: ~64 KB of input per CTA, but enough CTAs to fill 148 SMs at small batch
        per_img = HW * Cc * (2 if self.bf16 else 4)      # (split bf16 = 4 bytes per element too)
        nchunk = max(-(-per_img // 65536), -(-592 // self.B))
        nchunk = int(max(1, min(nchunk, max(1, HW // 32))))
        op = self._op(L.OP_GN)
        i = op.i
        i[L.GN_N], i[L.GN_HW], i[L.GN_C1], i[L.GN_C2], i[L.GN_G] = self.B, HW, C1, C2, G
        i[L.GN_SILU], i[L.GN_IN_DTYPE], i[L.GN_OUT_DTYPE], i[L.GN_NCHUNK] = int(silu), self.acode, self.acode, nchunk
        i[L.GN_AFFINE_ONLY] = int(affine_only)
        op.f[0] = float(gn_mod.eps)
        op.inp[0] = x1.data_ptr()
        op.inp[1] = x2.data_ptr() if x2 is not None else None
        op.inp[2] = self._w(gn_mod.weight).data_ptr()
        op.inp[3] = self._w(gn_mod.bias).data_ptr()
        op.out[0] = y.data_ptr()
        s1 = self.mg.get(x1.data_ptr())
        s2 = self.mg.get(x2.data_ptr()) if x2 is not None else None
        if s1 is not None and (x2 is None or s2 is not None) and (Cc // G) % 4 == 0:
            op.inp[4] = s1.data_ptr()
            op.inp[5] = s2.data_ptr() if s2 is not None else None
            self.engine_count["gn_fused_stats"] = self.engine_count.get("gn_fused_stats", 0) + 1
        need = self.B * nchunk * G * 2
        if self.gn_scratch is None or self.gn_scratch.numel() < need:
            self.gn_scratch = self._new(max(need, 1 << 16), dtype=torch.float64)
            for o in self.ops:       # re-point earlier GN ops at the (larger) scratch
                if o.kind == L.OP_GN:
                    o.out[1] = self.gn_scratch.data_ptr()
        op.out[1] = self.gn_scratch.data_ptr()
        self._push(op)
        return y

    def op_fir(self, x, taps, up, down, pad0, pad1, cact=0, f32=False):
        """upfirdn2d over NHWC ``x``; ``f32``: over a float32 tensor whatever the plan's format."""
        N, H, W, Cc = x.shape
        KH = taps.shape[0]
        OH = (H * up + pad0 + pad1 - KH) // down + 1
        OW = (W * up + pad0 + pad1 - KH) // down + 1
        if f32:
            cact = 0
            y = self._new(N, OH, OW, Cc, dtype=torch.float32)
        elif cact and cact < Cc:
            # only the first `cact` channels carry data (zero-padded network input): the output's
            # padding channels keep the zeros of a dedicated, never-pooled buffer
            y = torch.zeros(N, OH, OW, Cc, dtype=self.adt, device=self.dev)
            self.keep.append(y)
        else:
            cact = 0
            y = self._acquire(N, OH, OW, Cc)
        op = self._op(L.OP_FIR)
        i = op.i
        i[L.FIR_N], i[L.FIR_H], i[L.FIR_W], i[L.FIR_C] = N, H, W, Cc
        i[L.FIR_UP], i[L.FIR_DOWN], i[L.FIR_PAD0], i[L.FIR_PAD1] = up, down, pad0, pad1
        i[L.FIR_KH], i[L.FIR_DTYPE], i[L.FIR_CACT] = KH, L.F32 if f32 else self.acode, cact
        for j, v in enumerate(taps.reshape(-1)):
            op.f[j] = float(v)
        op.inp[0], op.out[0] = x.data_ptr(), y.data_ptr()
        self._push(op)
        return y

    def op_conv(self, x1, x2, w_oihw, bias, *, ks, stride=1, pad=None, residual=None,
                temb_off=-1, scale=1.0, out=None, in_nchw=False, out_nchw_f32=False,
                hw=None, allow_tc=True, want_stats=True, affine=None, gn_silu=True, ext=None):
        """y = scale * (conv(cat(x1,x2), w) + bias + temb + residual); w is [Cout, Cin, ks, ks].
        With ``out_nchw_f32`` the residual, if any, is an fp32 NCHW [N, Cout, OH, OW] tensor."""
        pad = ks // 2 if pad is None else pad
        if in_nchw:
            N, C1, H, W = x1.shape
        else:
            N, H, W, C1 = x1.shape
        C2 = x2.shape[-1] if x2 is not None else 0
        Cout = w_oihw.shape[0]
        cin_real = None
        if x2 is None and w_oihw.shape[1] < C1:       # zero-padded input channels (6 -> 64)
            cin_real = int(w_oihw.shape[1])
            w_oihw = torch.cat([w_oihw.detach(), w_oihw.new_zeros(
                Cout, C1 - w_oihw.shape[1], *w_oihw.shape[2:])], 1)
        assert w_oihw.shape[1] == C1 + C2, (tuple(w_oihw.shape), C1, C2)
        OH = (H + 2 * pad - ks) // stride + 1
        OW = (W + 2 * pad - ks) // stride + 1
        if out is None:
            out = self._new(N, Cout, OH, OW, dtype=torch.float32) if out_nchw_f32 \
                else self._acquire(N, OH, OW, Cout)
        op = self._op(L.OP_CONV)
        i = op.i
        i[L.CONV_N], i[L.CONV_H], i[L.CONV_W], i[L.CONV_C1], i[L.CONV_C2] = N, H, W, C1, C2
        i[L.CONV_COUT], i[L.CONV_KS], i[L.CONV_STRIDE], i[L.CONV_PAD] = Cout, ks, stride, pad
        i[L.CONV_OH], i[L.CONV_OW] = OH, OW
        i[L.CONV_IN_LAYOUT] = L.NCHW if in_nchw else L.NHWC
        i[L.CONV_OUT_LAYOUT] = L.NCHW if out_nchw_f32 else L.NHWC
        i[L.CONV_IN_DTYPE] = L.F32 if in_nchw else self.acode
        i[L.CONV_OUT_DTYPE] = L.F32 if out_nchw_f32 else self.acode
        i[L.CONV_RES_DTYPE] = L.F32 if (out_nchw_f32 and residual is not None) else self.acode
        if temb_off >= 0:
            i[L.CONV_TEMB_OFF] = temb_off
            i[L.CONV_TEMB_BSTRIDE] = 0 if self.nt == 1 else self.total_c
            op.inp[3] = self.temb_proj.data_ptr()
        op.f[0] = float(scale)
        op.inp[0] = x1.data_ptr()
        op.inp[1] = x2.data_ptr() if x2 is not None else None
        op.inp[2] = residual.data_ptr() if residual is not None else None
        b32 = self._w(bias) if bias is not None else None
        op.inp[5] = b32.data_ptr() if b32 is not None else None
        op.out[0] = out.data_ptr()
        w = w_oihw.detach().to(self.dev, torch.float32)
        done = False
        if affine is not None:
            # GroupNorm(+SiLU) applied on load inside the tensor-core kernel; the network head's
            # zero rows fill a 64-wide N tile
            op.engine = L.ENGINE_TC_GN
            op.inp[6] = affine.data_ptr()
            i[L.CONV_GN_SILU] = int(gn_silu)
            self._pack_tc_conv(op, w, b32, ext, -(-Cout // 64) * 64 if out_nchw_f32 else Cout)
            if out_nchw_f32:
                op.f[1] = float(Cout)
            mg = None
            if want_stats and not out_nchw_f32 and (OH * OW) % 32 == 0:
                mg = self._mg_buffer(N, Cout)
                op.out[1] = mg.data_ptr()
            if not self.dry:
                L.check(self.lib.psld_op_prepare(C.byref(op)), "psld_op_prepare(conv_gn)")
            if mg is not None:
                self.mg[out.data_ptr()] = mg
            self.engine_count["tc_gn"] = self.engine_count.get("tc_gn", 0) + 1
            done = True
        elif self.tc and allow_tc and not in_nchw:
            op.engine = L.ENGINE_TC
            # NCHW head: zero rows up to a 32-wide N tile, the epilogue writes Cout planes
            self._pack_tc_conv(op, w, b32, ext, -(-Cout // 32) * 32 if out_nchw_f32 else Cout)
            op.f[1] = float(Cout)                    # valid output channels (NCHW f32 epilogue)
            mg = None
            if want_stats and not out_nchw_f32 and (OH * OW) % 32 == 0 and Cout % 32 == 0:
                mg = self._mg_buffer(N, Cout)
                op.out[1] = mg.data_ptr()
            rc = self._tc_eligible(op) if self.dry else self.lib.psld_op_prepare(C.byref(op))
            if rc == L.OK and mg is not None:
                self.mg[out.data_ptr()] = mg
            elif mg is not None:
                op.out[1] = None
            if rc == L.OK:
                done = True
                self.engine_count["tc"] += 1
            elif rc != L.EUNSUPPORTED:
                L.check(rc, "psld_op_prepare(conv)")
            else:
                if ext is not None:
                    raise RuntimeError("psld_b200: fused 1x1 shortcut requested for a conv the "
                                       "tensor-core engine rejected: " +
                                       self.lib.psld_last_error().decode(errors="replace"))
                i[L.CONV_COUT] = Cout
                if bias is not None:
                    op.inp[5] = self._w(bias).data_ptr()
        if not done:
            op.engine = L.ENGINE_SIMT
            ws = self._w(w.permute(2, 3, 1, 0).reshape(-1, Cout))     # [K, Cout] fp32
            op.inp[4] = ws.data_ptr()
            self.engine_count["simt"] += 1
        idx = self._push(op)
        if cin_real is not None:
            self.cin_valid[idx] = cin_real
        return out

    @staticmethod
    def _tc_eligible(op):
        """Host mirror of prepare_conv_tc's eligibility rules (csrc/conv_tc.cu), dry builds only."""
        i = op.i
        pow2 = lambda v: v > 0 and (v & (v - 1)) == 0
        ks = i[L.CONV_KS]
        same = i[L.CONV_STRIDE] == 1 and ks in (1, 3) and i[L.CONV_PAD] == ks // 2
        down2 = i[L.CONV_STRIDE] == 2 and i[L.CONV_PAD] == 0 and ks == 3 and i[L.CONV_C2] == 0
        # output rows up to 128 pixels wide are tiled by whole rows; 256-wide rows (stride 1 only) as two
        # 128-pixel halves
        ow_max = 256 if same else 128
        ok = (i[L.CONV_IN_DTYPE] in (L.BF16, L.BF16S) and i[L.CONV_IN_LAYOUT] == L.NHWC and (same or down2)
              and i[L.CONV_C1] % 64 == 0 and i[L.CONV_C2] % 64 == 0 and i[L.CONV_COUT] % 32 == 0
              and pow2(i[L.CONV_OW]) and pow2(i[L.CONV_OH]) and 4 <= i[L.CONV_OW] <= ow_max)
        if i[L.CONV_OUT_LAYOUT] == L.NCHW and op.inp[2]:      # head residual: the fp32 NCHW pyramid
            ok = ok and i[L.CONV_RES_DTYPE] == L.F32
        if i[L.CONV_IN_DTYPE] == L.BF16S and i[L.CONV_OUT_LAYOUT] == L.NHWC:
            ok = ok and (i[L.CONV_OH] * i[L.CONV_OW]) % 32 == 0
        return L.OK if ok else L.EUNSUPPORTED

    @staticmethod
    def _attn_tc_eligible(HW, Cc):
        """Mirrors prepare_attn_tc: attn_tc holds all keys of a query tile (64, 128, 256 tokens),
        attn_stream_tc streams them (multiples of 128 from 512); C > 256 would not fit TMEM."""
        return Cc % 64 == 0 and 64 <= Cc <= 256 and (HW in (64, 128, 256) or (HW % 128 == 0 and HW >= 512))

    def op_attn(self, qkv, HW, Cc, proj=None):
        """proj = (W3 [out, in], bias, x, scale, out): the output projection + skip connection are
        fused into the tensor-core attention kernel; returns None if that is not possible."""
        op = self._op(L.OP_ATTN)
        op.i[L.ATTN_N], op.i[L.ATTN_HW], op.i[L.ATTN_C], op.i[L.ATTN_DTYPE] = self.B, HW, Cc, self.acode
        op.f[0] = float(int(Cc) ** (-0.5))
        op.inp[0] = qkv.data_ptr()
        tc_ok = self._attn_tc_eligible(HW, Cc)
        fusable = tc_ok and HW % 128 == 0
        if proj is not None:
            if not (self.tc and fusable):
                return None
            w3, b3, x, scale, o = proj
            op.i[L.ATTN_PROJ] = 1
            op.f[1] = float(scale)
            op.inp[1] = self._w_bf16(w3.detach().to(self.dev, torch.float32)).data_ptr()
            op.inp[2] = self._w(b3).data_ptr() if b3 is not None else None
            op.inp[3] = x.data_ptr()
            mg = None
            if Cc % 32 == 0:
                mg = self._mg_buffer(self.B, Cc)
                op.out[1] = mg.data_ptr()
        else:
            o = self._acquire(*qkv.shape[:-1], Cc)
        op.out[0] = o.data_ptr()
        if self.tc:
            op.engine = L.ENGINE_TC
            if self.dry:
                rc = L.OK if tc_ok else L.EUNSUPPORTED
            else:
                rc = self.lib.psld_op_prepare(C.byref(op))
            if rc == L.EUNSUPPORTED:
                if proj is not None:
                    raise RuntimeError("psld_b200: fused attention projection rejected: " +
                                       self.lib.psld_last_error().decode(errors="replace"))
                op.engine = L.ENGINE_SIMT
            elif rc != L.OK:
                L.check(rc, "psld_op_prepare(attn)")
        if proj is not None and op.out[1]:
            self.mg[o.data_ptr()] = mg
        key = ("attn_tc_proj" if proj is not None else "attn_tc") if op.engine == L.ENGINE_TC else "attn_simt"
        self.engine_count[key] = self.engine_count.get(key, 0) + 1
        if proj is not None:
            self.engine_count["attn_tc"] = self.engine_count.get("attn_tc", 0) + 1
        self._push(op)
        return o

    # ---------------------------------------------------------------- blocks
    def _resample(self, up):
        """(taps, up, down, pad0, pad1) of the network's x2 up- or downsampler as an upfirdn2d."""
        if self.net.fir:
            if up:      # upsample_2d: upfirdn2d(up=2, pad=(2,1)), taps * factor^2 (:195-224)
                return _fir_taps(self.net.fir_kernel, 4.0), 2, 1, 2, 1
            # downsample_2d: upfirdn2d(down=2, pad=(1,1)) (:227-257)
            return _fir_taps(self.net.fir_kernel, 1.0), 1, 2, 1, 1
        if up:          # naive_upsample_2d: nearest x2
            return np.ones((2, 2), np.float32), 2, 1, 1, 0
        # naive_downsample_2d: 2x2 mean
        return np.full((2, 2), 0.25, np.float32), 1, 2, 0, 0

    def resblock(self, m, x1, x2, temb_off):
        """ResnetBlockBigGANpp.forward (reference layerspp.py:242-274)."""
        net = self.net
        N, H, W, _ = x1.shape
        scale = _SQRT1_2 if net.skip_rescale else 1.0
        if not (m.up or m.down) and self._gn_fusable(x1, x2, m.out_ch):
            # act(GroupNorm_0(.)) -> Conv_0 runs as ONE GroupNorm-on-load convolution: the
            # GroupNorm op only emits a per-(sample, channel) affine, there is no apply pass.  The
            # same for act(GroupNorm_1(.)) -> Conv_1 of the identity-shortcut blocks (residual add
            # in the epilogue).
            aff0 = self.op_gn(x1, x2, m.GroupNorm_0, True, H * W, affine_only=True)
            h = self.op_conv(x1, x2, m.Conv_0.weight, None, ks=3, temb_off=temb_off, affine=aff0)
            self._release_affine(aff0)
            return self._block_tail(m, h, x1, x2, scale)
        a = self.op_gn(x1, x2, m.GroupNorm_0, True, H * W)
        xs1, xs2 = x1, x2
        fir_tmp = []
        if m.up or m.down:
            assert x2 is None
            rs = self._resample(m.up)
            a2 = self.op_fir(a, *rs)
            self._release(a)
            a = a2
            xs1 = self.op_fir(x1, *rs)
            fir_tmp.append(xs1)
        h = self.op_conv(a, None, m.Conv_0.weight, None, ks=3, temb_off=temb_off)  # bias: see temb
        self._release(a)
        out = self._block_tail(m, h, xs1, xs2, scale)
        for t in fir_tmp:
            self._release(t)
        return out

    def _block_tail(self, m, h, x1, x2, scale):
        """act(GroupNorm_1(h)) -> Conv_1 (+ Conv_2 shortcut over cat(x1, x2) or identity skip) -> * scale
        (layerspp.py:264-274).  ``h`` is consumed."""
        N, H, W, _ = h.shape
        has_sc = hasattr(m, "Conv_2")
        # GroupNorm_1 is applied on load inside Conv_1 of identity-shortcut blocks.  Blocks with a
        # Conv_2 shortcut: bf16 keeps the unfused Conv_1 (apply pass + conv_tc with the shortcut as
        # K-extension): the fused kernel accepts the extension too, but its two big operand buffers
        # cannot hide the load latency of one-tap chunks (measured +1.1 ms of conv for -0.64 ms of
        # GroupNorm per step).  bf16x3: the fused kernel streams the shortcut tiles through a
        # 3-slot ring of their own, so the extension costs what it costs in conv_tc and the apply
        # pass goes away.
        gn1 = not has_sc or (self.x3 and self._ext_fusable(h, x1, x2, m.out_ch))
        if gn1 and self._gn_fusable(h, None, m.out_ch):
            aff1 = self.op_gn(h, None, m.GroupNorm_1, True, H * W, affine_only=True)
            b, b_aff = h, aff1
        else:
            b = self.op_gn(h, None, m.GroupNorm_1, True, H * W)
            self._release(h)
            b_aff = None
        ext, sc = None, None
        if has_sc:
            if self._ext_fusable(b, x1, x2, m.out_ch):
                ext = (x1, x2, m.Conv_2.weight, m.Conv_2.bias)
            else:
                sc = self.op_conv(x1, x2, m.Conv_2.weight, m.Conv_2.bias, ks=1, want_stats=False)
        else:
            assert x2 is None
            sc = x1
        out = self.op_conv(b, None, m.Conv_1.weight, m.Conv_1.bias, ks=3, residual=sc, scale=scale,
                           out=self._new(N, H, W, m.out_ch), affine=b_aff, ext=ext)
        if b_aff is not None:
            self._release_affine(b_aff)
        self._release(b)
        if has_sc and sc is not None:
            self._release(sc)
        return out

    def attnblock(self, m, x):
        """AttnBlockpp.forward (reference layerspp.py:75-91)."""
        N, H, W, Cc = x.shape
        a = self.op_gn(x, None, m.GroupNorm_0, False, H * W)
        wqkv = torch.cat([m.NIN_0.W, m.NIN_1.W, m.NIN_2.W], dim=1)          # [C, 3C]
        bqkv = torch.cat([m.NIN_0.b, m.NIN_1.b, m.NIN_2.b], dim=0)
        qkv = self.op_conv(a, None, wqkv.t().reshape(3 * Cc, Cc, 1, 1), bqkv, ks=1, want_stats=False)
        self._release(a)
        scale = _SQRT1_2 if self.net.skip_rescale else 1.0
        # h = (NIN_3(attention) + x) * scale inside the attention kernel where it is eligible
        out = self.op_attn(qkv, H * W, Cc, proj=(m.NIN_3.W.t().contiguous(), m.NIN_3.b, x, scale,
                                                 self._new(N, H, W, Cc)))
        if out is not None:
            self._release(qkv)
            return out
        o = self.op_attn(qkv, H * W, Cc)
        self._release(qkv)
        out = self.op_conv(o, None, m.NIN_3.W.t().reshape(Cc, Cc, 1, 1), m.NIN_3.b, ks=1,
                           residual=x, scale=scale, out=self._new(N, H, W, Cc))
        self._release(o)
        return out

    # ---------------------------------------------------------------- whole network
    def _build(self):
        net, B = self.net, self.B
        mods = net.all_modules
        H = net.image_size
        self.gn_scratch = None
        self.x_in = self._new(B, net.in_ch, H, H, dtype=torch.float32)        # NCHW fp32 input
        self.time_buf = self._new(self.nt, dtype=torch.float32)
        # the GroupNorm statistics accumulators are cleared first (pointers / sizes filled in at the end)
        zero_ops = [self._push(self._op(L.OP_ZERO)) for _ in range(self._STAT_SLOTS)]
        i = 0
        # ---- time embedding + every Dense_0 projection in one op
        if not net.noise_cond:
            raise NotImplementedError("psld_b200 NCSNpp: noise_cond=False is not supported")
        fourier_w = None
        if net.embedding_type == "fourier":
            fourier_w = self._w(mods[i].W); i += 1
        lin0, lin1 = mods[i], mods[i + 1]; i += 2
        rbs = [m for m in mods if hasattr(m, "Dense_0")]
        offs, tot = {}, 0
        for m in rbs:
            offs[id(m)] = tot
            tot += m.out_ch
        self.total_c = tot
        wd = self._w(torch.cat([m.Dense_0.weight for m in rbs], 0))
        # Conv_0's bias is folded into the Dense_0 bias: both are per-(n, channel) terms added
        # to the same accumulator (layerspp.py:260-263), so the conv epilogue adds ONE vector
        bd = self._w(torch.cat([m.Dense_0.bias + m.Conv_0.bias for m in rbs], 0))
        E = 2 * net.nf if net.embedding_type == "fourier" else net.nf
        self.temb_proj = self._new(self.nt, tot, dtype=torch.float32)
        scratch = self._new(self.nt, E + 8 * net.nf, dtype=torch.float32)
        op = self._op(L.OP_TEMB)
        op.i[L.TEMB_NT], op.i[L.TEMB_NF] = self.nt, net.nf
        op.i[L.TEMB_EMB] = 0 if net.embedding_type == "fourier" else 1
        op.i[L.TEMB_TOTALC], op.i[L.TEMB_LOGGED] = tot, int(self.logged)
        op.inp[0] = self.time_buf.data_ptr()
        op.inp[1] = fourier_w.data_ptr() if fourier_w is not None else None
        op.inp[2], op.inp[3] = self._w(lin0.weight).data_ptr(), self._w(lin0.bias).data_ptr()
        op.inp[4], op.inp[5] = self._w(lin1.weight).data_ptr(), self._w(lin1.bias).data_ptr()
        op.inp[6], op.inp[7] = wd.data_ptr(), bd.data_ptr()
        op.out[0], op.out[1] = self.temb_proj.data_ptr(), scratch.data_ptr()
        self.temb_op = self._push(op)

        # ---- input: NCHW fp32 -> NHWC activations
        # bf16 plans zero-pad the 6 input channels to 64 so that the input conv and the first
        # pyramid conv are tensor-core eligible (K chunks are 64 channels)
        cpad = 64 if (self.tc and net.in_ch < 64) else net.in_ch
        if cpad > net.in_ch:     # padding channels: zeroed once here, never written again
            x = torch.zeros(B, H, H, cpad, dtype=self.adt, device=self.dev)
            self.keep.append(x)
            cwrite = min(cpad, -(-net.in_ch // 8) * 8)
        else:
            x, cwrite = self._new(B, H, H, cpad), 0
        self.op_layout(self.x_in, x, B, net.in_ch, H * H, 0, cpad, cwrite)
        pyr = x if net.progressive_input != "none" else None
        hs = [self.op_conv(x, None, mods[i].weight, mods[i].bias, ks=3,
                           out=self._new(B, H, H, net.nf))]; i += 1
        for lvl in range(net.num_resolutions):
            for _ in range(net.num_res_blocks):
                m = mods[i]; i += 1
                h = self.resblock(m, hs[-1], None, offs[id(m)])
                if h.shape[2] in net.attn_resolutions:
                    h = self.attnblock(mods[i], h); i += 1
                hs.append(h)
            if lvl != net.num_resolutions - 1:
                m = mods[i]; i += 1
                h = self.resblock(m, hs[-1], None, offs[id(m)])
                if net.progressive_input == "input_skip":
                    # Combine(sum): the pyramid keeps the input's channels, downsampled once per level;
                    # h + Conv_0(pyr) is the 1x1 conv with h as its epilogue residual
                    cact = 8 if (cpad > net.in_ch and net.in_ch <= 8) else 0
                    pyr = self.op_fir(pyr, *self._resample(False), cact=cact)
                    cm = mods[i]; i += 1
                    h = self.op_conv(pyr, None, cm.Conv_0.weight, cm.Conv_0.bias, ks=1, residual=h,
                                     out=self._new(*h.shape))
                elif net.progressive_input == "residual":
                    pm = mods[i]; i += 1
                    # conv_downsample_2d: upfirdn2d(pad=(2,2)) then conv(stride 2, pad 0) + bias,
                    # merged with h: (pyr + h)/sqrt(2)   (ncsnpp.py:350-357)
                    cact = 8 if (pyr is x and cpad > net.in_ch and net.in_ch <= 8) else 0
                    padded = self.op_fir(pyr, _fir_taps(net.fir_kernel, 1.0), 1, 1, 2, 2, cact=cact)
                    scale = _SQRT1_2 if net.skip_rescale else 1.0
                    pyr = self.op_conv(padded, None, pm.Conv2d_0.weight, pm.Conv2d_0.bias, ks=3,
                                       stride=2, pad=0, residual=h, scale=scale,
                                       out=self._new(*h.shape))
                    if not cact:                    # (the zero-padded buffer is never pooled)
                        self._release(padded)
                    h = pyr
                hs.append(h)
        h = hs[-1]
        m = mods[i]; i += 1
        h = self.resblock(m, h, None, offs[id(m)])
        h = self.attnblock(mods[i], h); i += 1
        m = mods[i]; i += 1
        h = self.resblock(m, h, None, offs[id(m)])
        out_pyr = None
        for lvl in reversed(range(net.num_resolutions)):
            for _ in range(net.num_res_blocks + 1):
                m = mods[i]; i += 1
                h = self.resblock(m, h, hs.pop(), offs[id(m)])     # cat([h, skip]) is virtual
            if h.shape[2] in net.attn_resolutions:
                h = self.attnblock(mods[i], h); i += 1
            if net.progressive == "output_skip":
                out_pyr = self.head(h, mods[i], mods[i + 1], out_pyr); i += 2
            if lvl != 0:
                m = mods[i]; i += 1
                h = self.resblock(m, h, None, offs[id(m)])
        assert not hs
        if net.progressive == "output_skip":
            self.eps = out_pyr
        else:
            self.eps = self.head(h, mods[i], mods[i + 1], None); i += 2
        assert i == len(mods), (i, len(mods))
        self._finish_stat_arenas(zero_ops)

    def head(self, h, gn, conv, pyr):
        """conv3x3(act(GroupNorm(h))) -> fp32 NCHW [B, out_ch, H, W], plus the x2-upsampled output
        pyramid ``pyr`` of the level below when given (progressive=output_skip, ncsnpp.py:405-418).
        The pyramid is upsampled as B*out_ch single-channel planes and added in the conv epilogue."""
        HW = h.shape[1] * h.shape[2]
        res = None
        if pyr is not None:
            B, Cc, H, W = pyr.shape
            res = self.op_fir(pyr.view(B * Cc, H, W, 1), *self._resample(True), f32=True)
            res = res.view(B, Cc, 2 * H, 2 * W)
        if self._gn_fusable(h, None, 64):
            # act(GroupNorm(h)) -> conv3x3 -> fp32 NCHW as one GroupNorm-on-load conv
            aff = self.op_gn(h, None, gn, True, HW, affine_only=True)
            out = self.op_conv(h, None, conv.weight, conv.bias, ks=3, out_nchw_f32=True, affine=aff,
                               residual=res)
            self._release_affine(aff)
        else:
            a = self.op_gn(h, None, gn, True, HW)
            out = self.op_conv(a, None, conv.weight, conv.bias, ks=3, out_nchw_f32=True, residual=res)
            self._release(a)
        return out

    # ---------------------------------------------------------------- execution
    def run(self, stream=None):
        if self.dry:
            raise RuntimeError("dry plan cannot run")
        s = stream if stream is not None else L.stream_ptr(self.dev)
        L.check(self.lib.psld_program_run(self.op_array, self.n_ops, s), "psld_program_run")

    def release(self):
        arr = self.__dict__.get("op_array")
        if arr is not None:
            for k in range(self.n_ops):
                if arr[k].aux:
                    self.lib.psld_op_release(C.byref(arr[k]))
        self.__dict__["op_array"] = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


def build_plan(net, B, nt, logged, dry=False):
    with torch.no_grad():
        return Plan(net, B, nt, logged, dry=dry)
