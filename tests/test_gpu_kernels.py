"""GPU parity tests of every kernel through the C ABI, against the CPU oracle.

Tolerances (stated, per kernel):
  fused phase-space update, fp64 state ... max-abs/max|ref| <= 1e-13 (same algebra in double)
  fused phase-space update, fp32 state ... <= 2e-6 relative (fp32 rounding of the state)
  GroupNorm / FIR / temb / conv fp32 ...... rel-L2 <= 2e-6 (fp32 summation order)
  bf16 storage paths ...................... rel-L2 <= 6e-3 (8-bit mantissa)
"""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from _ops import attn_op, conv_op, conv_ref, fir_op, gn_op, max_rel, mg_ref, rel_l2, run_op
from oracle import psld_oracle as O
from oracle.weights import noise_bank, prior
from psld_b200 import _lib as L
from psld_b200 import tiny_config
from psld_b200.schedule import PSLDSchedule, StepTables

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _rng(seed):
    return np.random.default_rng(seed)


def _t(a, dtype=torch.float32):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV, dtype)


# ------------------------------------------------------------------ fused phase-space update
def _half_ref(h, u, z):
    x, m = torch.chunk(u, 2, 1)
    zx, zm = torch.chunk(z.double(), 2, 1)
    return torch.cat([h.a_xx * x + h.a_xm * m + (h.c11 * zx + h.c12 * zm),
                      h.a_mx * x + h.a_mm * m + (h.c21 * zx + h.c22 * zm)], 1)


def _score_ref(sc, u, eps):
    """Oracle algebra of the SCORE stage from the table entry (psld.py:252-259, sde.py:325-328)."""
    x, m = torch.chunk(u, 2, 1)
    f32 = lambda v: torch.tensor(v, dtype=torch.float32)
    if sc.mode == 0:
        ex, em = torch.chunk(eps, 2, 1)
        sx = -f32(sc.li11) * ex - f32(sc.li12) * em
        sm = -f32(sc.li21) * ex - f32(sc.li22) * em
    elif sc.mode == 1:
        sx, sm = torch.zeros_like(eps), -f32(sc.li22) * eps
    else:
        sx, sm = -f32(sc.li11) * eps, torch.zeros_like(eps)
    x = x + sc.k_x * (sx.double() + x)
    m = m + sc.k_m * (sm.double() + sc.m_inv * m)
    return torch.cat([x, m], 1)


@pytest.mark.parametrize("state_dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("gamma", [0.01, 0.0])
def test_sscs_update_stages(state_dtype, gamma):
    cfg = tiny_config(sampler="sscs_sde", n_discrete_steps=10)
    cfg.model.sde.gamma = gamma
    cfg.model.sde.nu = 4.01 if gamma else 4.0
    sch = PSLDSchedule(cfg)
    ts = torch.linspace(0, 0.999, 10, dtype=torch.float64)
    tabs = StepTables(sch, ts, 9, "sscs_sde", True, 1e-3)
    B, Cc, H = 3, 3, 8
    chw = Cc * H * H
    u0 = prior((B, Cc, H, H), 0.5, 3).double()
    zs = noise_bank(3, (B, 2 * Cc, H, H), 4)
    r = _rng(5)
    e_ch = 2 * Cc if gamma else Cc
    eps = torch.from_numpy(r.standard_normal((B, e_ch, H, H)).astype(np.float32))
    co = tabs.sscs[4]
    lib = L.lib()
    for stages in [1, 2, 4, 6, 14, 15]:
        ref = u0.clone()
        if stages & 1:
            ref = _half_ref(co.half_a, ref, zs[0])
        if stages & 2:
            ref = _score_ref(co.score, ref, eps)
        if stages & 4:
            ref = _half_ref(co.half_b, ref, zs[1])
        if stages & 8:
            ref = _half_ref(co.half_c, ref, zs[2])
        u = u0.to(DEV, state_dtype).contiguous()
        out = torch.empty_like(u)
        net_in = torch.empty(B, 2 * Cc, H, H, dtype=torch.float32, device=DEV)
        zd = [z.to(DEV) for z in zs]
        ed = eps.to(DEV)
        L.check(lib.psld_sscs_update(L.ptr(out), L.ptr(u), L.dtype_code(state_dtype), L.ptr(net_in),
                                     L.ptr(ed), L.ptr(zd[0]), L.ptr(zd[1]), L.ptr(zd[2]),
                                     C.byref(co), stages, 0, 0, B, chw, L.stream_ptr()), "sscs")
        torch.cuda.synchronize()
        tol = 1e-13 if state_dtype == torch.float64 else 2e-6
        assert max_rel(out, ref) <= tol, (stages, max_rel(out, ref))
        assert torch.equal(net_in.cpu(), out.cpu().to(torch.float32))


@pytest.mark.parametrize("state_dtype", [torch.float64, torch.float32])
def test_em_update(state_dtype):
    cfg = tiny_config(sampler="em_sde", n_discrete_steps=10)
    sch = PSLDSchedule(cfg)
    ts = torch.linspace(0, 0.999, 10, dtype=torch.float64)
    tabs = StepTables(sch, ts, 9, "em_sde", True, 1e-3)
    B, Cc, H = 2, 3, 8
    u0 = prior((B, Cc, H, H), 0.5, 3).double()
    z = noise_bank(1, (B, 2 * Cc, H, H), 4)[0]
    eps = torch.from_numpy(_rng(5).standard_normal((B, 2 * Cc, H, H)).astype(np.float32))
    lib = L.lib()
    for co, zz in [(tabs.em[3], z), (tabs.den, None)]:
        x, m = torch.chunk(u0, 2, 1)
        f32 = lambda v: torch.tensor(v, dtype=torch.float32)
        ex, em = torch.chunk(eps, 2, 1)
        sx = (-f32(co.li11) * ex - f32(co.li12) * em).double()
        sm = (-f32(co.li21) * ex - f32(co.li22) * em).double()
        fx = co.half_beta * (co.m_inv * m - co.gamma * x)
        fm = co.half_beta * (-co.nu * m - x)
        nx = x + (-fx + co.g2_x * sx) * co.dt
        nm = m + (-fm + co.g2_m * sm) * co.dt
        if zz is not None:
            zx, zm = torch.chunk(zz.double(), 2, 1)
            nx, nm = nx + co.gs_x * zx, nm + co.gs_m * zm
        ref = torch.cat([nx, nm], 1)
        u = u0.to(DEV, state_dtype).contiguous()
        out = torch.empty_like(u)
        ed = eps.to(DEV)
        zd = zz.to(DEV) if zz is not None else None      # keep the device tensors alive
        L.check(lib.psld_em_update(L.ptr(out), L.ptr(u), L.dtype_code(state_dtype), None,
                                   L.ptr(ed), L.ptr(zd), 0, C.byref(co), 0, 0, B, Cc * H * H,
                                   L.stream_ptr()), "em")
        torch.cuda.synchronize()
        tol = 1e-13 if state_dtype == torch.float64 else 2e-6
        assert max_rel(out, ref) <= tol, max_rel(out, ref)


def test_philox_noise_and_prior():
    lib = L.lib()
    B, chw = 64, 3072
    u = torch.empty(B, 6, 32, 32, dtype=torch.float32, device=DEV)
    L.check(lib.psld_prior_sample(L.ptr(u), 0.5, 123, B, chw, L.stream_ptr()), "prior")
    x, m = torch.chunk(u.double().cpu(), 2, 1)
    n = x.numel()
    assert abs(x.mean()) < 5 / np.sqrt(n) and abs(x.var() - 1) < 0.02
    assert abs(m.mean()) < 5 * 0.5 / np.sqrt(n) and abs(m.var() - 0.25) < 0.005
    assert abs(float((x * m).mean())) < 5 * 0.5 / np.sqrt(n)
    # different seeds decorrelate, same seed reproduces
    u2 = torch.empty_like(u)
    L.check(lib.psld_prior_sample(L.ptr(u2), 0.5, 123, B, chw, L.stream_ptr()), "prior")
    assert torch.equal(u, u2)
    L.check(lib.psld_prior_sample(L.ptr(u2), 0.5, 124, B, chw, L.stream_ptr()), "prior")
    assert abs(float((u * u2).mean())) < 0.01
    # a pure-noise half step with Philox has the requested 2x2 covariance
    co = L.SscsCoeffs()
    co.half_a.c11, co.half_a.c21, co.half_a.c22 = 0.7, -0.3, 0.4
    z = torch.zeros(B, 6, 32, 32, dtype=torch.float64, device=DEV)
    out = torch.empty_like(z)
    L.check(lib.psld_sscs_update(L.ptr(out), L.ptr(z), L.F64, None, None, None, None, None,
                                 C.byref(co), 1, 7, 3, B, chw, L.stream_ptr()), "sscs")
    ox, om = torch.chunk(out.cpu(), 2, 1)
    assert abs(ox.var() - 0.49) < 0.01 and abs(om.var() - (0.09 + 0.16)) < 0.01
    assert abs(float((ox * om).mean()) - (-0.21)) < 0.01


def test_philox_normal_quality():
    """The in-kernel generator (Philox4x32-10 + Box-Muller) that produces every noise sample of a
    throughput run, on 2.5e7 draws per stream: Kolmogorov-Smirnov distance against N(0,1), moments
    up to the 6th, tail mass beyond 3/4/5 sigma, and independence between step streams, between
    the x and m halves, between neighbouring elements and between seeds."""
    from math import erfc, sqrt
    lib = L.lib()
    B, chw = 4096, 3072
    n = B * chw * 2                                     # 2.5e7 normals per launch
    co = L.SscsCoeffs()
    co.half_a.c11, co.half_a.c22 = 1.0, 1.0             # u = z: a pure-noise half step
    z0 = torch.zeros(B, 6, 32, 32, dtype=torch.float32, device=DEV)

    def draw(seed, step):
        out = torch.empty_like(z0)
        L.check(lib.psld_sscs_update(L.ptr(out), L.ptr(z0), L.F32, None, None, None, None, None,
                                     C.byref(co), 1, seed, step, B, chw, L.stream_ptr()), "sscs")
        return out

    a = draw(2024, 0)
    v = a.double().flatten()
    # moments: E z^k = 0, 1, 0, 3, 0, 15 with standard errors sqrt(Var(z^k) / n)
    se = {1: 1.0, 2: sqrt(2.0), 3: sqrt(15.0), 4: sqrt(96.0), 5: sqrt(945.0), 6: sqrt(10170.0)}
    want = {1: 0.0, 2: 1.0, 3: 0.0, 4: 3.0, 5: 0.0, 6: 15.0}
    for k in range(1, 7):
        mk = float((v ** k).mean())
        assert abs(mk - want[k]) <= 5.0 * se[k] / sqrt(n), (k, mk)
    # KS distance on a 4e6 subsample (stride keeps every stream position): D_crit(1e-3) = 1.95/sqrt(m)
    sub = v[::6].sort().values.cpu()
    m = sub.numel()
    cdf = 0.5 * (1.0 + torch.erf(sub / sqrt(2.0)))
    i = torch.arange(1, m + 1, dtype=torch.float64)
    D = float(torch.max(torch.max(i / m - cdf), torch.max(cdf - (i - 1) / m)))
    assert D <= 1.95 / sqrt(m), D
    # tails: two-sided mass beyond k sigma, binomial 5-sigma band
    for k in (3.0, 4.0, 5.0):
        p = erfc(k / sqrt(2.0))
        cnt = float((v.abs() > k).sum())
        assert abs(cnt - n * p) <= 5.0 * sqrt(n * p) + 1.0, (k, cnt, n * p)
    assert float(v.abs().max()) < 6.8
    # independence: correlation of two standard normals over n pairs has std 1/sqrt(n)
    lim = 5.0 / sqrt(n)
    b = draw(2024, 1).double().flatten()                 # next step's stream
    c = draw(2025, 0).double().flatten()                 # another seed
    assert abs(float((v * b).mean())) <= lim and abs(float((v * c).mean())) <= lim
    x, mm = torch.chunk(a.double(), 2, 1)
    assert abs(float((x * mm).mean())) <= lim * sqrt(2.0)
    assert abs(float((v[1:] * v[:-1]).mean())) <= lim    # neighbours (same Philox counter block)
    assert abs(float((v[4:] * v[:-4]).mean())) <= lim


# ------------------------------------------------------------------ GroupNorm
@pytest.mark.parametrize("dtype,tol", [(torch.float32, 2e-6), (torch.bfloat16, 6e-3)])
@pytest.mark.parametrize("shape", [(2, 16, 16, 64, 0), (3, 8, 8, 256, 128), (2, 32, 32, 32, 64),
                                   (1, 4, 4, 24, 0)])
@pytest.mark.parametrize("silu", [True, False])
def test_groupnorm(dtype, tol, shape, silu):
    N, H, W, C1, C2 = shape
    r = _rng(11)
    Cc = C1 + C2
    G = min(Cc // 4, 32)
    x1 = _t(r.standard_normal((N, H, W, C1)) * 2 + 0.7, dtype)
    x2 = _t(r.standard_normal((N, H, W, C2)) * 0.5 - 1.0, dtype) if C2 else None
    ga = _t(1 + 0.2 * r.standard_normal(Cc))
    be = _t(0.1 * r.standard_normal(Cc))
    op, out, keep = gn_op(x1, x2, ga, be, G, silu, nchunk=3)
    run_op(op)
    xx = x1.float().cpu() if x2 is None else torch.cat([x1.float().cpu(), x2.float().cpu()], -1)
    ref = F.group_norm(xx.permute(0, 3, 1, 2), G, ga.cpu(), be.cpu(), eps=1e-6)
    if silu:
        ref = F.silu(ref)
    assert rel_l2(out.float().permute(0, 3, 1, 2), ref) <= tol


# ------------------------------------------------------------------ FIR / upfirdn2d
def test_upfirdn2d_golden(golden_dir):
    g = np.load(f"{golden_dir}/upfirdn.npz")
    x = torch.from_numpy(g["x"]).to(DEV)
    lib = L.lib()
    for name in ["down", "up", "pad", "generic", "crop"]:
        up, down, p0, p1, gain = g["arg_" + name]
        k = (g["k"] * gain).astype(np.float32)
        y = torch.from_numpy(g["y_" + name])
        out = torch.full(tuple(y.shape), float("nan"), dtype=torch.float32, device=DEV)
        taps = (C.c_float * 16)(*k.reshape(-1))
        L.check(lib.psld_upfirdn2d(L.ptr(x), L.ptr(out), taps, 4, 4, x.shape[0] * x.shape[1],
                                   x.shape[2], x.shape[3], int(up), int(up), int(down), int(down),
                                   int(p0), int(p1), int(p0), int(p1), L.stream_ptr()), "upfirdn2d")
        torch.cuda.synchronize()
        assert rel_l2(out, y) <= 2e-6, (name, rel_l2(out, y))
        # NHWC op, fp32 and bf16, vectorised (C%4==0) and scalar channel counts
        for Cc in (5, 8):
            xn = torch.from_numpy(_rng(3).standard_normal((2, 8, 8, Cc)).astype(np.float32)).to(DEV)
            ref = O.upfirdn2d(xn.cpu().permute(0, 3, 1, 2), k, up=int(up), down=int(down),
                              pad=(int(p0), int(p1)))
            for dt, tol in [(torch.float32, 2e-6), (torch.bfloat16, 6e-3)]:
                op, o = fir_op(xn.to(dt), k, int(up), int(down), int(p0), int(p1))
                run_op(op)
                refd = O.upfirdn2d(xn.to(dt).float().cpu().permute(0, 3, 1, 2), k, up=int(up),
                                   down=int(down), pad=(int(p0), int(p1)))
                assert rel_l2(o.float().permute(0, 3, 1, 2), refd) <= tol, (name, Cc, dt)


def test_fir_up2_polyphase_and_channel_subset():
    """upsample_2d through the polyphase kernel (one thread per input pixel -> 2x2 output quad) on a
    ragged map, and the active-channel subset used for the zero-padded network input."""
    k = np.outer([1, 3, 3, 1], [1, 3, 3, 1]).astype(np.float32)
    k = k / k.sum()
    r = _rng(21)
    x = torch.from_numpy(r.standard_normal((3, 5, 7, 16)).astype(np.float32)).to(DEV)
    for dt, tol in [(torch.float32, 2e-6), (torch.bfloat16, 6e-3)]:
        op, o = fir_op(x.to(dt), k * 4, 2, 1, 2, 1)
        run_op(op)
        ref = O.upfirdn2d(x.to(dt).float().cpu().permute(0, 3, 1, 2), k * 4, up=2, down=1, pad=(2, 1))
        assert o.shape == (3, 10, 14, 16)
        assert rel_l2(o.float().permute(0, 3, 1, 2), ref) <= tol, dt
    # downsample_2d through the quad kernel (H, W multiples of 4) and the generic one (ragged)
    for shape in [(3, 8, 12, 16), (2, 6, 10, 8)]:
        xd = torch.from_numpy(r.standard_normal(shape).astype(np.float32)).to(DEV)
        for dt, tol in [(torch.float32, 2e-6), (torch.bfloat16, 6e-3)]:
            op, o = fir_op(xd.to(dt), k, 1, 2, 1, 1)
            run_op(op)
            ref = O.upfirdn2d(xd.to(dt).float().cpu().permute(0, 3, 1, 2), k, up=1, down=2, pad=(1, 1))
            assert rel_l2(o.float().permute(0, 3, 1, 2), ref) <= tol, (shape, dt)
    # channel subset: only [0, 8) filtered and written, the rest of the output untouched
    xp = torch.zeros(2, 8, 8, 64, dtype=torch.bfloat16, device=DEV)
    xp[..., :6] = torch.from_numpy(r.standard_normal((2, 8, 8, 6)).astype(np.float32)).to(DEV)
    op, o = fir_op(xp, k, 1, 1, 2, 2)
    o.zero_()
    op.i[L.FIR_CACT] = 8
    run_op(op)
    ref = O.upfirdn2d(xp.float().cpu().permute(0, 3, 1, 2), k, up=1, down=1, pad=(2, 2))
    assert rel_l2(o.float().permute(0, 3, 1, 2), ref) <= 6e-3
    assert float(o[..., 8:].abs().max()) == 0.0


# ------------------------------------------------------------------ convolution, CUDA-core engine
CONV_SIMT_CASES = [
    # N, H, W, C1, C2, Cout, ks, stride, pad
    (2, 8, 8, 6, 0, 32, 3, 1, 1),       # input conv
    (2, 8, 8, 32, 0, 6, 3, 1, 1),       # output conv
    (2, 9, 9, 6, 0, 32, 3, 2, 0),       # pyramid stride-2 conv after FIR pad
    (1, 16, 16, 64, 32, 64, 1, 1, 0),   # 1x1 shortcut over a virtual concat
    (3, 8, 8, 96, 0, 64, 3, 1, 1),
    (1, 5, 7, 20, 12, 10, 3, 1, 1),     # ragged everything
]


@pytest.mark.parametrize("case", CONV_SIMT_CASES)
@pytest.mark.parametrize("dtype,tol", [(torch.float32, 3e-6), (torch.bfloat16, 6e-3)])
def test_conv_simt(case, dtype, tol):
    N, H, W, C1, C2, Cout, ks, stride, pad = case
    r = _rng(sum(case))
    x1 = _t(r.standard_normal((N, H, W, C1)), dtype)
    x2 = _t(r.standard_normal((N, H, W, C2)), dtype) if C2 else None
    w = _t(r.standard_normal((Cout, C1 + C2, ks, ks)) / np.sqrt((C1 + C2) * ks * ks))
    b = _t(0.1 * r.standard_normal(Cout))
    OH = (H + 2 * pad - ks) // stride + 1
    OW = (W + 2 * pad - ks) // stride + 1
    res = _t(r.standard_normal((N, OH, OW, Cout)), dtype)
    temb = _t(r.standard_normal((N, Cout + 5)))
    kw = dict(stride=stride, pad=pad, residual=res, temb=temb, temb_off=5, temb_bstride=Cout + 5,
              scale=0.7071)
    op, out, keep = conv_op(x1, x2, w, b, **kw)
    run_op(op)
    wq = w if dtype == torch.float32 else w
    ref = conv_ref(x1, x2, wq, b, **kw)
    assert rel_l2(out.float().permute(0, 3, 1, 2), ref) <= tol
    # NCHW fp32 head, shared temb row
    op, out, keep = conv_op(x1, x2, w, b, stride=stride, pad=pad, temb=temb[:1].contiguous(),
                            temb_off=2, temb_bstride=0, out_nchw_f32=True)
    run_op(op)
    ref = conv_ref(x1, x2, w, b, stride=stride, pad=pad, temb=temb[:1], temb_off=2, temb_bstride=0)
    assert rel_l2(out, ref) <= (3e-6 if dtype == torch.float32 else 1e-5)


# ------------------------------------------------------------------ convolution, tcgen05 engine
CONV_TC_CASES = [
    # N, H, W, C1, C2, Cout, ks
    (2, 32, 32, 64, 0, 64, 1),
    (2, 32, 32, 64, 0, 128, 3),
    (1, 16, 16, 128, 0, 256, 3),
    (3, 8, 8, 128, 64, 128, 1),        # two-source 1x1 shortcut, BN_img = 2 with an odd batch
    (3, 8, 8, 256, 0, 256, 3),
    (2, 16, 16, 256, 0, 768, 1),       # fused q|k|v projection, 3 N-tiles
    (5, 4, 4, 64, 0, 96, 3),           # 4x4 maps, 8 images per tile, Cout = 3 x 32
    (1, 64, 64, 64, 0, 32, 3),         # CelebA-size map
    (2, 32, 32, 256, 256, 256, 1),
    (41, 32, 32, 128, 0, 256, 3),      # 164 tile pairs over 74 clusters: persistent multi-wave loop, both accumulators
    (37, 16, 16, 256, 128, 256, 3),    # odd tile count (partial last pair), two sources, 3 waves
]


@pytest.mark.parametrize("case", CONV_TC_CASES)
def test_conv_tc(case):
    N, H, W, C1, C2, Cout, ks = case
    r = _rng(sum(case) + 1)
    x1 = _t(r.standard_normal((N, H, W, C1)), torch.bfloat16)
    x2 = _t(r.standard_normal((N, H, W, C2)), torch.bfloat16) if C2 else None
    w = _t(r.standard_normal((Cout, C1 + C2, ks, ks)) / np.sqrt((C1 + C2) * ks * ks))
    b = _t(0.1 * r.standard_normal(Cout))
    res = _t(r.standard_normal((N, H, W, Cout)), torch.bfloat16)
    temb = _t(r.standard_normal((N, Cout + 32)))
    kw = dict(residual=res, temb=temb, temb_off=32, temb_bstride=Cout + 32, scale=0.7071)
    want_mg = (H * W) % 32 == 0
    op, out, keep = conv_op(x1, x2, w, b, engine=L.ENGINE_TC, mg_stats=want_mg, **kw)
    run_op(op, prepare=True)
    ref = conv_ref(x1, x2, w.to(torch.bfloat16), b, **kw)      # same bf16-rounded weights
    err = rel_l2(out.float().permute(0, 3, 1, 2), ref)
    assert err <= 4e-3, err                                     # bf16 output rounding only
    if want_mg:
        # fused GroupNorm micro-group statistics of the (unrounded) output
        mg = keep[-1]
        mref = mg_ref(ref.permute(0, 2, 3, 1))
        assert torch.isfinite(mg).all()
        assert float((mg.double().cpu() - mref).abs().max()) <= 2e-4 * float(mref.abs().max())
        # and a GroupNorm consuming them equals the GroupNorm that re-reads the tensor
        G = min(Cout // 4, 32)
        ga = _t(1 + 0.2 * r.standard_normal(Cout)); be = _t(0.1 * r.standard_normal(Cout))
        op1, o1, k1 = gn_op(out, None, ga, be, G, True, nchunk=2)
        run_op(op1)
        op2, o2, k2 = gn_op(out, None, ga, be, G, True, nchunk=2, mg1=mg)
        run_op(op2)
        assert rel_l2(o2.float(), o1.float()) <= 3e-3
    # plain (no epilogue terms), checks the accumulation itself at fp32-output precision
    op, out2, keep2 = conv_op(x1, x2, w, None, engine=L.ENGINE_TC, out_nchw_f32=True)
    run_op(op, prepare=True)
    ref2 = conv_ref(x1, x2, w.to(torch.bfloat16), None)
    err2 = rel_l2(out2, ref2)
    assert err2 <= 2e-5, err2


@pytest.mark.parametrize("case", [(2, 17, 17, 256, 256), (3, 33, 33, 64, 256), (1, 65, 65, 64, 128),
                                  (5, 9, 9, 128, 64)])
def test_conv_tc_stride2(case):
    """3x3 stride-2 conv on a FIR-padded map (conv_downsample_2d, up_or_down_sampling.py:178):
    the TMA box walks the input with element stride 2."""
    N, H, W, Cin, Cout = case
    r = _rng(sum(case))
    x = _t(r.standard_normal((N, H, W, Cin)), torch.bfloat16)
    w = _t(r.standard_normal((Cout, Cin, 3, 3)) / np.sqrt(Cin * 9))
    b = _t(0.1 * r.standard_normal(Cout))
    OH = (H - 3) // 2 + 1
    res = _t(r.standard_normal((N, OH, OH, Cout)), torch.bfloat16)
    kw = dict(stride=2, pad=0, residual=res, scale=0.7071)
    op, out, keep = conv_op(x, None, w, b, engine=L.ENGINE_TC, **kw)
    run_op(op, prepare=True)
    ref = conv_ref(x, None, w.to(torch.bfloat16), b, **kw)
    err = rel_l2(out.float().permute(0, 3, 1, 2), ref)
    assert err <= 4e-3, err


@pytest.mark.parametrize("case", [(2, 32, 32, 64, 0, 64), (3, 32, 32, 256, 0, 256), (2, 16, 16, 128, 128, 256),
                                  (5, 16, 16, 256, 0, 128), (1, 32, 32, 256, 128, 256)])
@pytest.mark.parametrize("silu", [True, False])
def test_conv_gn_fused(case, silu):
    """GroupNorm(+SiLU)-on-load 3x3 conv (PSLD_ENGINE_TC_GN): per-(sample, channel) affine + SiLU
    applied to the raw tile in shared memory, three shifted operand variants, 2-CTA MMA."""
    N, H, W, C1, C2, Cout = case
    r = _rng(sum(case) + 5)
    x1 = _t(r.standard_normal((N, H, W, C1)) * 1.7 + 0.3, torch.bfloat16)
    x2 = _t(r.standard_normal((N, H, W, C2)) * 0.6 - 0.2, torch.bfloat16) if C2 else None
    Cin = C1 + C2
    w = _t(r.standard_normal((Cout, Cin, 3, 3)) / np.sqrt(Cin * 9))
    b = _t(0.1 * r.standard_normal(Cout))
    aff = _t(np.stack([1 + 0.3 * r.standard_normal((N, Cin)), 0.2 * r.standard_normal((N, Cin))], -1))
    res = _t(r.standard_normal((N, H, W, Cout)), torch.bfloat16)
    temb = _t(r.standard_normal((N, Cout)))
    kw = dict(residual=res, temb=temb, temb_off=0, temb_bstride=Cout, scale=0.7071)
    op, out, keep = conv_op(x1, x2, w, b, engine=L.ENGINE_TC_GN, mg_stats=True, affine=aff, gn_silu=silu, **kw)
    run_op(op, prepare=True)
    xx = x1.float().cpu() if x2 is None else torch.cat([x1.float().cpu(), x2.float().cpu()], -1)
    a = xx * aff.cpu()[:, None, None, :, 0] + aff.cpu()[:, None, None, :, 1]
    if silu:
        a = F.silu(a)
    a = a.to(torch.bfloat16)
    ref = conv_ref(a, None, w.to(torch.bfloat16), b, **kw)
    err = rel_l2(out.float().permute(0, 3, 1, 2), ref)
    assert err <= 6e-3, err       # bf16 output rounding + tanh-form SiLU before the bf16 rounding of A
    mg = keep[-1]
    mref = mg_ref(ref.permute(0, 2, 3, 1))
    assert float((mg.double().cpu() - mref).abs().max()) <= 5e-3 * float(mref.abs().max())


@pytest.mark.parametrize("case", [(2, 32, 32, 256, 256, 256, 256), (3, 16, 16, 256, 256, 0, 256),
                                  (3, 8, 8, 128, 64, 64, 128), (2, 32, 32, 64, 128, 0, 64)])
def test_conv_tc_fused_shortcut(case):
    """Conv_1 (3x3) with the Conv_2 1x1 shortcut over cat(e1, e2) accumulated into the same
    accumulator as extra K-blocks (layerspp.py:266-274)."""
    N, H, W, Cb, E1, E2, Cout = case
    r = _rng(sum(case) + 9)
    b_in = _t(r.standard_normal((N, H, W, Cb)), torch.bfloat16)
    e1 = _t(r.standard_normal((N, H, W, E1)), torch.bfloat16)
    e2 = _t(r.standard_normal((N, H, W, E2)), torch.bfloat16) if E2 else None
    w = _t(r.standard_normal((Cout, Cb, 3, 3)) / np.sqrt(Cb * 9))
    we = _t(r.standard_normal((Cout, E1 + E2, 1, 1)) / np.sqrt(E1 + E2))
    bias = _t(0.1 * r.standard_normal(Cout))
    op, out, keep = conv_op(b_in, None, w, bias, engine=L.ENGINE_TC, scale=0.7071, ext=(e1, e2, we),
                            mg_stats=(H * W) % 32 == 0)
    run_op(op, prepare=True)
    ref = conv_ref(b_in, None, w.to(torch.bfloat16), bias) + conv_ref(e1, e2, we.to(torch.bfloat16), None)
    ref = ref * 0.7071
    err = rel_l2(out.float().permute(0, 3, 1, 2), ref)
    assert err <= 4e-3, err


@pytest.mark.parametrize("case", [(2, 32, 32, 256, 256, 256, 256), (3, 16, 16, 256, 256, 0, 256),
                                  (2, 32, 32, 128, 64, 0, 128), (3, 16, 16, 256, 128, 256, 256)])
def test_conv_gn_fused_with_shortcut(case):
    """GroupNorm_1+SiLU on load -> Conv_1, plus the Conv_2 1x1 shortcut over the RAW block input
    cat(e1, e2) as extra K-blocks of the same accumulation (layerspp.py:262-274)."""
    N, H, W, Cb, E1, E2, Cout = case
    r = _rng(sum(case) + 13)
    h = _t(r.standard_normal((N, H, W, Cb)) * 1.5 + 0.2, torch.bfloat16)
    e1 = _t(r.standard_normal((N, H, W, E1)), torch.bfloat16)
    e2 = _t(r.standard_normal((N, H, W, E2)), torch.bfloat16) if E2 else None
    w = _t(r.standard_normal((Cout, Cb, 3, 3)) / np.sqrt(Cb * 9))
    we = _t(r.standard_normal((Cout, E1 + E2, 1, 1)) / np.sqrt(E1 + E2))
    bias = _t(0.1 * r.standard_normal(Cout))
    aff = _t(np.stack([1 + 0.3 * r.standard_normal((N, Cb)), 0.2 * r.standard_normal((N, Cb))], -1))
    op, out, keep = conv_op(h, None, w, bias, engine=L.ENGINE_TC_GN, scale=0.7071, ext=(e1, e2, we),
                            mg_stats=True, affine=aff, gn_silu=True)
    run_op(op, prepare=True)
    a = F.silu(h.float().cpu() * aff.cpu()[:, None, None, :, 0] + aff.cpu()[:, None, None, :, 1])
    a = a.to(torch.bfloat16)
    ref = conv_ref(a, None, w.to(torch.bfloat16), bias) + conv_ref(e1, e2, we.to(torch.bfloat16), None)
    ref = ref * 0.7071
    err = rel_l2(out.float().permute(0, 3, 1, 2), ref)
    assert err <= 6e-3, err
    mref = mg_ref(ref.permute(0, 2, 3, 1))
    assert float((keep[-1].double().cpu() - mref).abs().max()) <= 5e-3 * float(mref.abs().max())


def test_conv_gn_fused_output_head():
    """Final act(GroupNorm(h)) -> conv3x3 -> 6 channels as fp32 NCHW through the GroupNorm-on-load
    kernel (Cout zero-padded to one 64-wide N tile)."""
    r = _rng(78)
    N, H, W, Cin = 3, 32, 32, 128
    x = _t(r.standard_normal((N, H, W, Cin)) * 1.3 + 0.1, torch.bfloat16)
    w = _t(r.standard_normal((6, Cin, 3, 3)) / 34.0)
    b = _t(0.1 * r.standard_normal(6))
    aff = _t(np.stack([1 + 0.3 * r.standard_normal((N, Cin)), 0.2 * r.standard_normal((N, Cin))], -1))
    op, out, keep = conv_op(x, None, w, b, engine=L.ENGINE_TC_GN, out_nchw_f32=True, affine=aff, gn_silu=True)
    run_op(op, prepare=True)
    a = F.silu(x.float().cpu() * aff.cpu()[:, None, None, :, 0] + aff.cpu()[:, None, None, :, 1]).to(torch.bfloat16)
    ref = conv_ref(a, None, w.to(torch.bfloat16), b)
    assert out.shape == (N, 6, H, W)
    assert rel_l2(out, ref) <= 3e-3


def test_conv_tc_output_head():
    """3x3 conv to 6 channels written as fp32 NCHW (network output head)."""
    r = _rng(77)
    x = _t(r.standard_normal((2, 32, 32, 128)), torch.bfloat16)
    w = _t(r.standard_normal((6, 128, 3, 3)) / 34.0)
    b = _t(0.1 * r.standard_normal(6))
    op, out, keep = conv_op(x, None, w, b, engine=L.ENGINE_TC, out_nchw_f32=True)
    run_op(op, prepare=True)
    ref = conv_ref(x, None, w.to(torch.bfloat16), b)
    assert out.shape == (2, 6, 32, 32)
    assert rel_l2(out, ref) <= 2e-5


def test_conv_tc_rejects_ineligible():
    x = torch.zeros(1, 8, 8, 48, dtype=torch.bfloat16, device=DEV)
    w = torch.zeros(64, 48, 3, 3, device=DEV)
    op, out, keep = conv_op(x, None, w, None, engine=L.ENGINE_TC)
    rc = L.lib().psld_op_prepare(C.byref(op))
    assert rc == L.EUNSUPPORTED
    assert b"Cin" in L.lib().psld_last_error()


# ------------------------------------------------------------------ attention core
@pytest.mark.parametrize("dtype,tol", [(torch.float32, 3e-6), (torch.bfloat16, 6e-3)])
@pytest.mark.parametrize("shape", [(2, 16, 16, 64), (1, 8, 8, 256), (2, 16, 16, 256), (1, 4, 4, 32)])
def test_attention(dtype, tol, shape):
    N, H, W, Cc = shape
    r = _rng(9)
    qkv = _t(r.standard_normal((N, H, W, 3 * Cc)), dtype)
    op, out = attn_op(qkv, Cc)
    run_op(op)
    q, k, v = qkv.float().cpu().reshape(N, H * W, 3 * Cc).split(Cc, dim=-1)
    wgt = torch.softmax(torch.einsum("bqc,bkc->bqk", q, k) * (int(Cc) ** -0.5), dim=-1)
    ref = torch.einsum("bqk,bkc->bqc", wgt, v)
    assert rel_l2(out.float().reshape(N, H * W, Cc), ref) <= tol


@pytest.mark.parametrize("shape", [(2, 16, 16, 256), (3, 8, 8, 256), (2, 16, 16, 64), (1, 8, 16, 128),
                                   (4, 8, 8, 64)])
def test_attention_tc(shape):
    """tcgen05 attention core (S = QK^T and O = PV in TMEM) vs the fp32 definition."""
    N, H, W, Cc = shape
    r = _rng(19)
    qkv = _t(r.standard_normal((N, H, W, 3 * Cc)) * 1.5, torch.bfloat16)
    op, out = attn_op(qkv, Cc, engine=L.ENGINE_TC)
    run_op(op, prepare=True)
    q, k, v = qkv.float().cpu().reshape(N, H * W, 3 * Cc).split(Cc, dim=-1)
    wgt = torch.softmax(torch.einsum("bqc,bkc->bqk", q, k) * (int(Cc) ** -0.5), dim=-1)
    ref = torch.einsum("bqk,bkc->bqc", wgt, v)
    err = rel_l2(out.float().reshape(N, H * W, Cc), ref)
    assert err <= 8e-3, err          # P and the output are rounded to bf16


@pytest.mark.parametrize("shape", [(2, 16, 16, 256), (3, 16, 8, 128), (5, 16, 16, 64), (1, 16, 16, 192)])
def test_attention_tc_fused_projection(shape):
    """Attention core + NIN_3 output projection + skip connection + GroupNorm statistics in one
    kernel (AttnBlockpp, layerspp.py:82-91) vs the fp32 definition."""
    N, H, W, Cc = shape
    r = _rng(23)
    qkv = _t(r.standard_normal((N, H, W, 3 * Cc)) * 1.5, torch.bfloat16)
    x = _t(r.standard_normal((N, H, W, Cc)), torch.bfloat16)
    w3 = _t(r.standard_normal((Cc, Cc)) / np.sqrt(Cc))           # [out, in]
    b3 = _t(0.1 * r.standard_normal(Cc))
    op, out, keep = attn_op(qkv, Cc, engine=L.ENGINE_TC, proj=(w3, b3, x, 0.7071))
    run_op(op, prepare=True)
    q, k, v = qkv.float().cpu().reshape(N, H * W, 3 * Cc).split(Cc, dim=-1)
    wgt = torch.softmax(torch.einsum("bqc,bkc->bqk", q, k) * (int(Cc) ** -0.5), dim=-1)
    o = torch.einsum("bqk,bkc->bqc", wgt, v)
    ref = (o @ w3.to(torch.bfloat16).float().cpu().t() + b3.cpu() + x.float().cpu().reshape(N, H * W, Cc)) * 0.7071
    err = rel_l2(out.float().reshape(N, H * W, Cc), ref)
    assert err <= 8e-3, err
    mref = mg_ref(ref.reshape(N, H, W, Cc))
    assert float((keep[-1].cpu() - mref).abs().max()) <= 1e-2 * float(mref.abs().max())


# ------------------------------------------------------------------ error behaviour
def test_error_codes():
    lib = L.lib()
    co = L.SscsCoeffs()
    rc = lib.psld_sscs_update(None, None, L.F64, None, None, None, None, None, C.byref(co), 1, 0, 0,
                              1, 12, None)
    assert rc == L.EINVAL and b"null" in lib.psld_last_error()
    u = torch.zeros(1, 6, 1, 1, dtype=torch.float64, device=DEV)
    rc = lib.psld_sscs_update(L.ptr(u), L.ptr(u), L.F64, None, None, None, None, None, C.byref(co),
                              1, 0, 0, 1, 3, None)
    assert rc == L.EINVAL
