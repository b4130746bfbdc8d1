"""Every in-kernel Philox consumer against the host reference of the generator (tests/_philox.py),
and the sampler configuration the benchmark times, pathwise, against an fp64 host chain.

Philox is counter based, so every normal a kernel draws is recomputed on the host from
(seed, stream, index); the phase-space updates are pointwise per pair, so the host follows a
subset of pairs (or, at the 8x8 test sizes, the whole state) through the same draws.  The only
difference left is the device's logf / __sincosf inside Box-Muller: |dz| <= ~3.5e-6 at the tail.

Gates, with the values measured on an NVIDIA B200 at a 1000 W power limit:
  device normals vs host, every entry point, max |dz| ...... 3e-6 (measured 1.53e-6 .. 1.66e-6)
  phase-space updates, per call: |d| <= 3e-6 x (noise coefficients carried through the later stages)
      + 1e-13 max|ref| (f64 state) or + 2e-6 max|ref| (f32 state); and per kernel, the worst
      max-abs / max|ref| over the calls at most 2x the measured value (UPDATE_GATES)
  bb_ode vector kernels, max-abs / max|ref| ................ 1e-15, a few fp64 ulps (measured: drifts
      2.6e-16, psld_rk_combine 1.7e-16);
      psld_rk_error's atomically reduced sum ............... 1e-13 (measured 1.7e-15)
  samplers, pathwise, max-abs / max|ref| ................... per test, measured value beside the gate
"""
import ctypes as C
import subprocess

import numpy as np
import pytest
import torch

import _philox as P
from _net import cc_config, fake_score, make_net, vp_config
from oracle import psld_oracle as O
from oracle.weights import fake_classifier, inpaint_inputs, prior
from psld_b200 import (ClassCondEulerMaruyamaSampler, EulerMaruyamaSampler, InpaintEulerMaruyamaSampler,
                       PSLD, SSCSSampler, VPSDE, cifar10_config, time_grid, tiny_config)
from psld_b200 import _lib as L
from psld_b200.distributed import call_seed
from psld_b200.schedule import InpaintTables, PSLDSchedule, StepTables, VPSchedule, VPStepTables

pytestmark = pytest.mark.gpu
DEV = "cuda"
SEED = call_seed(7, 1, 3)            # nonzero high key word
STEP = 70001                         # step above 2^16
GRID_VECS = 148 * 16 * 256           # vectors one sweep of the capped grid covers
DZ = 3e-6                            # device vs host normal
# (B, chw): the benchmark's CIFAR-10 batch, CelebA-64, the guided CIFAR-10 batch, the 256^2 network
# at B = 32 (2.6 sweeps of the capped grid), one vector, and chw % 8 == 4
SHAPES = [(256, 3072), (64, 12288), (128, 3072), (32, 196608), (1, 4), (3, 20)]
# worst max-abs / max|ref| over the calls of one test, per kernel and state dtype (measured, worst shape)
UPDATE_GATES = {("sscs", torch.float64): 8e-8,     # 4.1e-8
                ("sscs", torch.float32): 4e-7,     # 2.0e-7
                ("em", torch.float64): 5.5e-8,     # 2.7e-8
                ("em", torch.float32): 1.6e-7,     # 8.1e-8
                ("vp", torch.float64): 7.5e-8,     # 3.9e-8
                ("vp", torch.float32): 1.6e-7,     # 8.0e-8
                ("inpaint", torch.float64): 4e-7,  # 2.0e-7
                ("inpaint", torch.float32): 4.3e-7}  # 2.2e-7


@pytest.fixture(scope="module", autouse=True)
def _card():
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True,
                            timeout=30).stdout.strip()
    except Exception:
        pl = "unknown"
    print(f"\n[{torch.cuda.get_device_name()}, power limit {pl}]")


def _vecs(B, chw, rng):
    """4-pair vectors to check: all of a small tensor, else both ends, every grid-sweep boundary
    and a seeded random set."""
    nvec = B * chw // 4
    if nvec <= 1 << 14:
        return np.arange(nvec)
    v = {0, 1, nvec - 2, nvec - 1}
    for k in range(1, nvec // GRID_VECS + 1):
        v |= {k * GRID_VECS - 1, k * GRID_VECS, k * GRID_VECS + 1}
    v |= set(rng.integers(0, nvec, 4096).tolist())
    return np.array(sorted(x for x in v if x < nvec))


def _elems(B, chw, rng):
    """(b, j) of every pair of the chosen vectors."""
    v = _vecs(B, chw, rng)
    q = chw // 4
    b = np.repeat(v // q, 4)
    j = np.repeat((v % q) * 4, 4) + np.tile(np.arange(4), v.size)
    return b, j


def _np(t):
    return t.detach().double().cpu().numpy()


def _at(t, b, col):
    """t.reshape(B, -1)[b, col] gathered on the device, as float64 on the host."""
    ix = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(t.device)
    return _np(t.reshape(t.shape[0], -1)[ix(b), ix(col)])


def _pairs(t, b, j, chw):
    """(x, m) of pairs (b, j) of a [B, 2 chw] state on the host."""
    return _at(t, b, j), _at(t, b, chw + j)


# ------------------------------------------------------------------ device normals, per entry point
def _extract(kind, B, chw):
    """Run a pure-noise call (zero state, unit noise coefficients, f32 state); return the device's
    normals and the host's for the same (seed, stream, index): dict name -> (dev, host)."""
    lib, s = L.lib(), L.stream_ptr()
    u = torch.zeros(B, 2 * chw, dtype=torch.float32, device=DEV)
    out = torch.empty_like(u)
    n = B * chw
    if kind in ("sscs_a", "sscs_b", "sscs_c"):
        st = kind[-1]
        co = L.SscsCoeffs()
        h = getattr(co, "half_" + st)
        h.c11 = h.c22 = 1.0
        L.check(lib.psld_sscs_update(L.ptr(out), L.ptr(u), L.F32, None, None, None, None, None, C.byref(co),
                                     {"a": 1, "b": 4, "c": 8}[st], SEED, STEP, B, chw, s), kind)
        zx, zm = P.pair_normals(SEED, P.sscs_stream(STEP, st), B, chw)
    elif kind in ("em", "em_guided"):
        co = L.ScoreStep()
        co.gs_x = co.gs_m = 1.0
        eps = torch.zeros(B, 2 * chw, dtype=torch.float32, device=DEV)
        guide = torch.zeros_like(eps) if kind == "em_guided" else None
        L.check(lib.psld_em_update_guided(L.ptr(out), L.ptr(u), L.F32, None, L.ptr(eps), L.ptr(guide), 1.0,
                                          None, 1, C.byref(co), SEED, STEP, B, chw, s), kind)
        zx, zm = P.pair_normals(SEED, STEP, B, chw)
    elif kind == "prior":
        L.check(lib.psld_prior_sample(L.ptr(out), 1.0, SEED, B, chw, s), kind)
        zx, zm = P.pair_normals(SEED, P.PRIOR_STREAM, B, chw)
    elif kind == "vp":
        co = L.VpStep()
        co.gs = 1.0
        eps = torch.zeros(n, dtype=torch.float32, device=DEV)
        x = torch.zeros(n, dtype=torch.float32, device=DEV)
        L.check(lib.psld_vp_em_update(L.ptr(x), L.ptr(x), L.F32, None, L.ptr(eps), None, 1, C.byref(co),
                                      SEED, STEP, n, s), kind)
        torch.cuda.synchronize()
        return {"z": (_np(x), P.flat_normals(SEED, STEP, n))}
    elif kind == "inpaint":
        out.zero_()                                   # in place: the masked-out part must be finite
        x0 = torch.zeros(B, chw, dtype=torch.float32, device=DEV)
        mask = torch.ones_like(x0)
        co = L.InpaintStep()
        co.c11 = co.c22 = 1.0                         # x = e_x, m = e_m
        L.check(lib.psld_inpaint_combine(L.ptr(out), L.F32, None, L.ptr(x0), L.ptr(mask), None, None,
                                         C.byref(co), SEED, STEP, B, chw, s), kind)
        co2 = L.InpaintStep()
        co2.a_xm, co2.m0_std, co2.mean_only = 1.0, 1.0, 1   # x = m0 = z_m0
        u2 = torch.zeros_like(u)
        L.check(lib.psld_inpaint_combine(L.ptr(u2), L.F32, None, L.ptr(x0), L.ptr(mask), None, None,
                                         C.byref(co2), SEED, STEP, B, chw, s), kind)
        torch.cuda.synchronize()
        o, o2 = _np(out), _np(u2)
        fl = lambda w: P.flat_normals(SEED, P.inpaint_stream(STEP, w), n).reshape(B, chw)
        return {"e_x": (o[:, :chw], fl(1)), "e_m": (o[:, chw:], fl(2)), "z_m0": (o2[:, :chw], fl(0))}
    torch.cuda.synchronize()
    o = _np(out)
    return {"z_x": (o[:, :chw], zx), "z_m": (o[:, chw:], zm)}


@pytest.mark.parametrize("kind", ["sscs_a", "sscs_b", "sscs_c", "em", "em_guided", "prior", "vp", "inpaint"])
@pytest.mark.parametrize("shape", [(256, 3072), (1, 4), (3, 20)])
def test_device_normals_equal_host_philox(kind, shape):
    """The normals a pure-noise call writes are the host's normal4 at the documented (stream, index),
    over the whole tensor: a wrong stream, index, half or sign would give an O(1) difference."""
    res = _extract(kind, *shape)
    worst = 0.0
    for name, (dev, host) in res.items():
        d = float(np.abs(dev - host).max())
        worst = max(worst, d)
        assert d <= DZ, (kind, name, d)
    print(f"normals {kind} {shape}: max |dz| {worst:.2e}")
    if "z_x" in res and shape[0] * shape[1] >= 8:        # the halves are distinct draws
        assert np.abs(res["z_x"][0] - res["z_m"][1]).max() > 0.5


# ------------------------------------------------------------------ phase-space updates vs fp64 host
def _sscs_row(gamma, nu, decomp="lower"):
    cfg = cifar10_config(n_discrete_steps=1000)
    cfg.model.sde.update(gamma=gamma, nu=nu, decomp_mode=decomp, beta_min=0.1, beta_max=20.0)
    ts, n = time_grid(cfg)
    return StepTables(PSLDSchedule(cfg), ts, n, "sscs_sde", True, 1e-3, merge_noise=True).sscs[400]


def _half(h, x, m, zx, zm):
    return (h.a_xx * x + h.a_xm * m + (h.c11 * zx + h.c12 * zm),
            h.a_mx * x + h.a_mm * m + (h.c21 * zx + h.c22 * zm))


def _score32(sc, ex, em):
    """score from eps in fp32, as the kernel evaluates it (psld.py:252-259)."""
    f = np.float32
    ex, em = ex.astype(np.float32), em.astype(np.float32)
    if sc.mode == 0:
        return f(-f(sc.li11)) * ex - f(sc.li12) * em, f(-f(sc.li21)) * ex - f(sc.li22) * em
    if sc.mode == 1:
        return np.zeros_like(ex), f(-f(sc.li22)) * ex
    return f(-f(sc.li11)) * ex, np.zeros_like(ex)


def _noise_coeff(h):
    return max(abs(h.c11) + abs(h.c12), abs(h.c21) + abs(h.c22))


def _gate(err, scale, bound, dtype):
    """f64 state: the normal bound; f32 state: plus fp32 rounding of the state."""
    return err <= bound + (1e-13 if dtype == torch.float64 else 2e-6) * scale


@pytest.mark.parametrize("state_dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("shape", SHAPES)
def test_sscs_update_philox_vs_host(shape, state_dtype):
    """psld_sscs_update, all 15 stage masks, Philox with some z_* given and others NULL, eps modes
    0/1/2, in place and out of place, net_in on and off, against fp64 on the host."""
    B, chw = shape
    rng = np.random.default_rng(sum(shape))
    b, j = _elems(B, chw, rng)
    lib, s = L.lib(), L.stream_ptr()
    g = torch.Generator(device=DEV).manual_seed(11)
    rows = {0: _sscs_row(0.01, 4.01), 1: _sscs_row(0.0, 4.0), 2: _sscs_row(0.01, 0.0, "upper")}
    worst = 0.0
    for stages in range(1, 16):
        mode, inplace, with_net = stages % 3, bool(stages & 1), bool(stages & 2) == bool(stages & 8)
        co = rows[mode]
        u0 = (torch.randn(B, 2 * chw, generator=g, device=DEV, dtype=torch.float64) * 1.5).to(state_dtype)
        eps = torch.randn(B, (2 if mode == 0 else 1) * chw, generator=g, device=DEV)
        # pre-drawn noise for one stage in three (which one rotates with the mask), Philox elsewhere
        given = {st: torch.randn(B, 2 * chw, generator=g, device=DEV) if (stages + k) % 3 == 0 else None
                 for k, st in enumerate("abc")}
        x, m = _pairs(u0, b, j, chw)
        out = u0 if inplace else torch.empty_like(u0)
        net_in = torch.full((B, 2 * chw), float("nan"), device=DEV) if with_net else None
        L.check(lib.psld_sscs_update(L.ptr(out), L.ptr(u0), L.dtype_code(state_dtype), L.ptr(net_in),
                                     L.ptr(eps), L.ptr(given["a"]), L.ptr(given["b"]), L.ptr(given["c"]),
                                     C.byref(co), stages, SEED, STEP, B, chw, s), "sscs")
        torch.cuda.synchronize()
        bound = 0.0
        for bit, st in ((1, "a"), (2, None), (4, "b"), (8, "c")):
            if not stages & bit:
                continue
            if st is None:
                ex = _at(eps, b, j)
                em = _at(eps, b, chw + j) if mode == 0 else np.zeros_like(ex)
                sx, sm = _score32(co.score, ex, em)
                x = x + co.score.k_x * (sx.astype(np.float64) + x)
                m = m + co.score.k_m * (sm.astype(np.float64) + co.score.m_inv * m)
                bound *= max(abs(1 + co.score.k_x), abs(1 + co.score.k_m * co.score.m_inv))
                continue
            h = getattr(co, "half_" + st)
            bound *= max(abs(h.a_xx) + abs(h.a_xm), abs(h.a_mx) + abs(h.a_mm))
            if given[st] is not None:
                zx, zm = _pairs(given[st], b, j, chw)
            else:
                zx, zm = P.pair_normals_at(SEED, P.sscs_stream(STEP, st), b, j, chw)
                bound += DZ * _noise_coeff(h)
            x, m = _half(h, x, m, zx, zm)
        gx, gm = _pairs(out, b, j, chw)
        err = max(np.abs(gx - x).max(), np.abs(gm - m).max())
        scale = max(np.abs(x).max(), np.abs(m).max())
        worst = max(worst, err / scale)
        assert _gate(err, scale, bound, state_dtype), (stages, err, bound, scale)
        if with_net:
            assert torch.equal(net_in, out.to(torch.float32))
    print(f"sscs {shape} {state_dtype}: worst max-abs/max|ref| {worst:.2e}")
    assert worst <= UPDATE_GATES["sscs", state_dtype], worst


@pytest.mark.parametrize("state_dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("shape", SHAPES)
def test_em_update_philox_vs_host(shape, state_dtype):
    """psld_em_update[_guided]: Philox, pre-drawn and no noise; guided and plain; eps modes 0/1/2;
    in place and out of place; net_in on and off."""
    B, chw = shape
    rng = np.random.default_rng(sum(shape) + 1)
    b, j = _elems(B, chw, rng)
    lib, s = L.lib(), L.stream_ptr()
    g = torch.Generator(device=DEV).manual_seed(12)
    worst = 0.0
    for case in range(12):
        mode, noise, guided = case % 3, (case // 3) % 3, case >= 6      # noise: 0 Philox, 1 given, 2 none
        inplace, with_net = bool(case & 1), bool(case & 2)
        gamma, nu, dec = {0: (0.01, 4.01, "lower"), 1: (0.0, 4.0, "lower"), 2: (0.01, 0.0, "upper")}[mode]
        cfg = cifar10_config(n_discrete_steps=1000)
        cfg.model.sde.update(gamma=gamma, nu=nu, decomp_mode=dec, beta_min=0.1, beta_max=20.0)
        ts, n = time_grid(cfg)
        co = StepTables(PSLDSchedule(cfg), ts, n, "em_sde", True, 1e-3).em[300]
        u0 = (torch.randn(B, 2 * chw, generator=g, device=DEV, dtype=torch.float64) * 1.5).to(state_dtype)
        eps = torch.randn(B, (2 if mode == 0 else 1) * chw, generator=g, device=DEV)
        guide = torch.randn(B, 2 * chw, generator=g, device=DEV) if guided else None
        z = torch.randn(B, 2 * chw, generator=g, device=DEV) if noise == 1 else None
        out = u0 if inplace else torch.empty_like(u0)
        net_in = torch.empty(B, 2 * chw, device=DEV) if with_net else None
        x, m = _pairs(u0, b, j, chw)
        L.check(lib.psld_em_update_guided(L.ptr(out), L.ptr(u0), L.dtype_code(state_dtype), L.ptr(net_in),
                                          L.ptr(eps), L.ptr(guide), 2.5, L.ptr(z), int(noise == 0),
                                          C.byref(co), SEED, STEP, B, chw, s), "em")
        torch.cuda.synchronize()
        ex = _at(eps, b, j)
        em = _at(eps, b, chw + j) if mode == 0 else np.zeros_like(ex)
        sx, sm = _score32(co, ex, em)
        fx = co.half_beta * (co.m_inv * m - co.gamma * x)
        fm = co.half_beta * (-co.nu * m - x)
        fbx, fbm = -fx + co.g2_x * sx.astype(np.float64), -fm + co.g2_m * sm.astype(np.float64)
        if guided:
            gx, gm = _pairs(guide, b, j, chw)
            fbx, fbm = fbx + co.g2_x * (gx * 2.5), fbm + co.g2_m * (gm * 2.5)
        nx, nm = x + fbx * co.dt, m + fbm * co.dt
        bound = 0.0
        if noise == 0:
            zx, zm = P.pair_normals_at(SEED, STEP, b, j, chw)
            bound = DZ * max(abs(co.gs_x), abs(co.gs_m))
        elif noise == 1:
            zx, zm = _pairs(z, b, j, chw)
        if noise != 2:
            nx, nm = nx + co.gs_x * zx, nm + co.gs_m * zm
        ox, om = _pairs(out, b, j, chw)
        err = max(np.abs(ox - nx).max(), np.abs(om - nm).max())
        scale = max(np.abs(nx).max(), np.abs(nm).max())
        worst = max(worst, err / scale)
        assert _gate(err, scale, bound, state_dtype), (case, err, bound, scale)
        if with_net:
            assert torch.equal(net_in, out.to(torch.float32))
    print(f"em {shape} {state_dtype}: worst max-abs/max|ref| {worst:.2e}")
    assert worst <= UPDATE_GATES["em", state_dtype], worst


@pytest.mark.parametrize("state_dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("shape", SHAPES)
def test_vp_em_update_philox_vs_host(shape, state_dtype):
    """psld_vp_em_update over the flat [n] state: Philox, pre-drawn and no noise."""
    B, chw = shape
    n = B * chw
    rng = np.random.default_rng(sum(shape) + 2)
    b, j = _elems(B, chw, rng)
    e = b * chw + j
    lib, s = L.lib(), L.stream_ptr()
    g = torch.Generator(device=DEV).manual_seed(13)
    cfg = vp_config(n_discrete_steps=1000)
    ts, nn = time_grid(cfg)
    co = VPStepTables(VPSchedule(cfg), ts, nn, True, 1e-3).steps[250]
    worst = 0.0
    for case in range(4):
        noise, inplace = case % 3, bool(case & 1)
        x0 = (torch.randn(n, generator=g, device=DEV, dtype=torch.float64) * 1.5).to(state_dtype)
        eps = torch.randn(n, generator=g, device=DEV)
        z = torch.randn(n, generator=g, device=DEV) if noise == 1 else None
        out = x0 if inplace else torch.empty_like(x0)
        net_in = torch.empty(n, device=DEV) if case == 3 else None
        flat = lambda t: _at(t.view(1, -1), np.zeros_like(e), e)
        x = flat(x0)
        L.check(lib.psld_vp_em_update(L.ptr(out), L.ptr(x0), L.dtype_code(state_dtype), L.ptr(net_in),
                                      L.ptr(eps), L.ptr(z), int(noise == 0), C.byref(co), SEED, STEP, n, s), "vp")
        torch.cuda.synchronize()
        score = flat(eps) * co.neg_inv_std
        ref = (x + (co.half_beta * x + co.g2 * score) * co.dt)
        bound = 0.0
        if noise == 0:
            ref = ref + co.gs * P.flat_normals_at(SEED, STEP, e)
            bound = DZ * abs(co.gs)
        elif noise == 1:
            ref = ref + co.gs * flat(z)
        err = np.abs(flat(out) - ref).max()
        scale = np.abs(ref).max()
        worst = max(worst, err / scale)
        assert _gate(err, scale, bound, state_dtype), (case, err, bound, scale)
        if net_in is not None:
            assert torch.equal(net_in, out.to(torch.float32))
    print(f"vp em {shape} {state_dtype}: worst max-abs/max|ref| {worst:.2e}")
    assert worst <= UPDATE_GATES["vp", state_dtype], worst


@pytest.mark.parametrize("state_dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("shape", SHAPES)
def test_inpaint_combine_philox_vs_host(shape, state_dtype):
    """psld_inpaint_combine: the three Philox streams, (z_m0 NULL, z_eps given), both given; DSM and
    HSM coefficients; mean_only; net_in on and off."""
    B, chw = shape
    rng = np.random.default_rng(sum(shape) + 3)
    b, j = _elems(B, chw, rng)
    e = b * chw + j
    lib, s = L.lib(), L.stream_ptr()
    g = torch.Generator(device=DEV).manual_seed(14)
    worst = 0.0
    for case in range(6):
        noise, hsm, mean_only = case % 3, case < 3, case == 5     # noise: 0 Philox, 1 z_eps only, 2 both
        cfg = tiny_config(sampler="ip_em_sde", n_discrete_steps=1000)
        cfg.training.mode = "hsm" if hsm else "dsm"
        ts, n = time_grid(cfg)
        co = InpaintTables(PSLDSchedule(cfg), ts, n, True, 1e-3, hsm).steps[600]
        co.mean_only = int(mean_only)
        u = (torch.randn(B, 2 * chw, generator=g, device=DEV, dtype=torch.float64) * 1.5).to(state_dtype)
        x0 = torch.rand(B, chw, generator=g, device=DEV) * 2 - 1
        mask = (torch.rand(B, chw, generator=g, device=DEV) < 0.5).float()
        zm0 = torch.randn(B, chw, generator=g, device=DEV) if noise == 2 else None
        zeps = torch.randn(B, 2 * chw, generator=g, device=DEV) if noise >= 1 else None
        net_in = torch.empty(B, 2 * chw, device=DEV) if case & 1 else None
        x, m = _pairs(u, b, j, chw)
        L.check(lib.psld_inpaint_combine(L.ptr(u), L.dtype_code(state_dtype), L.ptr(net_in), L.ptr(x0),
                                         L.ptr(mask), L.ptr(zm0), L.ptr(zeps), C.byref(co), SEED, STEP, B,
                                         chw, s), "inpaint")
        torch.cuda.synchronize()
        if noise == 0:
            z0, ex, em = (P.flat_normals_at(SEED, P.inpaint_stream(STEP, w), e) for w in range(3))
        else:
            z0 = _at(zm0, b, j) if noise == 2 else np.zeros(e.size)
            ex, em = _pairs(zeps, b, j, chw)
        xo, mk = _at(x0, b, j), _at(mask, b, j)
        m0 = co.m0_std * z0
        xk, mkk = co.a_xx * xo + co.a_xm * m0, co.a_mx * xo + co.a_mm * m0
        if not mean_only:
            xk, mkk = xk + co.c11 * ex + co.c12 * em, mkk + co.c21 * ex + co.c22 * em
        rx, rm = x * (1 - mk) + xk * mk, m * (1 - mk) + mkk * mk
        bound = 0.0
        if noise == 0:
            bound = DZ * (co.m0_std * max(abs(co.a_xm), abs(co.a_mm)) + (0 if mean_only else _noise_coeff(co)))
        ox, om = _pairs(u, b, j, chw)
        err = max(np.abs(ox - rx).max(), np.abs(om - rm).max())
        scale = max(np.abs(rx).max(), np.abs(rm).max())
        worst = max(worst, err / scale)
        assert _gate(err, scale, bound, state_dtype), (case, err, bound, scale)
        if net_in is not None:
            assert torch.equal(net_in, u.to(torch.float32))
    print(f"inpaint {shape} {state_dtype}: worst max-abs/max|ref| {worst:.2e}")
    assert worst <= UPDATE_GATES["inpaint", state_dtype], worst


# ------------------------------------------------------------------ bb_ode vector kernels
@pytest.mark.parametrize("state_dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("shape", SHAPES)
def test_reverse_drifts_vs_fp64(shape, state_dtype):
    """psld_reverse_drift (eps modes 0/1/2) and psld_vp_reverse_drift at the benchmark and grid-stride
    sizes: f32 state evaluates the drift bracket in fp32 like the reference, the rest in fp64."""
    B, chw = shape
    rng = np.random.default_rng(sum(shape) + 4)
    b, j = _elems(B, chw, rng)
    lib, s = L.lib(), L.stream_ptr()
    g = torch.Generator(device=DEV).manual_seed(15)
    f = np.float32
    worst = 0.0
    for mode in range(3):
        gamma, nu, dec = {0: (0.01, 4.01, "lower"), 1: (0.0, 4.0, "lower"), 2: (0.01, 0.0, "upper")}[mode]
        cfg = cifar10_config(n_discrete_steps=1000)
        cfg.model.sde.update(gamma=gamma, nu=nu, decomp_mode=dec, beta_min=0.1, beta_max=20.0)
        ts, n = time_grid(cfg)
        co = StepTables(PSLDSchedule(cfg), ts, n, "em_sde", True, 1e-3).em[700]
        u = (torch.randn(B, 2 * chw, generator=g, device=DEV, dtype=torch.float64) * 1.5).to(state_dtype)
        eps = torch.randn(B, (2 if mode == 0 else 1) * chw, generator=g, device=DEV)
        out = torch.full((B, 2 * chw), float("nan"), dtype=torch.float64, device=DEV)
        L.check(lib.psld_reverse_drift(L.ptr(out), L.ptr(u), L.dtype_code(state_dtype), L.ptr(eps), C.byref(co),
                                       0.5, B, chw, s), "reverse_drift")
        torch.cuda.synchronize()
        x, m = _pairs(u, b, j, chw)
        ex = _at(eps, b, j)
        em = _at(eps, b, chw + j) if mode == 0 else np.zeros_like(ex)
        sx, sm = _score32(co, ex, em)
        if state_dtype == torch.float32:
            x32, m32 = x.astype(f), m.astype(f)
            bx = (f(co.m_inv) * m32 - f(co.gamma) * x32).astype(np.float64)
            bm = (f(-f(co.nu)) * m32 - x32).astype(np.float64)
        else:
            bx, bm = co.m_inv * m - co.gamma * x, -co.nu * m - x
        rx = -(co.half_beta * bx) + co.g2_x * (sx * f(0.5)).astype(np.float64)
        rm = -(co.half_beta * bm) + co.g2_m * (sm * f(0.5)).astype(np.float64)
        ox, om = _pairs(out, b, j, chw)
        e = max(np.abs(ox - rx).max(), np.abs(om - rm).max()) / max(np.abs(rx).max(), np.abs(rm).max())
        worst = max(worst, e)
        assert e <= 1e-15, (mode, e)
    # VP-SDE twin over the flat state
    cfg = vp_config(n_discrete_steps=1000)
    ts, n = time_grid(cfg)
    co = VPStepTables(VPSchedule(cfg), ts, n, True, 1e-3).steps[700]
    x = (torch.randn(B * chw, generator=g, device=DEV, dtype=torch.float64) * 1.5).to(state_dtype)
    eps = torch.randn(B * chw, generator=g, device=DEV)
    out = torch.full((B * chw,), float("nan"), dtype=torch.float64, device=DEV)
    L.check(lib.psld_vp_reverse_drift(L.ptr(out), L.ptr(x), L.dtype_code(state_dtype), L.ptr(eps), C.byref(co),
                                      0.5, B * chw, s), "vp_reverse_drift")
    torch.cuda.synchronize()
    flat = lambda t: _at(t.view(1, -1), np.zeros_like(b), b * chw + j)
    ref = -(-co.half_beta * flat(x)) + co.g2 * (0.5 * (flat(eps) * co.neg_inv_std))
    e = np.abs(flat(out) - ref).max() / np.abs(ref).max()
    worst = max(worst, e)
    assert e <= 1e-15, e
    print(f"reverse drifts {shape} {state_dtype}: worst max-abs/max|ref| {worst:.2e}")


@pytest.mark.parametrize("n", [1000, 3 * GRID_VECS * 4 // 3 + 37])
def test_rk_combine_and_error_vs_fp64(n):
    """psld_rk_combine for 0..8 terms with out or out32 NULL, and psld_rk_error with n past the grid
    cap (several blocks add atomically), against fp64 on the host; n not a multiple of 256."""
    lib, s = L.lib(), L.stream_ptr()
    g = torch.Generator(device=DEV).manual_seed(16)
    y = torch.randn(n, generator=g, device=DEV, dtype=torch.float64)
    K = torch.randn(8, n, generator=g, device=DEV, dtype=torch.float64)
    coef = np.random.default_rng(n).standard_normal(8)
    yh, Kh = _np(y), _np(K)
    h = 0.0123
    worst = 0.0
    for terms in range(9):
        acc = np.zeros(n)
        for t in range(terms):
            acc = acc + Kh[t] * coef[t]
        ref = yh + acc * h
        for which in ("both", "out", "out32"):
            out = torch.full((n,), float("nan"), dtype=torch.float64, device=DEV) if which != "out32" else None
            o32 = torch.full((n,), float("nan"), device=DEV) if which != "out" else None
            L.check(lib.psld_rk_combine(L.ptr(out), L.ptr(o32), L.ptr(y), L.ptr(K) if terms else None,
                                        (C.c_double * 8)(*coef) if terms else None, terms, h, n, s), "rk_combine")
            torch.cuda.synchronize()
            if out is not None:
                e = np.abs(_np(out) - ref).max() / np.abs(ref).max()
                worst = max(worst, e)
                assert e <= 1e-15, (terms, which, e)
            if o32 is not None:       # the float32 rounding of the fp64 value (1 ulp for a last-bit tie)
                d = np.abs(_np(o32) - ref.astype(np.float32))
                assert (d <= np.abs(ref) * 2.0 ** -23).all(), (terms, which)
    print(f"rk_combine n={n}: worst max-abs/max|ref| {worst:.2e}")
    # error norm: sum of squares of the scaled error estimate, accumulated across blocks
    y_new = torch.randn(n, generator=g, device=DEV, dtype=torch.float64)
    atol, rtol = 1e-5, 1e-4
    sc = atol + np.maximum(np.abs(yh), np.abs(_np(y_new))) * rtol
    for terms in (1, 7, 8):
        acc = np.zeros(n)
        for t in range(terms):
            acc = acc + Kh[t] * coef[t]
        ref = float(np.sum(np.square(acc * h / sc)))
        tot = torch.full((1,), 3.0, dtype=torch.float64, device=DEV)   # the kernel adds to *sum_out
        L.check(lib.psld_rk_error(L.ptr(y), L.ptr(y_new), L.ptr(K), (C.c_double * 8)(*coef), terms, h, atol,
                                  rtol, n, L.ptr(tot), s), "rk_error")
        torch.cuda.synchronize()
        e = abs(float(tot) - 3.0 - ref) / ref
        print(f"rk_error n={n} terms={terms}: rel {e:.2e}")
        assert e <= 1e-13, (terms, e)


# ------------------------------------------------------------------ samplers, pathwise
def _state_noise(seed, stream, shape):
    """[B, 2C, H, W] normals of one PSLD-state draw."""
    B, C2, H, W = shape
    zx, zm = P.pair_normals(seed, stream, B, C2 // 2 * H * W)
    return torch.from_numpy(np.concatenate([zx, zm], 1).reshape(shape))


def _pixels(B, HW, rng, k=64):
    """(b, p) pixels to follow: the corners of the batch and of the map (j = 0 and j = chw - 4 among
    them) and a seeded random set."""
    b = [0, 0, 0, B - 1, B - 1, B - 1] + rng.integers(0, B, k).tolist()
    p = [0, HW - 4, HW - 1, 0, HW - 4, HW - 1] + rng.integers(0, HW, k).tolist()
    return np.array(b), np.array(p)


def _pixel_noise(seed, stream, bs, ps, C, HW):
    """[K, 2C, 1, 1] normals of one PSLD-state draw at pixels (bs, ps), all channels."""
    j = np.arange(C)[None, :] * HW + ps[:, None]
    zx, zm = P.pair_normals_at(seed, stream, np.broadcast_to(bs[:, None], j.shape), j, C * HW)
    return torch.from_numpy(np.concatenate([zx, zm], 1)[..., None, None])


def _merged_sscs(cfg, score_fn, u0, ts, n, z, denoise=True, eps=1e-3):
    """SSCS with half B of step i and half A of step i+1 drawn as one Gaussian (the sampler's
    merge_noise): oracle half-step and score algebra; the merged pair is A = A_c A_b, L the lower
    Cholesky factor of A_c L_b L_b^T A_c^T + L_c L_c^T; ``z(stream)`` gives the draws."""
    sde = O.PSLDScalars(cfg)
    halves = [sde.half_step(float(ts[i]), float(ts[i + 1] - ts[i]) / 2) for i in range(n)]

    def apply(a, c, u, zz):
        x, m = torch.chunk(u, 2, dim=1)
        zx, zm = torch.chunk(zz.to(torch.float64), 2, dim=1)
        return torch.cat([a[0] * x + a[1] * m + (c[0] * zx + c[1] * zm),
                          a[2] * x + a[3] * m + (c[2] * zx + c[3] * zm)], dim=1)

    u = u0.to(torch.float64)
    if n:
        u = apply(*halves[0], u, z(0))
    for i in range(n):
        t, dt = float(ts[i]), float(ts[i + 1] - ts[i])
        tau = sde.T - t
        beta = sde.beta_t(tau)
        e = score_fn(u.to(torch.float32), O._tvec(u, float(np.float32(tau))))
        sx, sm = torch.chunk(O.score_from_eps(sde, e, tau), 2, dim=1)
        x, m = torch.chunk(u, 2, dim=1)
        x = x + dt * sde.gamma * beta * (sx + x)
        m = m + dt * sde.m * sde.nu * beta * (sm + sde.m_inv * m)
        u = torch.cat([x, m], dim=1)
        if i + 1 < n:
            (ab, lb), (ac, lc) = ([np.array(v).reshape(2, 2) for v in h] for h in (halves[i], halves[i + 1]))
            S = ac @ lb @ lb.T @ ac.T + lc @ lc.T
            lo = np.linalg.cholesky(S)
            u = apply((ac @ ab).reshape(-1), lo.reshape(-1), u, z(2 * i + 1))
        else:
            u = apply(*halves[i], u, z(2 * i + 1))
    if denoise:
        u = O._denoise(sde, score_fn, u, eps)
    return u


def _err(out, ref):
    return float((out.double().cpu() - ref).abs().max() / ref.abs().max())


EPS_CONST = [0.3, -0.2, 0.1, -0.4, 0.25, 0.05]


@pytest.fixture(scope="module")
def cifar_const():
    """CIFAR-10 NCSN++ (default bf16x3 tier) whose output head returns a fixed per-channel eps:
    the whole native loop runs at the benchmark's batch while the host follows pairs exactly."""
    cfg = cifar10_config(n_discrete_steps=100)
    net, _ = make_net(cfg, "bf16x3")
    head = net.all_modules[-1]
    with torch.no_grad():
        head.weight.zero_()
        head.bias.copy_(torch.tensor(EPS_CONST))
    return cfg, net


def test_native_constant_head_is_exact(cifar_const):
    cfg, net = cifar_const
    u = prior((256, 3, 32, 32), 2.0, 3).cuda()
    e = net(u, torch.full((256,), 0.37, device=DEV))
    want = net.all_modules[-1].bias.detach().view(1, 6, 1, 1).expand(256, 6, 32, 32)
    assert torch.equal(e, want)


# (kind, fuse_halves, merge_noise, cuda_graph, state dtype, gate): the benchmark's configuration first
NATIVE = [("sscs_sde", True, True, True, torch.float64, 2.6e-7),     # measured 1.32e-7
          ("sscs_sde", True, True, False, torch.float64, 2.6e-7),    # 1.32e-7
          ("sscs_sde", True, False, True, torch.float64, 3.3e-7),    # 1.66e-7
          ("sscs_sde", True, False, False, torch.float64, 3.3e-7),   # 1.66e-7
          ("sscs_sde", False, False, True, torch.float64, 3.3e-7),   # 1.66e-7
          ("sscs_sde", False, False, False, torch.float64, 3.3e-7),  # 1.66e-7
          ("em_sde", False, False, True, torch.float64, 3.6e-7),     # 1.80e-7
          ("em_sde", False, False, False, torch.float64, 3.6e-7),    # 1.80e-7
          ("sscs_sde", True, True, True, torch.float32, 2.6e-6)]     # 1.32e-6


@pytest.mark.parametrize("kind,fuse,merge,graph,sdt,gate", NATIVE)
def test_native_sampler_pathwise(cifar_const, kind, fuse, merge, graph, sdt, gate):
    """SSCSSampler / EulerMaruyamaSampler.sample through psld_sampler_run at B = 256, 100 NFE, Philox
    noise, against an fp64 host chain on a subset of pixels (all six channels each)."""
    cfg, net = cifar_const
    cfg.evaluation.sampler.name = kind
    S = (SSCSSampler if kind == "sscs_sde" else EulerMaruyamaSampler)(cfg, PSLD(cfg), net)
    S.fuse_halves, S.merge_noise, S.use_graph, S.state_dtype = fuse, merge, graph, sdt
    S.calls = 3                                          # a key with a nonzero high word
    ts, n = time_grid(cfg)
    B, HW = 256, 1024
    u0 = prior((B, 3, 32, 32), float(np.sqrt(PSLD(cfg).m)), 1)
    out = S.sample(u0.cuda(), ts.cuda(), n, denoise=True, eps=1e-3)
    torch.cuda.synchronize()
    seed = S.seed
    assert seed >> 32
    bs, ps = _pixels(B, HW, np.random.default_rng(5))
    sub = lambda t: t.reshape(B, 6, HW)[bs, :, ps].reshape(-1, 6, 1, 1)
    e_const = torch.tensor(EPS_CONST, dtype=torch.float32).view(1, 6, 1, 1)
    score_fn = lambda u, t: e_const.expand(u.shape[0], 6, 1, 1)
    z = lambda stream: _pixel_noise(seed, stream, bs, ps, 3, HW)
    tsn, _ = O.time_grid(cfg)
    u0s = sub(u0)
    if kind == "em_sde":
        ref = O.em_sample(cfg, score_fn, u0s, tsn, n, [z(i) for i in range(n)])
    elif fuse and merge:
        ref = _merged_sscs(cfg, score_fn, u0s, tsn, n, z)
    else:
        ref = O.sscs_sample(cfg, score_fn, u0s, tsn, n, [z(k) for k in range(2 * n)])
    e = _err(sub(out.cpu()), ref)
    print(f"native {kind} fuse={fuse} merge={merge} graph={graph} {sdt}: max-abs/max|ref| {e:.2e}")
    assert e <= gate, e


def _generic(cls, cfg, score_fn, *extra, fuse=True, merge=True):
    S = cls(cfg, PSLD(cfg) if not str(cfg.model.sde.name) == "vpsde" else VPSDE(cfg), score_fn, *extra)
    S.state_dtype = torch.float64
    S.fuse_halves, S.merge_noise = fuse, merge
    S.calls = 3
    return S


@pytest.mark.parametrize("merge", [False, True])
def test_generic_sscs_pathwise(merge):
    """SSCS with a generic score_fn (Python loop over psld_sscs_update), fused halves with and without
    the merged draw, 1000 NFE, against the oracle chain on the host's Philox draws."""
    cfg = tiny_config(sampler="sscs_sde", n_discrete_steps=1000)
    cfg.data.image_size = 8
    cfg.model.sde.update(beta_min=0.1, beta_max=20.0)
    S = _generic(SSCSSampler, cfg, fake_score, merge=merge)
    ts, n = time_grid(cfg)
    u0 = prior((4, 3, 8, 8), float(np.sqrt(PSLD(cfg).m)), 2)
    out = S.sample(u0.cuda(), ts.cuda(), n)
    torch.cuda.synchronize()
    z = lambda k: _state_noise(S.seed, k, u0.shape)
    tsn, _ = O.time_grid(cfg)
    if merge:
        ref = _merged_sscs(cfg, fake_score, u0, tsn, n, z)
    else:
        ref = O.sscs_sample(cfg, fake_score, u0, tsn, n, [z(k) for k in range(2 * n)])
    e = _err(out, ref)
    print(f"generic sscs merge={merge} 1000 NFE: max-abs/max|ref| {e:.2e}")
    assert e <= (6.2e-7 if merge else 7.5e-7), e          # measured 3.11e-7 / 3.78e-7


def test_generic_cc_em_pathwise():
    """Classifier-guided EM (psld_em_update_guided) with Philox noise against oracle.cc_em_sample."""
    cfg = cc_config()
    S = _generic(ClassCondEulerMaruyamaSampler, cfg, fake_score, fake_classifier)
    ts, n = time_grid(cfg)
    u0 = prior((4, 3, 8, 8), float(np.sqrt(PSLD(cfg).m)), 3)
    out = S.sample(u0.cuda(), ts.cuda(), n)
    torch.cuda.synchronize()
    tsn, _ = O.time_grid(cfg)
    ref = O.cc_em_sample(cfg, fake_score, fake_classifier, u0, tsn, n,
                         [_state_noise(S.seed, i, u0.shape) for i in range(n)], 3, 2.5)
    e = _err(out, ref)
    print(f"generic cc_em: max-abs/max|ref| {e:.2e}")
    assert e <= 3.1e-7, e                                  # measured 1.55e-7


@pytest.mark.parametrize("mode", ["hsm", "dsm"])
def test_generic_inpaint_pathwise(mode):
    """Inpainting EM with the device prior, the predictor's and the three combine streams from
    Philox, against oracle.inpaint_em_sample on the host's draws."""
    cfg = tiny_config(sampler="ip_em_sde", n_discrete_steps=60)
    cfg.training.mode = mode
    cfg.data.image_size = 8
    S = _generic(InpaintEulerMaruyamaSampler, cfg, fake_score)
    ts, n = time_grid(cfg)
    B, Cc, H = 4, 3, 8
    x_0, mask = inpaint_inputs(B, H, 7)
    out = S.sample((x_0.cuda(), mask.cuda()), ts, n)
    torch.cuda.synchronize()
    seed, chw = S.seed, Cc * H * H
    sde = O.PSLDScalars(cfg)
    zx, zm = P.pair_normals(seed, P.PRIOR_STREAM, B, chw)
    m_std = np.float32(np.sqrt(sde.m))
    pri = np.concatenate([zx.astype(np.float32), zm.astype(np.float32) * m_std], 1).reshape(B, 2 * Cc, H, H)
    fl = lambda k, w: P.flat_normals(seed, P.inpaint_stream(k, w), B * chw).reshape(B, Cc, H, H)
    noise = {"pred": [_state_noise(seed, i, (B, 2 * Cc, H, H)) for i in range(n)],
             "m0": [torch.from_numpy(fl(k, 0)) for k in range(n + 2)],
             "eps": [torch.from_numpy(np.concatenate([fl(k, 1), fl(k, 2)], 1)) for k in range(n + 2)]}
    ref = O.inpaint_em_sample(cfg, fake_score, x_0, mask, torch.from_numpy(pri), O.time_grid(cfg)[0], n, noise)
    e = _err(out, ref)
    print(f"generic inpaint {mode}: max-abs/max|ref| {e:.2e}")
    assert e <= 5.5e-7, e                                  # measured 2.79e-7 (HSM and DSM)


def test_generic_vp_em_pathwise():
    """VP-SDE Euler-Maruyama (psld_vp_em_update) with Philox noise against oracle.vp_em_sample."""
    cfg = vp_config(n_discrete_steps=200)
    S = _generic(EulerMaruyamaSampler, cfg, fake_score)
    ts, n = time_grid(cfg)
    x0 = prior((4, 3, 8, 8), 1.0, 4)[:, :3].contiguous()
    out = S.sample(x0.cuda(), ts, n)
    torch.cuda.synchronize()
    noise = [torch.from_numpy(P.flat_normals(S.seed, i, x0.numel()).reshape(x0.shape)) for i in range(n)]
    ref = O.vp_em_sample(cfg, fake_score, x0, O.time_grid(cfg)[0], n, noise)
    e = _err(out, ref)
    print(f"generic vp em: max-abs/max|ref| {e:.2e}")
    assert e <= 5.6e-7, e                                  # measured 2.80e-7
