"""Sampler parity on the GPU: per-step states and final samples vs golden vectors produced by
the reference sampler (identical weights, identical pre-drawn noise).

Tolerances, relative to max|ref| (trajectories with random weights expand, SURVEY.md §8c):
  sampler algebra alone (fake score, fp64 state) ... max-abs/max|ref| <= 1e-6 and rel-L2 <= 1e-6
      (limited by the fp32 score network boundary, not by the fused update: ~1e-8 measured on CPU)
  tiny NCSN++, fp32 network, fp64 state, 100 NFE .... rel-L2 <= 1e-5, max-abs/max|ref| <= 1e-5
      (measured on B200: 3.4e-7 / 3.9e-7)
  bf16 network path (stated separately) ............. rel-L2 <= 6e-3 (measured 3.1e-3; gate <= 2x)
  bf16x3 network path (default tier) ................ rel-L2 <= 1e-4 (measured 4.8e-6; tests/test_gpu_x3.py)
"""
import numpy as np
import pytest
import torch

from _net import fake_score, make_net, sampler_inputs
from _ops import max_rel, rel_l2
from oracle import psld_oracle as O
from oracle.weights import inpaint_draws, inpaint_inputs, prior
from psld_b200 import (EulerMaruyamaSampler, InpaintEulerMaruyamaSampler, PSLD, SSCSSampler, time_grid,
                       tiny_config)

pytestmark = pytest.mark.gpu

SAMPLERS = {"sscs_sde": SSCSSampler, "em_sde": EulerMaruyamaSampler}


def _golden_cfg(tag):
    kw = {
        "sscs_fake_uniform": (dict(sampler="sscs_sde", n_discrete_steps=50), {}),
        "em_fake_uniform": (dict(sampler="em_sde", n_discrete_steps=50), {}),
        "sscs_fake_quad": (dict(sampler="sscs_sde", n_discrete_steps=40, stride_type="quadratic"),
                           dict(nu=4.02, gamma=0.02, beta_min=0.5, beta_max=12.0)),
        "em_fake_quad": (dict(sampler="em_sde", n_discrete_steps=40, stride_type="quadratic"),
                         dict(nu=4.02, gamma=0.02, beta_min=0.5, beta_max=12.0)),
        "sscs_fake_nodenoise": (dict(sampler="sscs_sde", n_discrete_steps=30, denoise=False), {}),
    }[tag]
    cfg = tiny_config(**kw[0])
    cfg.model.sde.update(kw[1])
    cfg.data.image_size = 8
    return cfg


def _run(cfg, score_fn, u0, nb, state_dtype=torch.float64, fuse=False, record=True, merge=False,
         graph=False):
    kind = cfg.evaluation.sampler.name
    S = SAMPLERS[kind](cfg, PSLD(cfg), score_fn)
    S.use_graph = graph
    S.state_dtype = state_dtype
    S.fuse_halves = fuse
    S.merge_noise = merge
    S.noise = torch.stack(nb).cuda() if nb is not None else None
    S.record = True if record else None
    ts, n = time_grid(cfg)
    out = S.sample(u0.cuda(), ts.cuda(), n, denoise=cfg.evaluation.denoise, eps=cfg.evaluation.eval_eps)
    torch.cuda.synchronize()
    return out, (S.record if record else None), n


def _check_against_golden(g, out, rec, tol_l2, tol_max):
    ref = torch.from_numpy(g["final"])
    e_l2, e_mx = rel_l2(out, ref), max_rel(out, ref)
    worst = 0.0
    if rec is not None:
        for i in g["probe"]:
            s_ref = torch.from_numpy(g[f"state_{int(i)}"])
            worst = max(worst, max_rel(rec[int(i)][: s_ref.shape[0]], s_ref))
        st = g["stats"]
        sums = rec.double().reshape(rec.shape[0], -1)
        l2 = (sums ** 2).sum(1).cpu().numpy()
        worst = max(worst, float(np.max(np.abs(l2 - st[:, 3]) / st[:, 3])) / 2)
    print(f"final rel-L2 {e_l2:.3e} max-abs/max|ref| {e_mx:.3e} worst per-step {worst:.3e}")
    assert e_l2 <= tol_l2 and e_mx <= tol_max and worst <= tol_max, (e_l2, e_mx, worst)


@pytest.mark.parametrize("tag", ["sscs_fake_uniform", "em_fake_uniform", "sscs_fake_quad",
                                 "em_fake_quad", "sscs_fake_nodenoise"])
def test_sampler_algebra_vs_reference_golden(golden_dir, tag):
    """Fused update kernels + host schedule vs the reference sampler (generic score_fn path)."""
    g = np.load(f"{golden_dir}/sampler_{tag}.npz")
    cfg = _golden_cfg(tag)
    n = int(g["n"])
    u0, nb = sampler_inputs(cfg, int(g["B"]), n, cfg.evaluation.sampler.name)
    out, rec, n2 = _run(cfg, fake_score, u0, nb)
    assert n2 == n
    _check_against_golden(g, out, rec, 1e-6, 1e-6)
    # fused half-steps give the same trajectory end point
    out_f, _, _ = _run(cfg, fake_score, u0, nb, fuse=True, record=False)
    assert max_rel(out_f, out) <= 1e-6
    # fp32 state (throughput mode) stays within fp32 rounding accumulated over the steps
    out32, _, _ = _run(cfg, fake_score, u0, nb, state_dtype=torch.float32, fuse=True, record=False)
    assert rel_l2(out32, torch.from_numpy(g["final"])) <= 2e-5


@pytest.mark.parametrize("tag", ["sscs_fake_uniform", "em_fake_quad", "sscs_fake_nodenoise"])
def test_reference_style_loop_over_single_step_api(golden_dir, tag):
    """The reference's own ``sample()`` loop (sde.py:38-58, 350-370) written against the public
    ``predictor_update_fn(u, t, dt)`` / ``denoising_fn(x, t, dt)`` methods reproduces the reference
    trajectory (pre-drawn noise handed to each call)."""
    g = np.load(f"{golden_dir}/sampler_{tag}.npz")
    cfg = _golden_cfg(tag)
    kind = cfg.evaluation.sampler.name
    n = int(g["n"])
    u0, nb = sampler_inputs(cfg, int(g["B"]), n, kind)
    S = SAMPLERS[kind](cfg, PSLD(cfg), fake_score)
    ts, n2 = time_grid(cfg)
    assert n2 == n
    x = u0.cuda().double()
    for i in range(n):
        dt = ts[i + 1] - ts[i]
        if kind == "sscs_sde":
            x = S.predictor_update_fn(x, ts[i], dt, z=(nb[2 * i], nb[2 * i + 1]))
        else:
            x, x_mean = S.predictor_update_fn(x, ts[i], dt, z=nb[i])
            assert x_mean.shape == x.shape
        x, _ = S.corrector_update_fn(x, ts[i], dt)
        s_ref = g[f"state_{i}"] if f"state_{i}" in g.files else None
        if s_ref is not None:
            assert max_rel(x[: s_ref.shape[0]], torch.from_numpy(s_ref)) <= 1e-6
    if cfg.evaluation.denoise:
        e = cfg.evaluation.eval_eps
        x = S.denoising_fn(x, torch.tensor(1.0 - e), torch.tensor(e))
    torch.cuda.synchronize()
    ref = torch.from_numpy(g["final"])
    assert rel_l2(x, ref) <= 1e-6 and max_rel(x, ref) <= 1e-6
    # without pre-drawn noise the same call draws from Philox: finite, and new noise on every call
    a = S.predictor_update_fn(u0.cuda().double(), ts[0], ts[1] - ts[0])
    b = S.predictor_update_fn(u0.cuda().double(), ts[0], ts[1] - ts[0])
    a, b = (a[0], b[0]) if isinstance(a, tuple) else (a, b)
    assert torch.isfinite(a).all() and not torch.equal(a, b)


@pytest.mark.parametrize("kind,fname", [("em_sde", "sampler_tiny_em100.npz"),
                                        ("sscs_sde", "sampler_tiny_sscs100.npz")])
def test_native_sampler_vs_reference_golden(golden_dir, kind, fname):
    """BASELINE.json configs[0] (tiny NCSN++, 100 steps, 8 samples): whole native loop
    (psld_sampler_run: NCSN++ program + fused update per step) vs the reference."""
    g = np.load(f"{golden_dir}/{fname}")
    cfg = tiny_config(sampler=kind)
    net, _ = make_net(cfg, "fp32")
    n = int(g["n"])
    u0, nb = sampler_inputs(cfg, int(g["B"]), n, kind)
    out, rec, _ = _run(cfg, net, u0, nb)
    _check_against_golden(g, out, rec, 1e-5, 1e-5)
    # fused halves + fp32 state: same answer to fp32 accuracy
    out_f, _, _ = _run(cfg, net, u0, nb, state_dtype=torch.float32, fuse=True, record=False)
    assert rel_l2(out_f, torch.from_numpy(g["final"])) <= 5e-5
    # bf16 network path, stated separately
    net16, _ = make_net(cfg, "bf16")
    out16, _, _ = _run(cfg, net16, u0, nb, fuse=True, record=False)
    e16 = rel_l2(out16, torch.from_numpy(g["final"]))
    print(f"bf16 network path: final rel-L2 {e16:.3e}")
    assert e16 <= 6e-3


def test_native_equals_generic_path():
    """psld_sampler_run (native loop) and the Python loop over the same kernels agree exactly."""
    cfg = tiny_config(sampler="sscs_sde", n_discrete_steps=6)
    net, _ = make_net(cfg, "fp32")
    u0, nb = sampler_inputs(cfg, 2, 5, "sscs_sde")
    a, _, _ = _run(cfg, net, u0, nb, record=False)
    b, _, _ = _run(cfg, lambda u, t: net(u, t), u0, nb, record=False)
    assert max_rel(a, b) <= 1e-6     # only log(t) differs: host fp32 log vs device logf


def test_score_m_mode_vs_oracle():
    """gamma = 0 ablation (reference scripts_psld/ablations/.../sample_uncond_psld.sh:6-16):
    out_ch = 3, score only in momentum space (psld.py:240-243)."""
    cfg = tiny_config(sampler="sscs_sde", n_discrete_steps=12)
    cfg.model.sde.update(nu=4.0, gamma=0.0)
    cfg.data.image_size = 8

    def fake3(u, t):
        return fake_score(u, t)[:, 3:]

    u0, nb = sampler_inputs(cfg, 2, 11, "sscs_sde")
    out, _, n = _run(cfg, fake3, u0, nb, record=False)
    ts, _ = O.time_grid(cfg)
    ref = O.sscs_sample(cfg, fake3, u0, ts, n, nb)
    assert max_rel(out, ref) <= 1e-6


def test_philox_mode_runs_and_is_reproducible():
    cfg = tiny_config(sampler="sscs_sde", n_discrete_steps=8)
    net, _ = make_net(cfg, "bf16")
    u0, _ = sampler_inputs(cfg, 4, 7, "sscs_sde")
    a, _, _ = _run(cfg, net, u0, None, state_dtype=torch.float32, fuse=True, record=False)
    b, _, _ = _run(cfg, net, u0, None, state_dtype=torch.float32, fuse=True, record=False)
    assert torch.isfinite(a).all() and torch.equal(a, b)
    c, _, _ = _run(cfg, net, u0, None, state_dtype=torch.float32, fuse=False, record=False)
    assert max_rel(c, a) <= 1e-5     # fused and unfused draw the same Philox streams
    # merged draw (one Gaussian per fused pair of half-steps): reproducible, finite
    m1, _, _ = _run(cfg, net, u0, None, state_dtype=torch.float32, fuse=True, record=False, merge=True)
    m2, _, _ = _run(cfg, net, u0, None, state_dtype=torch.float32, fuse=True, record=False, merge=True)
    assert torch.isfinite(m1).all() and torch.equal(m1, m2)


def test_consecutive_sample_calls_draw_fresh_noise():
    """One sampler instance serves every dataloader batch of a run (reference wrapper.py:101-122):
    each sample() call must inject different noise (the reference's torch generator advances), while
    a given (seed, rank, call index) stays reproducible."""
    cfg = tiny_config(sampler="sscs_sde", n_discrete_steps=6)
    net, _ = make_net(cfg, "bf16")
    u0, _ = sampler_inputs(cfg, 4, 5, "sscs_sde")
    ts, n = time_grid(cfg)
    for kind in ("sscs_sde", "em_sde"):
        S = SAMPLERS[kind](cfg, PSLD(cfg), net)
        S.state_dtype = torch.float32
        outs = [S.sample(u0.cuda(), ts.cuda(), n).clone() for _ in range(3)]
        assert S.calls == 3
        for i in range(3):
            for j in range(i + 1, 3):
                d = (outs[i] - outs[j]).abs().max().item()
                assert d > 1e-3, (kind, i, j, d)
        S2 = SAMPLERS[kind](cfg, PSLD(cfg), net)
        S2.state_dtype = torch.float32
        S2.calls = 2
        assert torch.equal(S2.sample(u0.cuda(), ts.cuda(), n), outs[2])


def test_merged_noise_is_exact_in_law():
    """Merging half B of step i with half A of step i+1 into one draw keeps the law of the chain:
    with a zero score network the end state is Gaussian with a known 2x2 covariance per pair."""
    cfg = tiny_config(sampler="sscs_sde", n_discrete_steps=6, denoise=False)
    cfg.data.image_size = 64
    zero = lambda u, t: torch.zeros_like(u)
    B = 16
    u0 = torch.zeros(B, 6, 64, 64)
    outs = {}
    for merge in (False, True):
        out, _, _ = _run(cfg, zero, u0, None, fuse=True, record=False, merge=merge)
        x, m = torch.chunk(out.double().cpu(), 2, 1)
        outs[merge] = (float(x.var()), float((x * m).mean()), float(m.var()))
    n = B * 3 * 64 * 64
    for a, b in zip(outs[False], outs[True]):
        assert abs(a - b) <= 6 * max(abs(a), 1e-3) / np.sqrt(n) * 2 + 1e-6, (outs)


@pytest.mark.parametrize("kind", ["sscs_sde", "em_sde"])
@pytest.mark.parametrize("fuse,merge", [(False, False), (True, False), (True, True)])
def test_cuda_graph_replay_equals_host_loop(kind, fuse, merge):
    """One captured predictor step replayed n times (device-side step counter + coefficient table)
    gives bit-identical states to launching every kernel from the host."""
    cfg = tiny_config(sampler=kind, n_discrete_steps=9)
    net, _ = make_net(cfg, "bf16")
    u0, _ = sampler_inputs(cfg, 3, 8, kind)
    for sd in (torch.float32, torch.float64):
        a, _, _ = _run(cfg, net, u0, None, state_dtype=sd, fuse=fuse, record=False, merge=merge, graph=False)
        b, _, _ = _run(cfg, net, u0, None, state_dtype=sd, fuse=fuse, record=False, merge=merge, graph=True)
        assert torch.isfinite(a).all() and torch.equal(a, b)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("B,H", [(7, 32), (256, 32), (64, 64), (32, 256)])
def test_image_quantisation_bit_exact(dtype, B, H):
    """Fused writer arithmetic (drop momentum, x*0.5+0.5, *255, clip, truncate) == the reference's
    numpy sequence, bit for bit (integer output), at the benchmark's batches and past the grid cap."""
    from psld_b200 import samples_to_uint8
    g = torch.Generator().manual_seed(5)
    st = (torch.randn(B, 6, H, H, generator=g, dtype=torch.float64) * 1.3).to(dtype)
    st[0, 0, 0, :4] = torch.tensor([-1.0, 1.0, 0.0, 0.999999], dtype=dtype)   # edges of the range
    st[-1, 2, -1, -4:] = torch.tensor([-1.0, 1.0, 0.0, 0.999999], dtype=dtype)
    got = samples_to_uint8(st.cuda()).cpu().numpy()
    ref = O.images_uint8(st)
    assert got.shape == ref.shape == (B, H, H, 3) and got.dtype == ref.dtype
    assert (got == ref).all()


def _inpaint_cfg(mode):
    cfg = tiny_config(sampler="ip_em_sde", n_discrete_steps=30)
    cfg.training.mode = mode
    cfg.data.image_size = 8
    return cfg


@pytest.mark.parametrize("mode", ["hsm", "dsm"])
def test_inpaint_sampler_vs_reference_golden(golden_dir, mode):
    """ip_em_sde (reference sde.py:125-224): EM predictor + fused Split-Perturb-Combine kernel vs the
    reference's own output on the same draws."""
    g = np.load(f"{golden_dir}/sampler_ip_em_fake_{mode}.npz")
    cfg = _inpaint_cfg(mode)
    n, B = int(g["n"]), int(g["B"])
    sde = PSLD(cfg)
    ts, n2 = time_grid(cfg)
    assert n2 == n
    x_0, mask = inpaint_inputs(B, 8, 3)
    S = InpaintEulerMaruyamaSampler(cfg, sde, fake_score)
    S.state_dtype = torch.float64
    S.prior = prior((B, 3, 8, 8), float(np.sqrt(sde.m)), 1)
    S.noise = inpaint_draws(n, B, 8, 2)
    out = S.sample((x_0.cuda(), mask.cuda()), ts, n, denoise=cfg.evaluation.denoise,
                   eps=cfg.evaluation.eval_eps).cpu()
    ref = torch.from_numpy(g["final"])
    e = max_rel(out, ref)
    print(f"ip_em_sde {mode}: max-abs/max|ref| {e:.3e}")
    assert e <= 1e-6
    # fp32 state
    S.state_dtype = torch.float32
    out32 = S.sample((x_0.cuda(), mask.cuda()), ts, n, denoise=cfg.evaluation.denoise,
                     eps=cfg.evaluation.eval_eps).cpu()
    assert rel_l2(out32, ref) <= 2e-5


@pytest.mark.parametrize("tag,kw", [("uniform", {}), ("quad_nodenoise", dict(stride_type="quadratic", denoise=False))])
def test_class_conditional_sampler_vs_reference_golden(golden_dir, tag, kw):
    """cc_em_sde (sde.py:61-122): guided drift + EM update in one fused pass, classifier gradient by
    autograd through the caller's classifier, vs the reference's own output; then Philox noise."""
    from _net import cc_config
    from oracle.weights import fake_classifier
    from psld_b200 import ClassCondEulerMaruyamaSampler
    g = np.load(f"{golden_dir}/sampler_cc_em_fake_{tag}.npz")
    cfg = cc_config(**kw)
    ts, n = time_grid(cfg)
    assert n == int(g["n"])
    B = int(g["B"])
    u0, nb = sampler_inputs(cfg, B, n, "em_sde")
    S = ClassCondEulerMaruyamaSampler(cfg, PSLD(cfg), fake_score, fake_classifier)
    S.state_dtype = torch.float64
    S.noise = torch.stack(nb)
    out = S.sample(u0.cuda(), ts.cuda(), n, denoise=cfg.evaluation.denoise, eps=cfg.evaluation.eval_eps)
    torch.cuda.synchronize()
    ref = torch.from_numpy(g["final"])
    e, m = rel_l2(out, ref), max_rel(out, ref)
    print(f"cc_em_sde {tag}: rel-L2 {e:.3e} max-abs/max|ref| {m:.3e}")
    assert e <= 1e-6 and m <= 1e-6
    S.noise = None
    a = S.sample(u0.cuda(), ts.cuda(), n)
    assert torch.isfinite(a).all()
    with torch.inference_mode():          # Lightning's predict loop runs under inference_mode
        b = S.sample(u0.cuda(), ts.cuda(), n)
    assert torch.isfinite(b).all()


@pytest.mark.parametrize("tag,tol,den", [("tol1e-5", 1e-5, True), ("tol1e-4_nodenoise", 1e-4, False)])
def test_bb_ode_sampler_vs_reference_golden(golden_dir, tag, tol, den):
    """bb_ode (ode.py:41-76): the RK45 driver restated on the device (stages, error norm and step
    control of scipy's solve_ivp) reproduces the reference's sample AND its number of score_fn calls."""
    from _net import ode_config
    from psld_b200 import BBODESampler
    g = np.load(f"{golden_dir}/sampler_bb_ode_gauss_{tag}.npz")
    cfg = ode_config(tol, denoise=den)
    B = int(g["B"])
    u0 = prior((B, 3, 8, 8), 0.5, 1)
    from oracle.weights import gaussian_score_fn
    S = BBODESampler(cfg, PSLD(cfg), gaussian_score_fn(cfg))
    out = S.sample(u0.cuda(), None, 0, denoise=den, eps=cfg.evaluation.eval_eps)
    torch.cuda.synchronize()
    ref = torch.from_numpy(g["final"])
    e, m = rel_l2(out, ref), max_rel(out, ref)
    print(f"bb_ode {tag}: rel-L2 {e:.3e} max {m:.3e} nfe {S.nfe} (reference {int(g['nfe'])}), "
          f"steps {S.steps_accepted}+{S.steps_rejected} rejected")
    assert S.nfe == int(g["nfe"]) and S.mean_nfe == S.nfe and S.n_steps == S.nfe
    assert e <= 1e-5 and m <= 1e-5
    assert out.dtype == (torch.float64 if den else torch.float32)


@pytest.mark.parametrize("tag,tol,den,dt", [("tol1e-5", 1e-5, True, torch.float32),
                                            ("tol1e-4_f64_nodenoise", 1e-4, False, torch.float64)])
def test_bb_ode_vp_sampler_vs_reference_golden(golden_dir, tag, tol, den, dt):
    """bb_ode over the VP-SDE baseline (scripts_psld/ablations/uncond/cifar10/sample_uncond_vpsde_ode.sh): the
    device RK45 driver + psld_vp_reverse_drift vs the reference's BBODESampler + VPSDE (same NFE count)."""
    from _net import vp_config
    from oracle.weights import vp_gaussian_score_fn
    from psld_b200 import BBODESampler, VPSDE
    g = np.load(f"{golden_dir}/sampler_bb_ode_vp_gauss_{tag}.npz")
    cfg = vp_config(sampler=dict(name="bb_ode", solver="RK45", rtol=tol, atol=tol), denoise=den)
    B = int(g["B"])
    x0 = prior((B, 3, 8, 8), 1.0, 1)[:, :3].contiguous().to(dt)
    S = BBODESampler(cfg, VPSDE(cfg), vp_gaussian_score_fn(cfg))
    out = S.sample(x0.cuda(), None, 0, denoise=den, eps=cfg.evaluation.eval_eps)
    torch.cuda.synchronize()
    ref = torch.from_numpy(g["final"])
    e, m = rel_l2(out, ref), max_rel(out, ref)
    print(f"bb_ode VP {tag}: rel-L2 {e:.3e} max {m:.3e} nfe {S.nfe} (reference {int(g['nfe'])})")
    assert S.nfe == int(g["nfe"]) and tuple(out.shape) == (B, 3, 8, 8)
    assert e <= 1e-5 and m <= 1e-5


def test_bb_ode_vp_with_network_vs_oracle():
    """bb_ode + VP-SDE over the native NCSN++ program (in_ch = out_ch = 3, fp32 tier) vs the oracle."""
    from _net import vp_config
    from psld_b200 import BBODESampler, VPSDE
    cfg = vp_config(sampler=dict(name="bb_ode", solver="RK45", rtol=1e-3, atol=1e-3))
    cfg.data.image_size = 32
    net, sd = make_net(cfg, "fp32")
    x0 = prior((2, 3, 32, 32), 1.0, 1)[:, :3].contiguous()
    S = BBODESampler(cfg, VPSDE(cfg), net)
    out = S.sample(x0.cuda(), None, 0, denoise=True, eps=1e-3)
    ref, nfe = O.bb_ode_sample(cfg, O.OracleScoreFn(cfg, sd), x0, 1e-3, 1e-3, denoise=True, eps=1e-3)
    e = rel_l2(out, ref)
    print(f"bb_ode VP + NCSN++ fp32: rel-L2 {e:.3e}, nfe {S.nfe} vs oracle {nfe}")
    assert S.nfe == nfe and e <= 1e-4


def test_bb_ode_with_network_vs_oracle():
    """bb_ode over the native NCSN++ program (tiny net, fp32 tier) vs the oracle's solve_ivp run."""
    from _net import ode_config
    from psld_b200 import BBODESampler
    cfg = ode_config(1e-3)
    cfg.data.image_size = 32
    net, sd = make_net(cfg, "fp32")
    B = 2
    u0 = prior((B, 3, 32, 32), 0.5, 1)
    S = BBODESampler(cfg, PSLD(cfg), net)
    out = S.sample(u0.cuda(), None, 0, denoise=True, eps=1e-3)
    ref, nfe = O.bb_ode_sample(cfg, O.OracleScoreFn(cfg, sd), u0, 1e-3, 1e-3, denoise=True, eps=1e-3)
    e = rel_l2(out, ref)
    print(f"bb_ode + NCSN++ fp32: rel-L2 {e:.3e}, nfe {S.nfe} vs oracle {nfe}")
    assert S.nfe == nfe and e <= 1e-4


def test_inpaint_sampler_philox_keeps_known_region():
    """Device-drawn prior and noise: reproducible, and the known region of the denoised result is
    the perturbation mean of x_0 (HSM), i.e. x_0 scaled by the mean coefficient at tau = eps."""
    cfg = _inpaint_cfg("hsm")
    sde = PSLD(cfg)
    ts, n = time_grid(cfg)
    x_0, mask = inpaint_inputs(4, 8, 5)
    S = InpaintEulerMaruyamaSampler(cfg, sde, fake_score)
    a = S.sample((x_0.cuda(), mask.cuda()), ts, n).cpu()
    c = S.sample((x_0.cuda(), mask.cuda()), ts, n).cpu()      # next call: fresh prior and noise
    S.calls = 0
    b = S.sample((x_0.cuda(), mask.cuda()), ts, n).cpu()      # same (seed, rank, call) -> same draws
    assert torch.equal(a, b) and torch.isfinite(a).all() and not torch.equal(a, c)
    s = O.PSLDScalars(cfg)
    axx = O.mean_coeffs(s, float(np.float32(1.0) - np.float32(1.0 - cfg.evaluation.eval_eps)))[0]
    known = mask == 1
    assert torch.allclose(a[:, :3][known], (axx * x_0.double())[known], rtol=1e-12, atol=1e-13)
    free = ~known
    assert (a[:, :3][free] - (axx * x_0.double())[free]).abs().max() > 1e-3


@pytest.mark.parametrize("tag,kw", [("uniform", {}), ("quad", dict(stride_type="quadratic"))])
def test_vp_sampler_vs_reference_golden(golden_dir, tag, kw):
    """The reference's em_sde also drives the VP-SDE baseline (sample_uncond_vpsde.sh): fused
    psld_vp_em_update + host schedule vs the reference's own output."""
    from _net import vp_config
    from oracle.weights import noise_bank
    from psld_b200 import VPSDE
    g = np.load(f"{golden_dir}/sampler_vp_em_fake_{tag}.npz")
    cfg = vp_config(**kw)
    ts, n = time_grid(cfg)
    B = int(g["B"])
    S = EulerMaruyamaSampler(cfg, VPSDE(cfg), fake_score)
    S.state_dtype = torch.float64
    S.noise = torch.stack(noise_bank(n, (B, 3, 8, 8), 2))
    x0 = noise_bank(1, (B, 3, 8, 8), 1)[0]
    out = S.sample(x0.cuda(), ts, n, denoise=cfg.evaluation.denoise, eps=cfg.evaluation.eval_eps).cpu()
    ref = torch.from_numpy(g["final"])
    e = max_rel(out, ref)
    print(f"vp em_sde {tag}: max-abs/max|ref| {e:.3e}")
    assert e <= 1e-6
    with pytest.raises(ValueError):
        SSCSSampler(cfg, VPSDE(cfg), fake_score)


def test_vp_sampler_with_network_vs_oracle():
    """VP-SDE + NCSN++ (in_ch = out_ch = 3) through the program path vs the CPU oracle."""
    from _net import vp_config
    from oracle.weights import noise_bank
    from psld_b200 import VPSDE
    cfg = vp_config(n_discrete_steps=12)
    cfg.data.image_size = 32
    net, sd = make_net(cfg, "fp32")
    ts, n = time_grid(cfg)
    B = 2
    nb = noise_bank(n, (B, 3, 32, 32), 2)
    x0 = noise_bank(1, (B, 3, 32, 32), 1)[0]
    S = EulerMaruyamaSampler(cfg, VPSDE(cfg), net)
    S.state_dtype = torch.float64
    S.noise = torch.stack(nb)
    out = S.sample(x0.cuda(), ts, n).cpu()
    ref = O.vp_em_sample(cfg, lambda u, t: O.ncsnpp_forward(cfg, sd, u, t), x0, ts, n, nb)
    e = rel_l2(out, ref)
    print(f"vp em_sde + NCSN++ fp32: rel-L2 {e:.3e}")
    assert e <= 1e-5
    # Philox noise: reproducible and finite
    S.noise = None
    a, c = S.sample(x0.cuda(), ts, n), S.sample(x0.cuda(), ts, n)
    S.calls -= 2
    b = S.sample(x0.cuda(), ts, n)
    assert torch.equal(a, b) and torch.isfinite(a).all() and not torch.equal(a, c)


def test_native_sampler_celeba64_vs_oracle():
    """BASELINE configs[3] network (CelebA-64 NCSN++: 64x64, ch_mult [1,2,2,2], nu/gamma = 4.005/0.005)
    through the whole native SSCS loop for a few steps vs the CPU oracle (fp32 path), plus the bf16
    tensor-core plan on the same inputs."""
    from psld_b200 import celeba64_config
    cfg = celeba64_config(n_discrete_steps=4)
    cfg.model.score_fn.init_scale = 1.0
    net, sd = make_net(cfg, "fp32")
    n, B = 3, 2
    u0, nb = sampler_inputs(cfg, B, n, "sscs_sde")
    out, _, n2 = _run(cfg, net, u0, nb, record=False)
    assert n2 == n
    ref = O.sscs_sample(cfg, O.OracleScoreFn(cfg, sd), u0, O.time_grid(cfg)[0], n, nb)
    e = rel_l2(out, ref)
    net16, _ = make_net(cfg, "bf16")
    out16, _, _ = _run(cfg, net16, u0, nb, fuse=True, record=False)
    e16 = rel_l2(out16, ref)
    print(f"celeba64 SSCS {n}+1 NFE: fp32 path rel-L2 {e:.3e}, bf16 path {e16:.3e}")
    assert e <= 1e-5 and e16 <= 1.4e-2
