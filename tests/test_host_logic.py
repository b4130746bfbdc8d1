"""CPU: host-side logic of the product (schedule tables, registry, program builder) and the
C-ABI library surface.  No kernel is launched here."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from emulate import run_plan
from oracle import psld_oracle as O
from oracle.weights import fill_state_dict
from psld_b200 import (NCSNpp, PSLD, PSLDSchedule, SSCSSampler, StepTables, get_module, mid_config,
                       register_module, time_grid, tiny_config)
from psld_b200 import _lib as L
from psld_b200.program import build_plan

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "psld_b200.h")).read()
    declared = set(re.findall(r"PSLD_API\s+(?:const\s+)?\w+\*?\s+(psld_\w+)\s*\(", hdr))
    assert declared == set(L.EXPORTS.keys()), declared ^ set(L.EXPORTS.keys())
    lib = L.lib()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.psld_version() == L.VERSION
    # struct sizes agree with the header's layout rules
    assert C.sizeof(L.HalfStep) == 64 and C.sizeof(L.ScoreStep) == 112
    assert C.sizeof(L.SscsCoeffs) == 3 * 64 + 112
    assert C.sizeof(L.Op) == 8 + 4 * L.OP_NI + 4 * L.OP_NF + 8 * 2 * L.OP_NP + 8


def test_schedule_tables_vs_golden(golden_dir):
    g = np.load(f"{golden_dir}/scalars.npz")
    cols = {c: i for i, c in enumerate(g["columns"])}
    for row in g["table"]:
        v = lambda k: row[cols[k]]
        cfg = tiny_config()
        cfg.model.sde.update(nu=v("nu"), gamma=v("gamma"), beta_min=v("beta0"), beta_max=v("beta1"),
                             decomp_mode="upper" if v("upper") else "lower")
        sch = PSLDSchedule(cfg)
        ts = torch.tensor([v("t"), v("t") + v("dt")], dtype=torch.float64)
        tab = StepTables(sch, ts, 1, "sscs_sde", False, 1e-3)
        h = tab.sscs[0].half_a
        np.testing.assert_allclose([h.a_xx, h.a_xm, h.a_mx, h.a_mm],
                                   [v("a_xx"), v("a_xm"), v("a_mx"), v("a_mm")], rtol=1e-14, atol=1e-17)
        np.testing.assert_allclose([h.c11, h.c12, h.c21, h.c22],
                                   [v("c11"), v("c12"), v("c21"), v("c22")], rtol=1e-12, atol=1e-17)
        s = tab.sscs[0].score
        f32 = lambda k: float(np.float32(v(k)))
        assert [s.li11, s.li12, s.li21, s.li22] == [f32("i11"), f32("i12"), f32("i21"), f32("i22")]
        np.testing.assert_allclose(s.k_x, v("dt") * v("gamma") * v("beta_tau"), rtol=1e-11)
        np.testing.assert_allclose(s.k_m, v("dt") * v("m") * v("nu") * v("beta_tau"), rtol=1e-11)
        assert s.mode == (1 if v("gamma") == 0 and not v("upper") else 0)


def test_time_grid_and_denoise_rounding():
    for stride in ("uniform", "quadratic"):
        cfg = tiny_config(stride_type=stride, n_discrete_steps=37)
        ts, n = time_grid(cfg)
        ts2, n2 = O.time_grid(cfg)
        assert n == n2 == 36
        np.testing.assert_allclose(ts.numpy(), ts2, atol=3e-16)
    tab = StepTables(PSLDSchedule(cfg), ts, n, "em_sde", True, 1e-3)
    # the reference's denoise step runs at t = fl32(T - eps) with dt = fl32(eps) (sde.py:52-57)
    assert tab.den.dt == float(np.float32(1e-3))
    assert tab.n_calls == n + 1
    assert abs(float(tab.tau32[-1]) - (1.0 - float(np.float32(0.999)))) < 1e-9


def test_nan_guard_raises_like_reference():
    cfg = tiny_config()
    cfg.model.sde.numerical_eps = -1.0       # forces sqrt of a negative variance
    with pytest.raises(ValueError, match="Numerical precision error"):
        StepTables(PSLDSchedule(cfg), torch.linspace(0, 0.999, 5, dtype=torch.float64), 4,
                   "sscs_sde", True, 1e-3)


def test_registry_semantics():
    assert get_module("samplers", "sscs_sde_b200") is SSCSSampler
    assert get_module("score_fn", "ncsnpp_b200") is NCSNpp
    assert get_module("sde", "psld_b200") is PSLD
    with pytest.raises(ValueError):
        get_module("samplers", "nope")
    with pytest.raises(ValueError):
        register_module(category="samplers", name="sscs_sde_b200")(SSCSSampler)


def test_sde_object_surface():
    sde = PSLD(tiny_config())
    assert sde.T == 1.0 and sde.mode == "score_xm" and sde.type == "psld-score_xm"
    assert sde.m_inv == 4.0 and sde.m == 0.25
    u = sde.prior_sampling([4, 3, 8, 8])
    assert tuple(u.shape) == (4, 6, 8, 8)
    assert float(sde.beta_t(0.3)) == 8.0 and float(sde.b_t(0.5)) == 4.0


@pytest.mark.parametrize("cfg_fn,precision,tol", [(tiny_config, "fp32", 1e-5), (mid_config, "fp32", 1e-5),
                                                  (mid_config, "bf16", 3e-2)])
def test_program_builder_vs_golden(golden_dir, cfg_fn, precision, tol):
    """The op program (weights packing, wiring, fused epilogues, temb offsets) interpreted on the
    host reproduces the reference forward."""
    cfg = cfg_fn()
    name = "tiny" if cfg_fn is tiny_config else "mid"
    g = np.load(f"{golden_dir}/forward_{name}.npz")
    net = NCSNpp(cfg).eval()
    net.precision = precision
    net.load_state_dict(fill_state_dict({k: tuple(v.shape) for k, v in net.state_dict().items()}, 0))
    x, t, y = (torch.from_numpy(g[k]) for k in ("x", "t", "y"))
    plan = build_plan(net, x.shape[0], x.shape[0], False, dry=True)
    out = run_plan(plan, x, t)
    assert float((out - y).norm() / y.norm()) <= tol
    assert plan.launches == L.lib().psld_program_launches(plan.op_array, plan.n_ops) > plan.n_ops
    if precision == "bf16":
        assert plan.engine_count["tc"] + plan.engine_count.get("tc_gn", 0) >= 35
        assert plan.engine_count["simt"] <= 3


def test_no_cpu_fallback():
    net = NCSNpp(tiny_config())
    with pytest.raises(RuntimeError, match="CUDA"):
        net(torch.zeros(1, 6, 32, 32), torch.ones(1))
    with pytest.raises(RuntimeError, match="no CPU path"):
        build_plan(net, 1, 1, False)


def test_checkpoint_loader(tmp_path):
    """Lightning-style checkpoint (prefixes score_fn./ema_score_fn.) -> NCSNpp, strict."""
    from psld_b200 import load_checkpoint, select_score_fn_state
    cfg = tiny_config()
    src = NCSNpp(cfg)
    sd = fill_state_dict({k: tuple(v.shape) for k, v in src.state_dict().items()}, 4)
    ema = {k: v + 1.0 for k, v in sd.items()}
    ck = {"state_dict": {**{"score_fn." + k: v for k, v in sd.items()},
                         **{"ema_score_fn." + k: v for k, v in ema.items()}}, "epoch": 3}
    path = tmp_path / "psld.ckpt"
    torch.save(ck, path)
    a = load_checkpoint(NCSNpp(cfg), str(path), sample_from="target")
    b = load_checkpoint(NCSNpp(cfg), str(path), sample_from="source")
    k0 = "all_modules.3.weight"
    assert torch.equal(a.state_dict()[k0], ema[k0]) and torch.equal(b.state_dict()[k0], sd[k0])
    with pytest.raises(KeyError):
        select_score_fn_state({"foo.x": torch.zeros(1)}, "target")


class _Hparams:          # what Lightning's save_hyperparameters can leave in a .ckpt
    pass


def test_checkpoint_loader_refuses_untrusted_pickles(tmp_path):
    """Tensors-only checkpoints load with weights_only=True; one that pickles an arbitrary object
    is refused unless the caller passes trust=True."""
    from psld_b200 import load_checkpoint
    cfg = tiny_config()
    sd = fill_state_dict({k: tuple(v.shape) for k, v in NCSNpp(cfg).state_dict().items()}, 2)

    path = tmp_path / "lightning_like.ckpt"
    torch.save({"state_dict": {"ema_score_fn." + k: v for k, v in sd.items()}, "hyper_parameters": _Hparams()},
               path)
    with pytest.raises(RuntimeError, match="trust=True"):
        load_checkpoint(NCSNpp(cfg), str(path))
    net = load_checkpoint(NCSNpp(cfg), str(path), trust=True)
    assert torch.equal(net.state_dict()["all_modules.3.weight"], sd["all_modules.3.weight"])


@pytest.mark.parametrize("name", ["tiny", "cifar10", "celeba64"])
def test_state_dict_contract_vs_reference(golden_dir, name):
    """Checkpoint contract (wrapper.py:30-31, sample.py:62-69): same tensor names, shapes and ORDER as
    the reference module for the shipped architectures (749 tensors for CIFAR-10, 571 for CelebA-64;
    fixture written from the reference's own modules by oracle/make_golden.py)."""
    import json
    from psld_b200 import celeba64_config, cifar10_config
    want = json.load(open(f"{golden_dir}/state_dict_contract.json"))[name]
    cfg = {"tiny": tiny_config, "cifar10": cifar10_config, "celeba64": celeba64_config}[name]()
    got = {k: list(v.shape) for k, v in NCSNpp(cfg).state_dict().items()}
    assert list(got.keys()) == list(want.keys())
    assert got == want


def test_inpaint_and_vp_tables_vs_oracle():
    """Host coefficient tables of the two widened samplers against the oracle's scalar algebra
    (which is pinned on the reference's outputs in test_oracle_vs_golden.py)."""
    from _net import vp_config
    from psld_b200.schedule import InpaintTables, VPSchedule, VPStepTables
    # inpainting: call 0 = T, calls 1..n = T - ts[i], call n+1 = T - fl32(T - eps), mean only
    for mode in ("hsm", "dsm"):
        cfg = tiny_config(sampler="ip_em_sde", n_discrete_steps=12)
        cfg.training.mode = mode
        sch, s = PSLDSchedule(cfg), O.PSLDScalars(cfg)
        ts, n = time_grid(cfg)
        tab = InpaintTables(sch, ts, n, True, cfg.evaluation.eval_eps, mode == "hsm")
        taus = [1.0] + [1.0 - float(t) for t in ts[:n]] + \
               [float(np.float32(1.0) - np.float32(1.0 - cfg.evaluation.eval_eps))]
        assert len(tab.steps) == n + 2
        for k, tau in enumerate(taus):
            st = tab.steps[k]
            np.testing.assert_allclose([st.a_xx, st.a_xm, st.a_mx, st.a_mm], O.mean_coeffs(s, tau), rtol=1e-13)
            cov = s.cov(0.0, s.mm_0 if mode == "hsm" else 0.0, tau)
            np.testing.assert_allclose([st.c11, st.c12, st.c21, st.c22], s.get_coeff(cov), rtol=1e-10,
                                       atol=1e-16)
            assert st.m0_std == (0.0 if mode == "hsm" else s.mm_0 ** 0.5)
            assert st.mean_only == int(k == n + 1)
    # VP-SDE Euler-Maruyama rows
    cfg = vp_config(n_discrete_steps=9, stride_type="quadratic")
    v, sch = O.VPScalars(cfg), VPSchedule(cfg)
    ts, n = time_grid(cfg)
    tab = VPStepTables(sch, ts, n, True, cfg.evaluation.eval_eps)
    for i in range(n):
        tau, dt = 1.0 - float(ts[i]), float(ts[i + 1] - ts[i])
        st = tab.steps[i]
        beta = v.beta_t(tau)
        np.testing.assert_allclose([st.half_beta, st.g2, st.neg_inv_std, st.dt, st.gs],
                                   [0.5 * beta, beta, -1.0 / v.std(tau), dt, (beta * dt) ** 0.5], rtol=1e-12)
    den = tab.steps[n]
    assert den.gs == 0.0 and den.dt == float(np.float32(cfg.evaluation.eval_eps))
    assert tab.tau32.numel() == n + 1


def test_call_seed_per_call_and_rank(monkeypatch):
    """Philox key derivation (psld_b200/distributed.py): call 0 keeps the reference's seed + rank
    (wrapper.py:93-99); later calls and other ranks get distinct 64-bit keys; the rank is resolved
    at call time from RANK, else NODE_RANK/LOCAL_RANK (Lightning's launcher does not export RANK)."""
    from psld_b200.distributed import call_seed, current_rank
    assert call_seed(7, 0, 0) == 7 and call_seed(7, 3, 0) == 10
    keys = {call_seed(7, r, c) for r in range(8) for c in range(64)}
    assert len(keys) == 8 * 64 and all(0 <= k < 2 ** 64 for k in keys)
    assert call_seed(7, 1, 5) == call_seed(7, 1, 5)
    for k in ("RANK", "LOCAL_RANK", "NODE_RANK", "GROUP_RANK", "LOCAL_WORLD_SIZE"):
        monkeypatch.delenv(k, raising=False)
    assert current_rank() == 0
    monkeypatch.setenv("LOCAL_RANK", "3")
    assert current_rank() == 3
    monkeypatch.setenv("NODE_RANK", "1")
    monkeypatch.setenv("LOCAL_WORLD_SIZE", "8")
    assert current_rank() == 11
    monkeypatch.setenv("RANK", "5")
    assert current_rank() == 5


def test_guided_program_vs_golden(golden_dir):
    """Classifier-free guidance (BASELINE configs[4]): the ONE program the guided score_fn compiles to
    ([cond | copy | uncond | axpby]) interpreted on the host reproduces the composition of two reference
    forwards; w = 0 returns the conditional network's output exactly; plans follow weight updates."""
    from psld_b200 import ClassifierFreeGuidance
    g = np.load(f"{golden_dir}/forward_cfg_mid.npz")
    cfg = mid_config()
    nets = []
    for seed in g["seeds"]:
        net = NCSNpp(cfg).eval()
        net.precision = "fp32"
        net.load_state_dict(fill_state_dict({k: tuple(v.shape) for k, v in net.state_dict().items()}, int(seed)))
        nets.append(net)
    x, t, y, yc = (torch.from_numpy(g[k]) for k in ("x", "t", "y", "y_cond"))
    from psld_b200.guidance import GuidedPlan
    a, b = (build_plan(n, 2, 2, False, dry=True) for n in nets)
    gp = GuidedPlan(a, b, float(g["weight"]))
    assert gp.n_ops == a.n_ops + b.n_ops + 2 and gp.launches == a.launches + b.launches + 2
    assert sum(op.kind == L.OP_TEMB for op in gp.ops) == 2 and gp.ops[gp.temb_op].kind == L.OP_TEMB
    assert all(op.inp[0] == a.time_buf.data_ptr() for op in gp.ops if op.kind == L.OP_TEMB)
    out = run_plan(gp, x, t)
    assert float((out - y).norm() / y.norm()) <= 1e-5
    out0 = run_plan(GuidedPlan(a, b, 0.0), x, t)
    assert torch.equal(out0, run_plan(a, x, t)) and float((out0 - yc).norm() / yc.norm()) <= 1e-5
    # module surface: registry name, cls(config) construction, state-dict prefixes, shape checks
    cls = get_module("score_fn", "cfg_ncsnpp_b200")
    assert cls is ClassifierFreeGuidance
    c2 = tiny_config()
    c2.model.score_fn["guidance_weight"] = 2.0
    m = cls(c2)
    assert m.weight == 2.0 and m.in_ch == 6
    keys = list(m.state_dict().keys())
    assert keys[0].startswith("cond.all_modules.") and keys[-1].startswith("uncond.all_modules.")
    assert len(keys) == 2 * len(NCSNpp(c2).state_dict())
    import copy
    m2 = copy.deepcopy(m)                       # main/eval/sample.py deep-copies the score_fn
    assert m2.weight == 2.0 and m2.cond is not m.cond and list(m2.state_dict().keys()) == keys
    m2.load_state_dict(m.state_dict())
    with pytest.raises(ValueError):
        ClassifierFreeGuidance(cond=nets[0], uncond=nets[0], weight=1.0)
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.zeros(1, 6, 32, 32), torch.ones(1))


# ------------------------------------------------------------------ in-kernel noise: host reference
@pytest.mark.parametrize("counter,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
    ((6, 0, 3, 0), (7, 0), (0x548d6e57, 0xd5e0b3d0, 0x332db457, 0x95ca6e68)),   # index 6, stream 3, seed 7
])
def test_philox_host_reference_known_answers(counter, key, want):
    """tests/_philox.py is Philox4x32-10: the Random123 / cuRAND known-answer vectors, and the
    (seed, stream, index) -> (key, counter) packing of the device's Philox::draw."""
    import _philox as P
    assert tuple(int(w) for w in P.philox4x32_10(counter, key)) == want
    idx = (counter[1] << 32) | counter[0]
    stream = (counter[3] << 32) | counter[2]
    seed = (key[1] << 32) | key[0]
    assert tuple(int(w) for w in P.draw(seed, stream, idx)) == want


def test_philox_host_index_rules():
    """The whole-tensor and single-pair forms of each index rule agree, and the rules keep the x and
    m halves, the SSCS stages and the inpainting draws on distinct (stream, index) pairs."""
    import _philox as P
    from psld_b200.distributed import call_seed
    seed, B, chw = call_seed(7, 1, 3), 3, 20
    assert seed >> 32                                      # the high key word is exercised
    zx, zm = P.pair_normals(seed, P.sscs_stream(70001, "b"), B, chw)
    b, j = np.meshgrid(np.arange(B), np.arange(chw), indexing="ij")
    ax, am = P.pair_normals_at(seed, P.sscs_stream(70001, "b"), b, j, chw)
    assert np.array_equal(zx, ax) and np.array_equal(zm, am)
    # x of vector v is draw 2v, m is draw 2v + 1
    assert np.array_equal(zx[1, 8:12], P.normal4(seed, 2 * 70001 + 1, 2 * (chw // 4 + 2)))
    assert np.array_equal(zm[1, 8:12], P.normal4(seed, 2 * 70001 + 1, 2 * (chw // 4 + 2) + 1))
    assert P.sscs_stream(5, "a") == 10 and P.sscs_stream(5, "c") == P.sscs_stream(6, "a") == 12
    assert P.inpaint_stream(3, 2) == (3 << 2) | (1 << 62) | 2
    f = P.flat_normals(seed, P.inpaint_stream(3, 1), B * chw)
    assert np.array_equal(f, P.flat_normals_at(seed, P.inpaint_stream(3, 1), np.arange(B * chw)))
    # standard normal to sampling accuracy, and the tail stays inside the device's 6.77 sigma
    z = P.flat_normals(seed, 9, 1 << 20)
    assert abs(z.mean()) < 5e-3 and abs(z.var() - 1) < 5e-3 and np.abs(z).max() < 6.77


def _merge_ref(hb, hc):
    """One draw for two consecutive half-steps, from the oracle's algebra: A = A_c A_b and
    L L^T = A_c L_b L_b^T A_c^T + L_c L_c^T."""
    (ab, lb), (ac, lc) = ([np.array(v, dtype=np.float64).reshape(2, 2) for v in h] for h in (hb, hc))
    S = ac @ lb @ lb.T @ ac.T + lc @ lc.T
    return ac @ ab, S


@pytest.mark.parametrize("n_steps,stride,sde", [(1000, "uniform", {}), (1000, "quadratic", {}),
                                                (1000, "uniform", dict(nu=4.0, gamma=0.0)),
                                                (4000, "uniform", dict(nu=4.0, gamma=0.0)),
                                                (1000, "uniform", dict(beta_min=0.5, beta_max=12.0))])
def test_merged_half_steps_identity(n_steps, stride, sde):
    """merge_noise tables (half B of step i and half A of step i+1 as one Gaussian draw) satisfy, row
    by row, A_bc = A_c A_b and L_bc L_bc^T = A_c L_b L_b^T A_c^T + L_c L_c^T with L_bc lower-triangular,
    computed from oracle.PSLDScalars.half_step; the last row and the other halves stay unmerged.
    (With a constant beta on a uniform grid A_b = A_c, so the linear-beta row pins A_c against A_b.)"""
    from psld_b200 import cifar10_config
    cfg = cifar10_config(n_discrete_steps=n_steps, stride_type=stride)
    cfg.model.sde.update(sde)
    s = O.PSLDScalars(cfg)
    ts, n = O.time_grid(cfg)
    tab = StepTables(PSLDSchedule(cfg), torch.from_numpy(ts), n, "sscs_sde", True, 1e-3, merge_noise=True)
    halves = [s.half_step(float(ts[i]), float(ts[i + 1] - ts[i]) / 2) for i in range(n)]
    err_a, err_s, size_s = [], [], []
    for i in range(n):
        r = tab.sscs[i]
        hb = r.half_b
        a = np.array([[hb.a_xx, hb.a_xm], [hb.a_mx, hb.a_mm]])
        lt = np.array([[hb.c11, hb.c12], [hb.c21, hb.c22]])
        if i + 1 < n:
            a_ref, S = _merge_ref(halves[i], halves[i + 1])
            assert hb.c12 == 0.0 and hb.c11 > 0 and hb.c22 > 0
        else:
            a_ref = np.array(halves[i][0]).reshape(2, 2)
            l_ref = np.array(halves[i][1]).reshape(2, 2)
            S = l_ref @ l_ref.T
        err_a.append(float(np.abs(a - a_ref).max() / np.abs(a_ref).max()))
        err_s.append(float(np.abs(lt @ lt.T - S).max()))
        size_s.append(float(np.abs(S).max()))
        np.testing.assert_allclose([r.half_a.a_xx, r.half_a.c11, r.half_a.c21, r.half_a.c22],
                                   [halves[i][0][0], *np.array(halves[i][1])[[0, 2, 3]]], rtol=1e-10)
    err_s, size_s = np.array(err_s), np.array(size_s)
    worst_a, worst_s = max(err_a), float(err_s.max() / size_s.max())
    # per row: the oracle (math.exp) and the tables (torch.exp) evaluate the half-step variance
    # separately; at the smallest quadratic-stride steps its bracket cancels to ~2e-13 of the row
    worst_row = float((err_s / size_s).max())
    print(f"merged rows: A {worst_a:.2e}, covariance {worst_s:.2e} of max|S| ({worst_row:.2e} per row)")
    assert worst_a <= 1e-13 and worst_s <= 1e-13 and worst_row <= 1e-11, (worst_a, worst_s, worst_row)
