"""The fp32-tolerance tensor-core tier ("bf16x3") on the GPU, through the C ABI.

Every contraction operand (activations AND weights) is split bf16: value = hi + lo, 16
significand bits; a product a*w is three bf16 tcgen05 MMAs (a_hi w_hi + a_hi w_lo + a_lo w_hi)
into one fp32 TMEM accumulator.  The dropped a_lo*w_lo term and the two operand roundings are
each <= 2^-17 relative, so a dot product is good to ~1e-5 of its terms' magnitude.

Stated tolerances (relative L2 unless noted):
  split-bf16 storage round trip ............ <= 2^-17 (8e-6) max relative per element
  tcgen05 x3 convolution vs fp64 conv ...... <= 2e-5   (measured ~3e-6)
  memory-bound kernels on split tensors .... <= 1e-5   (fp32 math, one split rounding of the result)
  NCSN++ forward vs reference goldens ...... <= 5e-5   (fp32 CUDA-core path: 2e-5, bf16 path: 3e-2)
  BASELINE configs[0] 100-NFE end state .... <= 1e-4   (rel-L2 and max-abs/max|ref|)
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from _net import make_net, sampler_inputs
from _ops import (Split, attn_op, conv_op, conv_ref, fir_op, from_split, gn_op, max_rel, mg_ref,
                  per_sample_rel_l2, rel_l2, run_op, to_split, val)
from psld_b200 import _lib as L
from psld_b200 import (EulerMaruyamaSampler, PSLD, SSCSSampler, celeba64_config, cifar10_config,
                       mid_config, time_grid, tiny_config)

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _rng(seed):
    return np.random.default_rng(seed)


def _t(a, dtype=torch.float32):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV, dtype)


def _s(a):
    """random fp32 values -> split-bf16 storage on the GPU"""
    return to_split(_t(a))


def test_split_roundtrip_and_layout_op():
    r = _rng(0)
    x = _t(r.standard_normal((3, 8, 8, 16)) * np.exp(r.uniform(-20, 20, (3, 8, 8, 16))))
    s = to_split(x)
    err = ((from_split(s) - x).abs() / x.abs()).max().item()
    assert err <= 2.0 ** -16, err
    # NCHW fp32 -> split NHWC (zero-padded channels) -> NCHW fp32 through PSLD_OP_LAYOUT
    N, Cc, HW, CP = 2, 6, 64, 16
    xin = _t(r.standard_normal((N, Cc, 8, 8)))
    mid = torch.zeros(N, 8, 8, CP, dtype=torch.float32, device=DEV).as_subclass(Split)
    op = L.Op()
    op.kind = L.OP_LAYOUT
    op.i[L.LAYOUT_N], op.i[L.LAYOUT_C], op.i[L.LAYOUT_HW] = N, Cc, HW
    op.i[L.LAYOUT_DIR], op.i[L.LAYOUT_DTYPE], op.i[L.LAYOUT_CPAD], op.i[L.LAYOUT_CWRITE] = 0, L.BF16S, CP, 8
    op.inp[0], op.out[0] = xin.data_ptr(), mid.data_ptr()
    run_op(op)
    v = from_split(mid)
    assert max_rel(v[..., :Cc].permute(0, 3, 1, 2), xin) <= 2.0 ** -16
    assert float(v[..., Cc:].abs().max()) == 0.0


X3_CASES = [
    # N, H, W, C1, C2, Cout, ks
    (2, 32, 32, 64, 0, 64, 1),
    (2, 32, 32, 64, 0, 128, 3),
    (1, 16, 16, 128, 0, 256, 3),
    (3, 8, 8, 128, 64, 128, 1),        # two-source 1x1, BN_img = 2 with an odd batch
    (3, 8, 8, 256, 0, 256, 3),
    (2, 16, 16, 256, 0, 768, 1),       # fused q|k|v projection, 3 N-tiles
    (1, 64, 64, 64, 0, 32, 3),         # CelebA-size map
    (2, 32, 32, 256, 256, 256, 1),
    (41, 32, 32, 128, 0, 256, 3),      # 328 M tiles = 164 pairs over 74 clusters: persistent loop, both accumulators
    (37, 16, 16, 256, 128, 256, 3),    # odd tile count (partial last pair), two sources
]


@pytest.mark.parametrize("case", X3_CASES)
def test_conv_tc_x3(case):
    N, H, W, C1, C2, Cout, ks = case
    r = _rng(sum(case) + 3)
    x1 = _s(r.standard_normal((N, H, W, C1)) * 1.3)
    x2 = _s(r.standard_normal((N, H, W, C2))) if C2 else None
    w = _t(r.standard_normal((Cout, C1 + C2, ks, ks)) / np.sqrt((C1 + C2) * ks * ks))
    b = _t(0.1 * r.standard_normal(Cout))
    res = _s(r.standard_normal((N, H, W, Cout)))
    temb = _t(r.standard_normal((N, Cout + 32)))
    kw = dict(residual=res, temb=temb, temb_off=32, temb_bstride=Cout + 32, scale=0.7071)
    op, out, keep = conv_op(x1, x2, w, b, engine=L.ENGINE_TC, mg_stats=True, **kw)
    run_op(op, prepare=True)
    ref = conv_ref(x1, x2, w, b, **kw)                 # exact fp32 weights: the tier's claim
    err = rel_l2(val(out).permute(0, 3, 1, 2), ref)
    emx = max_rel(val(out).permute(0, 3, 1, 2), ref)
    print(f"x3 conv {case}: rel-L2 {err:.2e} max {emx:.2e}")
    assert err <= 2e-5 and emx <= 2e-5, (err, emx)
    mg = keep[-1]
    mref = mg_ref(ref.permute(0, 2, 3, 1))
    assert float((mg.double().cpu() - mref).abs().max()) <= 2e-5 * float(mref.abs().max())
    # fp32 NCHW head output (no epilogue terms)
    op, out2, keep2 = conv_op(x1, x2, w, None, engine=L.ENGINE_TC, out_nchw_f32=True)
    run_op(op, prepare=True)
    assert rel_l2(out2, conv_ref(x1, x2, w, None)) <= 2e-5


@pytest.mark.parametrize("case", [(2, 17, 17, 256, 256), (3, 33, 33, 64, 256), (5, 9, 9, 128, 64)])
def test_conv_tc_x3_stride2(case):
    N, H, W, Cin, Cout = case
    r = _rng(sum(case))
    x = _s(r.standard_normal((N, H, W, Cin)))
    w = _t(r.standard_normal((Cout, Cin, 3, 3)) / np.sqrt(Cin * 9))
    b = _t(0.1 * r.standard_normal(Cout))
    OH = (H - 3) // 2 + 1
    if (OH * OH) % 32:
        pytest.skip("split output needs H*W % 32 == 0")
    res = _s(r.standard_normal((N, OH, OH, Cout)))
    kw = dict(stride=2, pad=0, residual=res, scale=0.7071)
    op, out, keep = conv_op(x, None, w, b, engine=L.ENGINE_TC, **kw)
    run_op(op, prepare=True)
    assert rel_l2(val(out).permute(0, 3, 1, 2), conv_ref(x, None, w, b, **kw)) <= 2e-5


@pytest.mark.parametrize("case", [(2, 32, 32, 256, 256, 256, 256), (3, 16, 16, 256, 256, 0, 256),
                                  (4, 8, 8, 128, 64, 64, 128)])
def test_conv_tc_x3_fused_shortcut(case):
    N, H, W, Cb, E1, E2, Cout = case
    r = _rng(sum(case) + 9)
    b_in = _s(r.standard_normal((N, H, W, Cb)))
    e1 = _s(r.standard_normal((N, H, W, E1)))
    e2 = _s(r.standard_normal((N, H, W, E2))) if E2 else None
    w = _t(r.standard_normal((Cout, Cb, 3, 3)) / np.sqrt(Cb * 9))
    we = _t(r.standard_normal((Cout, E1 + E2, 1, 1)) / np.sqrt(E1 + E2))
    bias = _t(0.1 * r.standard_normal(Cout))
    op, out, keep = conv_op(b_in, None, w, bias, engine=L.ENGINE_TC, scale=0.7071, ext=(e1, e2, we),
                            mg_stats=True)
    run_op(op, prepare=True)
    ref = (conv_ref(b_in, None, w, bias) + conv_ref(e1, e2, we, None)) * 0.7071
    assert rel_l2(val(out).permute(0, 3, 1, 2), ref) <= 2e-5


@pytest.mark.parametrize("case", [(2, 32, 32, 64, 0, 64), (3, 32, 32, 256, 0, 256), (2, 16, 16, 128, 128, 256),
                                  (5, 16, 16, 256, 0, 128), (1, 32, 32, 256, 128, 256), (37, 16, 16, 256, 0, 256)])
@pytest.mark.parametrize("silu", [True, False])
def test_conv_gn_fused_x3(case, silu):
    """GroupNorm(+SiLU)-on-load 3x3 conv of the split-bf16 tier (conv_gn_x3_kernel: fp32 normalisation of
    the raw hi+lo tile in shared memory, two-phase transform around a single operand set, three MMA
    groups per tap) vs the fp64 definition."""
    N, H, W, C1, C2, Cout = case
    r = _rng(sum(case) + 5)
    x1 = _s(r.standard_normal((N, H, W, C1)) * 1.7 + 0.3)
    x2 = _s(r.standard_normal((N, H, W, C2)) * 0.6 - 0.2) if C2 else None
    Cin = C1 + C2
    w = _t(r.standard_normal((Cout, Cin, 3, 3)) / np.sqrt(Cin * 9))
    b = _t(0.1 * r.standard_normal(Cout))
    aff = _t(np.stack([1 + 0.3 * r.standard_normal((N, Cin)), 0.2 * r.standard_normal((N, Cin))], -1))
    res = _s(r.standard_normal((N, H, W, Cout)))
    temb = _t(r.standard_normal((N, Cout)))
    kw = dict(residual=res, temb=temb, temb_off=0, temb_bstride=Cout, scale=0.7071)
    op, out, keep = conv_op(x1, x2, w, b, engine=L.ENGINE_TC_GN, mg_stats=True, affine=aff, gn_silu=silu, **kw)
    run_op(op, prepare=True)
    xx = val(x1).double().cpu() if x2 is None else torch.cat([val(x1).double().cpu(), val(x2).double().cpu()], -1)
    a = xx * aff.double().cpu()[:, None, None, :, 0] + aff.double().cpu()[:, None, None, :, 1]
    if silu:
        a = F.silu(a)
    ref = conv_ref(a, None, w, b, **kw)
    err, emx = rel_l2(val(out).permute(0, 3, 1, 2), ref), max_rel(val(out).permute(0, 3, 1, 2), ref)
    print(f"x3 GN-fused conv {case} silu={silu}: rel-L2 {err:.2e} max {emx:.2e}")
    assert err <= 2e-5 and emx <= 3e-5, (err, emx)
    mref = mg_ref(ref.permute(0, 2, 3, 1))
    assert float((keep[-1].double().cpu() - mref).abs().max()) <= 3e-5 * float(mref.abs().max())


@pytest.mark.parametrize("case", [(2, 32, 32, 256, 256, 256, 256), (3, 16, 16, 256, 256, 0, 256),
                                  (2, 32, 32, 128, 64, 0, 128), (3, 16, 16, 256, 128, 256, 256),
                                  (39, 16, 16, 256, 256, 256, 256)])
def test_conv_gn_fused_x3_with_shortcut(case):
    """GroupNorm_1+SiLU on load -> Conv_1, plus the Conv_2 1x1 shortcut over the RAW block input
    cat(e1, e2) as extra k-blocks from the kernel's 3-slot shortcut ring (layerspp.py:262-274)."""
    N, H, W, Cb, E1, E2, Cout = case
    r = _rng(sum(case) + 13)
    h = _s(r.standard_normal((N, H, W, Cb)) * 1.5 + 0.2)
    e1 = _s(r.standard_normal((N, H, W, E1)))
    e2 = _s(r.standard_normal((N, H, W, E2))) if E2 else None
    w = _t(r.standard_normal((Cout, Cb, 3, 3)) / np.sqrt(Cb * 9))
    we = _t(r.standard_normal((Cout, E1 + E2, 1, 1)) / np.sqrt(E1 + E2))
    bias = _t(0.1 * r.standard_normal(Cout))
    aff = _t(np.stack([1 + 0.3 * r.standard_normal((N, Cb)), 0.2 * r.standard_normal((N, Cb))], -1))
    op, out, keep = conv_op(h, None, w, bias, engine=L.ENGINE_TC_GN, scale=0.7071, ext=(e1, e2, we),
                            mg_stats=True, affine=aff, gn_silu=True)
    run_op(op, prepare=True)
    a = F.silu(val(h).double().cpu() * aff.double().cpu()[:, None, None, :, 0] + aff.double().cpu()[:, None, None, :, 1])
    ref = (conv_ref(a, None, w, bias) + conv_ref(e1, e2, we, None)) * 0.7071
    err, emx = rel_l2(val(out).permute(0, 3, 1, 2), ref), max_rel(val(out).permute(0, 3, 1, 2), ref)
    print(f"x3 GN-fused conv + shortcut {case}: rel-L2 {err:.2e} max {emx:.2e}")
    assert err <= 2e-5 and emx <= 3e-5, (err, emx)
    mref = mg_ref(ref.permute(0, 2, 3, 1))
    assert float((keep[-1].double().cpu() - mref).abs().max()) <= 3e-5 * float(mref.abs().max())


def test_conv_gn_fused_x3_output_head():
    """Final act(GroupNorm(h)) -> conv3x3 -> 6 channels as fp32 NCHW through the split-bf16 fused kernel."""
    r = _rng(78)
    N, H, W, Cin = 3, 32, 32, 128
    x = _s(r.standard_normal((N, H, W, Cin)) * 1.3 + 0.1)
    w = _t(r.standard_normal((6, Cin, 3, 3)) / 34.0)
    b = _t(0.1 * r.standard_normal(6))
    aff = _t(np.stack([1 + 0.3 * r.standard_normal((N, Cin)), 0.2 * r.standard_normal((N, Cin))], -1))
    op, out, keep = conv_op(x, None, w, b, engine=L.ENGINE_TC_GN, out_nchw_f32=True, affine=aff, gn_silu=True)
    run_op(op, prepare=True)
    a = F.silu(val(x).double().cpu() * aff.double().cpu()[:, None, None, :, 0] + aff.double().cpu()[:, None, None, :, 1])
    ref = conv_ref(a, None, w, b)
    assert out.shape == (N, 6, H, W)
    assert rel_l2(out, ref) <= 2e-5


def test_memory_bound_kernels_on_split_tensors():
    """GroupNorm(+SiLU) over a virtual concat, the three FIR resamplers and the CUDA-core attention
    core with split-bf16 input and output vs fp64 references of the same (hi + lo) inputs."""
    r = _rng(21)
    N, H, W, C1, C2 = 3, 16, 16, 64, 32
    x1, x2 = _s(r.standard_normal((N, H, W, C1)) * 2 + 0.5), _s(r.standard_normal((N, H, W, C2)))
    Cc, G = C1 + C2, 24
    ga, be = _t(1 + 0.2 * r.standard_normal(Cc)), _t(0.1 * r.standard_normal(Cc))
    op, y, keep = gn_op(x1, x2, ga, be, G, True)
    run_op(op)
    xx = torch.cat([val(x1), val(x2)], -1).double().cpu().permute(0, 3, 1, 2)
    ref = F.silu(F.group_norm(xx, G, ga.double().cpu(), be.double().cpu(), eps=1e-6)).permute(0, 2, 3, 1)
    assert rel_l2(y, ref) <= 1e-5
    # with producer-side statistics
    op, y2, keep = gn_op(x1, x2, ga, be, G, True, mg1=mg_ref(val(x1)).to(DEV), mg2=mg_ref(val(x2)).to(DEV))
    run_op(op)
    assert rel_l2(y2, ref) <= 1e-5
    k = np.outer([1, 3, 3, 1], [1, 3, 3, 1]).astype(np.float32)
    k /= k.sum()
    from oracle import psld_oracle as O
    for (taps, up, down, p0, p1) in [(k * 4, 2, 1, 2, 1), (k, 1, 2, 1, 1), (k, 1, 1, 2, 2)]:
        op, yf = fir_op(x1, taps, up, down, p0, p1)
        run_op(op)
        rf = O.upfirdn2d(val(x1).cpu().permute(0, 3, 1, 2), torch.from_numpy(taps), up, down, (p0, p1))
        assert rel_l2(val(yf).permute(0, 3, 1, 2), rf) <= 1e-5, (up, down)
    Ca = 64
    qkv = _s(r.standard_normal((2, 16, 16, 3 * Ca)))
    op, o = attn_op(qkv, Ca)
    run_op(op)
    q, kk, v = val(qkv).double().cpu().reshape(2, 256, 3 * Ca).split(Ca, -1)
    wgt = torch.softmax(q @ kk.transpose(1, 2) * Ca ** -0.5, -1)
    assert rel_l2(val(o).reshape(2, 256, Ca), wgt @ v) <= 1e-5


@pytest.mark.parametrize("shape", [(2, 16, 16, 256), (3, 8, 8, 256), (2, 16, 16, 64), (1, 8, 16, 128),
                                   (4, 8, 8, 64)])
def test_attention_tc_x3(shape):
    """tcgen05 attention core with split-bf16 q|k|v, P and output: three MMA groups per GEMM."""
    N, H, W, Cc = shape
    r = _rng(19)
    qkv = _s(r.standard_normal((N, H, W, 3 * Cc)) * 1.5)
    op, out = attn_op(qkv, Cc, engine=L.ENGINE_TC)
    run_op(op, prepare=True)
    q, k, v = val(qkv).double().cpu().reshape(N, H * W, 3 * Cc).split(Cc, dim=-1)
    wgt = torch.softmax(torch.einsum("bqc,bkc->bqk", q, k) * (int(Cc) ** -0.5), dim=-1)
    ref = torch.einsum("bqk,bkc->bqc", wgt, v)
    err = rel_l2(val(out).reshape(N, H * W, Cc), ref)
    print(f"x3 attention {shape}: rel-L2 {err:.2e}")
    assert err <= 2e-5, err


@pytest.mark.parametrize("shape", [(2, 16, 16, 256), (3, 16, 8, 128), (5, 16, 16, 64), (1, 16, 16, 192)])
def test_attention_tc_x3_fused_projection(shape):
    """Attention core + NIN_3 projection + skip connection + GroupNorm statistics in one kernel
    (AttnBlockpp, layerspp.py:82-91), split-bf16 tier, vs the fp64 definition."""
    N, H, W, Cc = shape
    r = _rng(23)
    qkv = _s(r.standard_normal((N, H, W, 3 * Cc)) * 1.5)
    x = _s(r.standard_normal((N, H, W, Cc)))
    w3 = _t(r.standard_normal((Cc, Cc)) / np.sqrt(Cc))          # [out, in]
    b3 = _t(0.1 * r.standard_normal(Cc))
    op, out, keep = attn_op(qkv, Cc, engine=L.ENGINE_TC, proj=(w3, b3, x, 0.7071))
    run_op(op, prepare=True)
    q, k, v = val(qkv).double().cpu().reshape(N, H * W, 3 * Cc).split(Cc, dim=-1)
    wgt = torch.softmax(torch.einsum("bqc,bkc->bqk", q, k) * (int(Cc) ** -0.5), dim=-1)
    o = torch.einsum("bqk,bkc->bqc", wgt, v)
    ref = (o @ w3.double().cpu().t() + b3.double().cpu() + val(x).double().cpu().reshape(N, H * W, Cc)) * 0.7071
    err = rel_l2(val(out).reshape(N, H * W, Cc), ref)
    print(f"x3 attention+proj {shape}: rel-L2 {err:.2e}")
    assert err <= 2e-5, err
    mref = mg_ref(ref.reshape(N, H, W, Cc))
    assert float((keep[-1].double().cpu() - mref).abs().max()) <= 2e-5 * float(mref.abs().max())


# ------------------------------------------------------------------ whole network
def _full(c):
    c.model.score_fn.init_scale = 1.0
    return c


FWD = {
    "tiny": (tiny_config, "forward_tiny.npz"), "mid": (mid_config, "forward_mid.npz"),
    "cifar10": (lambda: _full(cifar10_config()), "forward_cifar10.npz"),
    "cifar10_b3": (lambda: _full(cifar10_config()), "forward_cifar10_b3.npz"),
    "celeba64": (lambda: _full(celeba64_config()), "forward_celeba64.npz"),
    "celeba64_b2": (lambda: _full(celeba64_config()), "forward_celeba64_b2.npz"),
}


@pytest.mark.parametrize("name", list(FWD))
def test_forward_x3_vs_golden(golden_dir, name):
    mk, fname = FWD[name]
    g = np.load(f"{golden_dir}/{fname}")
    net, _ = make_net(mk(), "bf16x3")
    y = net(torch.from_numpy(g["x"]).cuda(), torch.from_numpy(g["t"]).cuda())
    torch.cuda.synchronize()
    ref = torch.from_numpy(g["y"])
    err, emx = rel_l2(y, ref), max_rel(y, ref)
    plan = net.plan(g["x"].shape[0], g["x"].shape[0], False)
    print(f"forward {name} bf16x3: rel-L2 {err:.3e} max-abs/max|ref| {emx:.3e} engines {plan.engine_count}")
    assert err <= 5e-5 and emx <= 5e-5, (err, emx)
    if name not in ("tiny",):
        assert plan.engine_count["simt"] == 0, plan.engine_count     # every contraction on tcgen05
    assert torch.equal(y, net(torch.from_numpy(g["x"]).cuda(), torch.from_numpy(g["t"]).cuda()))


def _run(cfg, kind, net, u0, nb, state_dtype=torch.float64, fuse=False, record=True):
    S = (SSCSSampler if kind == "sscs_sde" else EulerMaruyamaSampler)(cfg, PSLD(cfg), net)
    S.use_graph = False
    S.state_dtype = state_dtype
    S.fuse_halves = fuse
    S.merge_noise = False
    S.noise = torch.stack(nb).cuda()
    S.record = True if record else None
    ts, n = time_grid(cfg)
    out = S.sample(u0.cuda(), ts.cuda(), n, denoise=cfg.evaluation.denoise, eps=cfg.evaluation.eval_eps)
    torch.cuda.synchronize()
    return out, (S.record if record else None)


def _traj_errors(g, out, rec):
    ref = torch.from_numpy(g["final"])
    e_l2, e_mx = rel_l2(out, ref), max_rel(out, ref)
    worst = 0.0
    for i in g["probe"]:
        s_ref = torch.from_numpy(g[f"state_{int(i)}"])
        worst = max(worst, max_rel(rec[int(i)][: s_ref.shape[0]], s_ref))
    st = g["stats"]
    l2 = (rec.double().reshape(rec.shape[0], -1) ** 2).sum(1).cpu().numpy()
    worst = max(worst, float(np.max(np.abs(l2 - st[:, 3]) / st[:, 3])) / 2)
    return e_l2, e_mx, worst


@pytest.mark.parametrize("kind,fname", [("em_sde", "sampler_tiny_em100.npz"),
                                        ("sscs_sde", "sampler_tiny_sscs100.npz")])
def test_x3_sampler_configs0_vs_reference_golden(golden_dir, kind, fname):
    """BASELINE.json configs[0] (tiny NCSN++, 100 NFE, 8 samples) through the native loop with the
    bf16x3 network: end state and per-step probes within the tier's stated 1e-4."""
    g = np.load(f"{golden_dir}/{fname}")
    cfg = tiny_config(sampler=kind)
    net, _ = make_net(cfg, "bf16x3")
    u0, nb = sampler_inputs(cfg, int(g["B"]), int(g["n"]), kind)
    out, rec = _run(cfg, kind, net, u0, nb)
    e_l2, e_mx, worst = _traj_errors(g, out, rec)
    print(f"configs[0] {kind} bf16x3: final rel-L2 {e_l2:.3e} max {e_mx:.3e} worst per-step {worst:.3e}")
    assert e_l2 <= 1e-4 and e_mx <= 1e-4 and worst <= 1e-4


# measured on B200 (printed by the test); gates are <= 2x measured, rounded up
CIFAR_TRAJ_GATES = {"fp32": 2e-5, "bf16x3": 1e-4, "bf16": 2e-2}


@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
def test_configs1_trajectory_vs_reference_golden(golden_dir, precision):
    """The BENCHMARKED configuration (BASELINE.json configs[1]: CIFAR-10 NCSN++ nf=128,
    ch_mult=[2,2,2], 8 res blocks, SSCS) on a 50-NFE trajectory of 2 samples generated by the
    unmodified reference (oracle/make_golden.py::golden_full_size, init_scale=1, pre-drawn noise):
    per-step probe states, per-step energy and the final samples, for all three precision tiers."""
    g = np.load(f"{golden_dir}/sampler_cifar10_sscs50.npz")
    cfg = _full(cifar10_config(n_discrete_steps=50, batch_size=2, n_samples=2))
    net, _ = make_net(cfg, precision)
    u0, nb = sampler_inputs(cfg, int(g["B"]), int(g["n"]), "sscs_sde")
    out, rec = _run(cfg, "sscs_sde", net, u0, nb)
    e_l2, e_mx, worst = _traj_errors(g, out, rec)
    print(f"configs[1] SSCS 50 NFE {precision}: final rel-L2 {e_l2:.3e} max-abs/max|ref| {e_mx:.3e} "
          f"worst per-step {worst:.3e}")
    tol = CIFAR_TRAJ_GATES[precision]
    assert e_l2 <= tol and e_mx <= 2 * tol and worst <= 2 * tol, (e_l2, e_mx, worst)


@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
def test_configs1_full_length_vs_reference_golden(golden_dir, precision):
    """BASELINE.json configs[1] at FULL length: all 1000 SSCS steps of the benchmarked CIFAR-10 NCSN++ against the
    trajectory of the unmodified reference (oracle/make_golden.py::golden_full_length, B = 2, init_scale = 1,
    pre-drawn noise): per-step energy of all 1000 states, probe states and the final samples."""
    g = np.load(f"{golden_dir}/sampler_cifar10_sscs1000.npz")
    cfg = _full(cifar10_config(n_discrete_steps=1000, batch_size=2, n_samples=2))
    net, _ = make_net(cfg, precision)
    assert int(g["n"]) == 999
    u0, nb = sampler_inputs(cfg, int(g["B"]), int(g["n"]), "sscs_sde")
    out, rec = _run(cfg, "sscs_sde", net, u0, nb)
    e_l2, e_mx, worst = _traj_errors(g, out, rec)
    print(f"configs[1] SSCS 1000 NFE {precision}: final rel-L2 {e_l2:.3e} max-abs/max|ref| {e_mx:.3e} "
          f"worst per-step {worst:.3e}")
    # measured on B200: fp32 2.5e-7 / 3.4e-7, bf16x3 1.2e-5 / 1.7e-5, bf16 3.6e-3 / 4.0e-3
    tol = {"fp32": 2e-6, "bf16x3": 5e-5, "bf16": 8e-3}[precision]
    assert e_l2 <= tol and e_mx <= 2 * tol and worst <= 2 * tol, (e_l2, e_mx, worst)


@pytest.mark.parametrize("precision", ["bf16x3", "bf16"])
def test_configs3_full_length_vs_reference_golden(golden_dir, precision):
    """BASELINE.json configs[3] at FULL length: all 1000 SSCS steps of the CelebA-64 NCSN++ (B = 1) against the
    unmodified reference (oracle/make_golden.py --only-full-length --celeba)."""
    g = np.load(f"{golden_dir}/sampler_celeba64_sscs1000.npz")
    cfg = _full(celeba64_config(n_discrete_steps=1000, batch_size=1, n_samples=1))
    net, _ = make_net(cfg, precision)
    u0, nb = sampler_inputs(cfg, int(g["B"]), int(g["n"]), "sscs_sde")
    out, rec = _run(cfg, "sscs_sde", net, u0, nb)
    e_l2, e_mx, worst = _traj_errors(g, out, rec)
    print(f"configs[3] SSCS 1000 NFE {precision}: final rel-L2 {e_l2:.3e} max-abs/max|ref| {e_mx:.3e} "
          f"worst per-step {worst:.3e}")
    tol = {"bf16x3": 5e-5, "bf16": 8e-3}[precision]      # measured 8.3e-6 / 3.8e-3
    assert e_l2 <= tol and e_mx <= 2 * tol and worst <= 2 * tol, (e_l2, e_mx, worst)


def test_configs3_trajectory_vs_reference_golden(golden_dir):
    """BASELINE.json configs[3] (CelebA-64 NCSN++, SSCS): 20-NFE reference trajectory, bf16x3 tier."""
    g = np.load(f"{golden_dir}/sampler_celeba64_sscs20.npz")
    cfg = _full(celeba64_config(n_discrete_steps=20, batch_size=2, n_samples=2))
    net, _ = make_net(cfg, "bf16x3")
    u0, nb = sampler_inputs(cfg, int(g["B"]), int(g["n"]), "sscs_sde")
    out, rec = _run(cfg, "sscs_sde", net, u0, nb)
    e_l2, e_mx, worst = _traj_errors(g, out, rec)
    print(f"configs[3] SSCS 20 NFE bf16x3: final rel-L2 {e_l2:.3e} max {e_mx:.3e} worst per-step {worst:.3e}")
    assert e_l2 <= 1e-4 and e_mx <= 2e-4 and worst <= 2e-4


def test_x3_full_batch_properties():
    """bf16x3 plan at the bench batch (B = 256, CIFAR-10 NCSN++): finite, per-sample independent
    (same samples through a B = 4 plan with different tiling), equal to the fp32 CUDA-core path."""
    cfg = _full(cifar10_config())
    net, _ = make_net(cfg, "bf16x3")
    r = np.random.default_rng(11)
    x = torch.from_numpy(r.standard_normal((256, 6, 32, 32)).astype(np.float32)).cuda()
    t = torch.full((256,), 0.43, device="cuda")
    y = net(x, t)
    torch.cuda.synchronize()
    assert torch.isfinite(y).all()
    idx = [0, 1, 130, 255]
    ys = net(x[idx].contiguous(), t[:4])
    net32, _ = make_net(cfg, "fp32")
    y32 = net32(x[idx].contiguous(), t[:4])
    e_shard, e_prec = rel_l2(ys, y[idx]), rel_l2(y[idx], y32)
    # every sample of the B = 256 plan against the fp32 CUDA-core plan at B = 256
    e_each = per_sample_rel_l2(y, net32(x, t))
    worst = int(e_each.argmax())
    print(f"bf16x3 B=256 vs B=4 plan {e_shard:.3e}; vs fp32 CUDA-core path {e_prec:.3e}; worst of 256 samples "
          f"vs fp32 B=256 plan {float(e_each[worst]):.3e} (sample {worst})")
    assert e_shard <= 1e-5 and e_prec <= 5e-5
    assert float(e_each.max()) <= 5e-5, (worst, float(e_each[worst]))
