"""NCSN++ forward on the GPU (C ABI program) vs golden vectors produced by the reference.

Tolerances (relative L2 over the whole output, stated per path):
  fp32 path (CUDA-core fp32 convolutions) ... <= 2e-5   (measured ~2e-6; fp32 summation order)
  bf16 path (tcgen05 convolutions) .......... <= 2e-2   (measured 0.85e-2..1.2e-2: bf16 activations +
                                                         weights; the reference under bf16 autocast
                                                         sits at 4e-3..6e-3 per SURVEY.md §8c, bf16
                                                         storage adds to it; gate <= 2x measured)
  bf16x3 path (default tier) ................ <= 5e-5   (measured 1.4e-5..2.2e-5; tests/test_gpu_x3.py)
"""
import numpy as np
import pytest
import torch

from _net import make_net
from _ops import per_sample_rel_l2, rel_l2
from oracle import psld_oracle as O
from psld_b200 import celeba64_config, cifar10_config, mid_config, tiny_config

pytestmark = pytest.mark.gpu

CASES = {
    "tiny": tiny_config, "mid": mid_config,
    "cifar10": lambda: _full(cifar10_config()), "celeba64": lambda: _full(celeba64_config()),
}


def _full(c):
    c.model.score_fn.init_scale = 1.0
    return c


@pytest.mark.parametrize("name", ["tiny", "mid", "cifar10", "celeba64"])
@pytest.mark.parametrize("precision,tol", [("fp32", 2e-5), ("bf16", 2e-2)])
def test_forward_vs_golden(golden_dir, name, precision, tol):
    g = np.load(f"{golden_dir}/forward_{name}.npz")
    cfg = CASES[name]()
    net, _ = make_net(cfg, precision)
    x = torch.from_numpy(g["x"]).cuda()
    t = torch.from_numpy(g["t"]).cuda()
    y = net(x, t)
    torch.cuda.synchronize()
    err = rel_l2(y, torch.from_numpy(g["y"]))
    print(f"forward {name} {precision}: rel-L2 {err:.3e}")
    assert err <= tol, err
    if precision == "bf16" and name != "tiny":
        plan = net.plan(x.shape[0], x.shape[0], False)
        assert plan.engine_count["tc"] > plan.engine_count["simt"], plan.engine_count
    # second call reuses the plan and is deterministic
    y2 = net(x, t)
    assert torch.equal(y, y2)


def test_forward_shared_time_row_and_batch_invariance():
    """nt = 1 (sampling: one time for the whole batch) equals per-sample times; per-sample
    independence (GroupNorm/attention are per-sample, SURVEY.md §8e)."""
    cfg = tiny_config()
    net, sd = make_net(cfg, "fp32")
    r = np.random.default_rng(3)
    x = torch.from_numpy(r.standard_normal((5, 6, 32, 32)).astype(np.float32)).cuda()
    t = torch.full((5,), 0.37, device="cuda")
    y = net(x, t)
    p1 = net.plan(5, 1, True)
    p1.x_in.copy_(x)
    p1.time_buf.copy_(torch.log(t[:1].cpu()).cuda())
    p1.run()
    torch.cuda.synchronize()
    assert rel_l2(p1.eps, y) <= 1e-6
    y3 = net(x[1:3].contiguous(), t[1:3])
    assert rel_l2(y3, y[1:3]) <= 1e-6
    ref = O.ncsnpp_forward(cfg, sd, x.cpu(), t.cpu())
    assert rel_l2(y, ref) <= 2e-5


def test_module_contract():
    """state-dict names/shapes, deepcopy, load_state_dict, loud failure on CPU tensors."""
    import copy
    cfg = tiny_config()
    net, sd = make_net(cfg, "fp32")
    assert set(net.state_dict().keys()) == set(sd.keys())
    twin = copy.deepcopy(net)
    x = torch.randn(2, 6, 32, 32, device="cuda")
    t = torch.tensor([0.5, 0.2], device="cuda")
    assert torch.equal(net(x, t), twin(x, t))
    with pytest.raises(RuntimeError):
        net(x.cpu(), t.cpu())


def test_checkpoint_to_samples_cifar10(golden_dir, tmp_path):
    """Real-size checkpoint path on the GPU (sample.py:62-69): a Lightning-style .ckpt holding the
    749-tensor CIFAR-10 state dict under ``score_fn.`` / ``ema_score_fn.`` -> ``load_checkpoint`` into
    a module already on the GPU -> forward equals the reference's output for those weights ->
    ``samples_to_uint8`` image writer arithmetic."""
    from oracle.weights import fill_state_dict
    from psld_b200 import NCSNpp, load_checkpoint, samples_to_uint8
    cfg = _full(cifar10_config())
    net = NCSNpp(cfg).eval().cuda()                 # default precision tier
    assert net.precision == "bf16x3"
    sd = fill_state_dict({k: tuple(v.shape) for k, v in net.state_dict().items()}, 0)
    assert len(sd) == 749
    other = {k: v + 1.0 for k, v in list(sd.items())[:3]}
    path = tmp_path / "cifar10_psld.ckpt"
    torch.save({"state_dict": {**{"ema_score_fn." + k: v for k, v in sd.items()},
                               **{"score_fn." + k: other.get(k, v) for k, v in sd.items()}},
                "epoch": 2500, "global_step": 1}, path)
    load_checkpoint(net, str(path), sample_from="target")
    g = np.load(f"{golden_dir}/forward_cifar10_b3.npz")
    y = net(torch.from_numpy(g["x"]).cuda(), torch.from_numpy(g["t"]).cuda())
    err = rel_l2(y, torch.from_numpy(g["y"]))
    print(f"checkpoint -> forward (CIFAR-10, {net.precision}): rel-L2 {err:.3e}")
    assert err <= 5e-5
    img = samples_to_uint8(torch.cat([y[:, :3] * 0.4, y[:, 3:]], 1).double())
    ref = ((y[:, :3].double().cpu() * 0.4 * 0.5 + 0.5).permute(0, 2, 3, 1).numpy() * 255).clip(0, 255).astype(np.uint8)
    assert img.shape == (3, 32, 32, 3) and np.array_equal(img.cpu().numpy(), ref)


def test_in_place_weight_update_invalidates_plans():
    """A plan snapshots re-packed weights; an in-place parameter update (EMA / optimizer step /
    ``p.data.copy_``) must be picked up by the next call, as the reference module would."""
    cfg = tiny_config()
    net, sd = make_net(cfg, "bf16")
    x = torch.randn(2, 6, 32, 32, device="cuda")
    t = torch.tensor([0.5, 0.2], device="cuda")
    y0 = net(x, t).clone()
    assert torch.equal(net(x, t), y0)
    with torch.no_grad():
        for p in net.parameters():
            if p.dim() == 4:
                p.mul_(1.05)                       # in place: same storage, new version
    y1 = net(x, t).clone()
    assert not torch.equal(y1, y0)
    twin, _ = make_net(cfg, "bf16")
    twin.load_state_dict(net.state_dict())
    assert torch.equal(twin(x, t), y1)


@pytest.mark.parametrize("sf,B,precision,tol", [
    (dict(nf=96, ch_mult=[1, 2], num_res_blocks=1), 3, "bf16", 2e-2),     # channels 96/192/288: SIMT fallbacks, odd group sizes
    (dict(nf=64, ch_mult=[1, 1, 2], num_res_blocks=1), 5, "bf16", 2.4e-2),  # 8x8 level, 2 images per tile, odd batch
    (dict(nf=64, ch_mult=[1, 1, 2], num_res_blocks=1), 1, "bf16", 2.4e-2),  # single sample (single-tile layers)
    (dict(nf=64, ch_mult=[1, 2], num_res_blocks=1, fir=False, progressive_input="none",
          embedding_type="positional"), 2, "fp32", 2e-5),                 # ablation-script architecture flags
    (dict(nf=64, ch_mult=[1, 2], num_res_blocks=1, fir=False, progressive_input="none",
          embedding_type="positional"), 2, "bf16", 2.4e-2),
    (dict(nf=32, ch_mult=[1, 2], num_res_blocks=1, out_ch=3), 2, "fp32", 2e-5),   # score_m nets (out_ch = C)
    # the default tier (bf16x3) on the same odd shapes: split-bf16 CUDA-core fallbacks, 8x8 tiles with two
    # images, single-sample plans, the ablation-script switches, score_m nets
    (dict(nf=96, ch_mult=[1, 2], num_res_blocks=1), 3, "bf16x3", 5e-5),
    (dict(nf=64, ch_mult=[1, 1, 2], num_res_blocks=1), 5, "bf16x3", 5e-5),
    (dict(nf=64, ch_mult=[1, 1, 2], num_res_blocks=1), 1, "bf16x3", 5e-5),
    (dict(nf=64, ch_mult=[1, 2], num_res_blocks=1, fir=False, progressive_input="none",
          embedding_type="positional"), 2, "bf16x3", 5e-5),
    (dict(nf=32, ch_mult=[1, 2], num_res_blocks=1, out_ch=3), 2, "bf16x3", 5e-5),
    (dict(nf=128, ch_mult=[1, 2, 2, 2], num_res_blocks=1, attn_resolutions=[8]), 2, "bf16x3", 5e-5),  # attention at 8x8 only
])
def test_forward_odd_configs_vs_oracle(sf, B, precision, tol):
    """Shapes outside the tensor-core sweet spot, odd batches and the non-default architecture
    switches go through the same program (with CUDA-core fallbacks) and match the oracle."""
    from psld_b200 import make_config
    sf = dict(sf, init_scale=1.0)
    cfg = make_config(score_fn=sf)
    net, sd = make_net(cfg, precision)
    r = np.random.default_rng(B)
    x = torch.from_numpy(r.standard_normal((B, 6, 32, 32)).astype(np.float32))
    t = torch.from_numpy(r.uniform(0.01, 1.0, B).astype(np.float32))
    y = net(x.cuda(), t.cuda())
    torch.cuda.synchronize()
    ref = O.ncsnpp_forward(cfg, sd, x, t)
    err = rel_l2(y, ref)
    print(f"odd config {sf} B={B} {precision}: rel-L2 {err:.3e} engines {net.plan(B, B, False).engine_count}")
    assert err <= tol, err


def test_full_size_workload_properties():
    """BASELINE configs[1] at its full size (CIFAR-10 NCSN++, B = 256, bf16 tensor-core plan, the
    bench workload), checked through size-independent properties: per-sample independence (the
    same samples through a B = 4 plan, whose tiling / grid sizes differ), the shared-time-row
    fast path, and agreement with the fp32 CUDA-core path on a slice."""
    cfg = _full(cifar10_config())
    net, _ = make_net(cfg, "bf16")
    r = np.random.default_rng(11)
    x = torch.from_numpy(r.standard_normal((256, 6, 32, 32)).astype(np.float32)).cuda()
    t = torch.full((256,), 0.43, device="cuda")
    y = net(x, t)
    torch.cuda.synchronize()
    assert torch.isfinite(y).all()
    idx = [0, 1, 130, 255]
    ys = net(x[idx].contiguous(), t[:4])
    e_shard = rel_l2(ys, y[idx])
    p1 = net.plan(256, 1, True)             # sampling plan: one time row for the whole batch
    p1.x_in.copy_(x)
    p1.time_buf.copy_(torch.log(t[:1].cpu()).cuda())
    p1.run()
    torch.cuda.synchronize()
    e_row = rel_l2(p1.eps, y)
    net32, _ = make_net(cfg, "fp32")
    y32 = net32(x[idx].contiguous(), t[:4])
    e_prec = rel_l2(ys, y32)
    # every sample of the B = 256 plan against the fp32 CUDA-core plan at B = 256: a wrong tile in any
    # one image is not diluted by the other 255
    e_each = per_sample_rel_l2(y, net32(x, t))
    worst = int(e_each.argmax())
    print(f"B=256 vs B=4 plan {e_shard:.3e}; shared time row {e_row:.3e}; bf16 vs fp32 path {e_prec:.3e}; "
          f"worst of 256 samples vs fp32 B=256 plan {float(e_each[worst]):.3e} (sample {worst})")
    assert e_shard <= 1e-3 and e_row <= 1e-3 and e_prec <= 2e-2
    assert float(e_each.max()) <= 2e-2, (worst, float(e_each[worst]))
