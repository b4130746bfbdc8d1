"""Host (no GPU): attention at 32x32 and 64x64 maps.  The dry plan of a 64x64 net with attention at
64, 32 and 16 (4096, 1024 and 256 tokens) puts every attention block on the tensor cores in both
tensor-core tiers, fused with its output projection, and the planner's eligibility rule is the one
prepare_attn_tc states (include/psld_b200.h)."""
import pytest

from psld_b200 import NCSNpp, celeba64_config
from psld_b200 import _lib as L
from psld_b200.program import Plan, build_plan


def attn64_config(**ev):
    cfg = celeba64_config(**ev)
    cfg.model.score_fn.update(attn_resolutions=[64, 32, 16], init_scale=1.0)
    return cfg


@pytest.mark.parametrize("precision", ["bf16x3", "bf16"])
def test_attn64_net_puts_attention_on_tensor_cores(precision):
    net = NCSNpp(attn64_config()).eval()
    net.precision = precision
    plan = build_plan(net, 2, 1, True, dry=True)
    attn = [op for op in plan.ops if op.kind == L.OP_ATTN]
    assert attn and all(op.engine == L.ENGINE_TC for op in attn)
    # the projection is fused wherever HW % 128 == 0 (all but the 8x8 mid block)
    assert all(op.i[L.ATTN_PROJ] == (op.i[L.ATTN_HW] % 128 == 0) for op in attn)
    hw = sorted({op.i[L.ATTN_HW] for op in attn})
    assert hw == [64, 256, 1024, 4096], hw          # the mid block attends at 8x8
    assert plan.engine_count.get("attn_simt", 0) == 0, plan.engine_count


def test_attn_tc_eligibility():
    ok = Plan._attn_tc_eligible
    for c in (64, 128, 192, 256):
        for hw in (64, 128, 256, 512, 640, 1024, 4096, 16384):
            assert ok(hw, c), (hw, c)
        for hw in (32, 100, 192, 384, 576, 1000):
            assert not ok(hw, c), (hw, c)
    for c in (32, 96, 320, 512):
        assert not ok(1024, c), c
