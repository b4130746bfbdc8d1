"""CPU: the oracle against the UNMODIFIED reference, through outputs of the reference stored under
``tests/golden/`` (written by ``oracle/make_golden.py`` from the reference's own modules and samplers)."""
import json
import types

import numpy as np
import pytest
import torch

from oracle import psld_oracle as O
from oracle.weights import fill_state_dict, noise_bank, prior
from psld_b200 import NCSNpp, tiny_config
from _net import fake_score
from test_gpu_sampler import _golden_cfg


def test_state_dict_contract(golden_dir):
    """psld_b200.NCSNpp exposes exactly the reference's parameter names and shapes."""
    ref = json.load(open(f"{golden_dir}/state_dict_contract.json"))
    for name, cfg in (("tiny", tiny_config()),):
        mine = NCSNpp(cfg).state_dict()
        assert list(ref[name].keys()) == list(mine.keys())
        for k in ref[name]:
            assert tuple(ref[name][k]) == tuple(mine[k].shape), k


def test_forward_bit_exact(golden_dir):
    """The oracle forward is the reference forward op for op.  CPU convolutions partition their
    sums by thread count, so the oracle runs with the 8 threads the fixture was written with."""
    g = np.load(f"{golden_dir}/forward_tiny.npz")
    cfg = tiny_config()
    sd = fill_state_dict({k: tuple(v.shape) for k, v in NCSNpp(cfg).state_dict().items()}, int(g["seed"]))
    threads = torch.get_num_threads()
    torch.set_num_threads(8)
    try:
        y = O.ncsnpp_forward(cfg, sd, torch.from_numpy(g["x"]), torch.from_numpy(g["t"]))
    finally:
        torch.set_num_threads(threads)
    assert torch.equal(y, torch.from_numpy(g["y"]))


@pytest.mark.parametrize("kind", ["sscs_sde", "em_sde"])
def test_sampler(golden_dir, kind):
    """The reference's own SSCS / EM sampler with a stand-in score, step by step: per-step sum,
    |sum|, max|.| and sum of squares of the state, and the final samples."""
    tag = kind.split("_")[0] + "_fake_uniform"
    g = np.load(f"{golden_dir}/sampler_{tag}.npz")
    cfg = _golden_cfg(tag)
    ts, n = O.time_grid(cfg)
    B = int(g["B"])
    u0 = prior((B, 3, 8, 8), float(np.sqrt(O.PSLDScalars(cfg).m)), 1)
    nb = noise_bank((2 if kind == "sscs_sde" else 1) * n, (B, 6, 8, 8), 2)
    stats = []
    rec = lambda i, u: stats.append([u.sum().item(), u.abs().sum().item(), u.abs().max().item(),
                                     (u.double() ** 2).sum().item()])
    fn = O.sscs_sample if kind == "sscs_sde" else O.em_sample
    out = fn(cfg, fake_score, u0, ts, n, nb, record=rec)
    # 5e-7: the reference does its first step partly in fp32 (fp32 prior x python scalars), the
    # oracle promotes the prior to fp64 first (documented in oracle/psld_oracle.py)
    ref = torch.from_numpy(g["final"])
    assert (out - ref).abs().max() <= 5e-7 * ref.abs().max()
    got, want = np.asarray(stats), g["stats"]
    assert got.shape == want.shape
    assert np.all(np.abs(got[:, 0] - want[:, 0]) <= 5e-7 * want[:, 1])
    np.testing.assert_allclose(got[:, 1:], want[:, 1:], rtol=5e-7, atol=0)


def _reference_util():
    """The reference's registry (``main/util.py:33-62``): the ``_MODULES`` table holding the
    reference's own names, and ``get_module``."""
    util = types.ModuleType("util")
    util._MODULES = {"samplers": {"sscs_sde": type("SSCSSampler", (), {}),
                                  "em_sde": type("EulerMaruyamaSampler", (), {})},
                     "score_fn": {"ncsnpp": type("NCSNpp", (), {})}}

    def get_module(category, name):
        module = util._MODULES.get(category, dict()).get(name, None)
        if module is None:
            raise ValueError(f"No module named `{name}` found in category: `{category}`")
        return module

    util.get_module = get_module
    return util


def test_registry_install():
    """install() publishes the B200 classes into the reference registry (util.py:33-62)."""
    import psld_b200
    util = _reference_util()
    ref_sscs = util.get_module("samplers", "sscs_sde")
    psld_b200.install(util)
    assert util.get_module("samplers", "sscs_sde_b200") is psld_b200.SSCSSampler
    assert util.get_module("score_fn", "ncsnpp_b200") is psld_b200.NCSNpp
    assert util.get_module("samplers", "sscs_sde") is ref_sscs                  # no override
    psld_b200.install(util, override=True)
    assert util.get_module("samplers", "sscs_sde") is psld_b200.SSCSSampler
    assert util.get_module("score_fn", "ncsnpp") is psld_b200.NCSNpp
