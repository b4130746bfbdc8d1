#!/bin/bash
# Fused update with in-kernel Box-Muller noise, float32 state, timed alone at B=256 and at 2^24 pairs
# (share of the measured HBM copy bandwidth)
cd "$(dirname "$0")/.."
python - <<'PY'
import torch, json
import bench
from psld_b200 import NCSNpp, PSLD, cifar10_config, time_grid, _lib as L
cfg = cifar10_config(); sde = PSLD(cfg); ts, n = time_grid(cfg)
dev = torch.device("cuda", 0)
class P: pass
B, chw = 256, 3072
plan = P(); plan.x_in = torch.empty(B, 6, 32, 32, device=dev); plan.eps = torch.randn(B, 6, 32, 32, device=dev)
state = torch.randn(B, 6, 32, 32, device=dev)
r = bench.time_update(L.lib(), state, plan, B, chw, L.stream_ptr(dev), dev, torch.float32, sde, ts)
pk = bench.peaks()["hbm"]
print("B=256:", round(r["achieved"] / pk, 3), " 2^24 pairs:", round(r["large"]["achieved"] / pk, 3), round(r["large"]["avg_launch_ms"], 4), "ms")
PY
