"""Local-correlation prologue kernels alone: smooth vs random flow, tile-cooperative pass on / off (fp32 maps)."""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench

dev = torch.device("cuda:0")
out = {}
for mode in ("engine", "per_pixel", "tile_all"):
    out[mode] = bench.local_corr_flow_sweep(dev, "fp32", mode)
print(json.dumps(out))
for k, v in out.items():
    for kind, r in v.items():
        print(k, kind, "ms/pair", r["ms_per_pair"], "GB/s", r["hbm_gbs"], {a: b["ms"] for a, b in r["launches"].items()})
