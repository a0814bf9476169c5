"""Per-kernel launch list of one eager match() 560 -> 864 (symmetric pair) under torch.profiler (CUDA activities), in the
format of scripts/launch_table.py.

    python scripts/launches_torch_profiler.py [fp32|fp16|bf16] > launches.txt
"""
import collections
import os
import re
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from torch.profiler import ProfilerActivity, profile

from roma_b200 import roma_outdoor, synthetic

prec = sys.argv[1] if len(sys.argv) > 1 else "fp32"
amp = {"fp16": torch.float16, "bf16": torch.bfloat16, "fp32": torch.float32}[prec]
mw, dw = synthetic.make_weights(0)
model = roma_outdoor("cuda", weights=mw, dinov2_weights=dw, amp_dtype=amp)
model.use_cuda_graph = False
A, B, Ah, Bh = [t.cuda() for t in synthetic.make_pair(1, 560, 864, 1)]
for _ in range(2):
    model.match(A, B, im_A_high_res=Ah, im_B_high_res=Bh)
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    model.match(A, B, im_A_high_res=Ah, im_B_high_res=Bh)
    torch.cuda.synchronize()
agg = collections.defaultdict(lambda: [0, 0.0])
for e in prof.events():
    if e.device_type != torch.autograd.DeviceType.CUDA or "memcpy" in e.name.lower() or "memset" in e.name.lower():
        continue
    name = re.sub(r"\(.*", "", e.name).replace("void rb::", "void ").replace("rb::", "")
    agg[name][0] += 1
    agg[name][1] += e.time_range.elapsed_us()
tot = sum(t for _, t in agg.values())
print(f"{torch.cuda.get_device_name()}, {prec}: total {tot / 1e3:.2f} ms over {sum(n for n, _ in agg.values())} launches (torch.profiler, kernels serialised per stream)")
for k, (n, t) in sorted(agg.items(), key=lambda kv: -kv[1][1])[:40]:
    print(f"{t:10.1f} us {100 * t / tot:5.1f}%  n={n:5d} avg={t / n:8.1f}  {k}")
