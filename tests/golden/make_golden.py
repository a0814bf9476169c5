"""Generate the golden fixtures in this directory FROM THE UNMODIFIED REFERENCE.

Run from the repository root with a checkout of the original RoMa (the `romatch` package) on the path:

    PYTHONPATH=<RoMa checkout> PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py [fixture names]

The reference (`romatch.roma_outdoor`, model_zoo/__init__.py:31-61) is built on CPU (fp32,
`use_custom_corr=False` because the fused-local-corr wheel is absent) with the seeded synthetic weights of
`roma_b200.synthetic`, which load with strict=True, and run on seeded N(0,1) tensors / seeded PIL images.
Stage tensors are captured with forward hooks on the reference's own modules.  No fixture may exceed 1 MB, so
large tensors are stored sub-sampled: warp / certainty as `[:, ::step, ::step]` (step = meta[6]) together with
float64 checksums of the full tensor, and a stage tensor `key` [B, C, H, W] as `[:, ::c, ::s, ::s]` with
`key_step` = (c, s) from STAGE_STEP.  `sample()` of small_sym_up runs on the stored (sub-sampled) warp / certainty.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from roma_b200 import synthetic  # noqa: E402
from romatch import roma_indoor, roma_outdoor  # noqa: E402  (the reference)


# stage tensor -> (channel step, spatial step); the channel step of cls_and_cert divides 4096, so the certainty
# channel (index 4096) is the last one kept
STAGE_STEP = {"gp_mu": (4, 1), "cls_and_cert": (32, 1), "proj16": (4, 1), "proj8": (2, 3), "proj4": (4, 3), "proj2": (2, 3),
              "proj1": (1, 3), "delta16": (1, 1), "delta8": (1, 1), "delta4": (1, 1), "delta2": (1, 3), "delta1": (1, 3)}


def checksum(t):
    t = t.double()
    return np.array([t.sum().item(), t.abs().sum().item(), (t * t).sum().item()])


def run(name, coarse, up, symmetric=True, upsample_preds=True, batch=1, seed=1, step=1, hooks=True, pil=False, factory=roma_outdoor):
    mw, dw = synthetic.make_weights(0)
    model = factory("cpu", weights=mw, dinov2_weights=dw, coarse_res=coarse,
                         upsample_res=up if up else coarse, symmetric=symmetric,
                         upsample_preds=upsample_preds, use_custom_corr=False)
    out = {}
    handles = []
    if hooks:
        dec = model.decoder

        def save(key):
            def fn(mod, inp, res):
                res = res if isinstance(res, torch.Tensor) else torch.cat([r for r in res if r is not None], 1)
                out.setdefault(key, res.detach().clone().numpy())     # first call = coarse pass
            return fn
        handles.append(dec.gps["16"].register_forward_hook(save("gp_mu")))
        handles.append(dec.embedding_decoder.register_forward_hook(save("cls_and_cert")))
        for s in ("16", "8", "4", "2", "1"):
            handles.append(dec.conv_refiner[s].register_forward_hook(save(f"delta{s}")))
            handles.append(dec.proj[s].register_forward_hook(save(f"proj{s}")))
    if pil:
        from PIL import Image
        a, b = synthetic.make_pil_pair(seed)
        warp, cert = model.match(a, b)
    else:
        A, B, Ah, Bh = synthetic.make_pair(batch, coarse, up if upsample_preds else None, seed)
        warp, cert = model.match(A, B, im_A_high_res=Ah, im_B_high_res=Bh)
    for h in handles:
        h.remove()
    for key, (c, s) in STAGE_STEP.items():
        if key in out:
            out[key] = np.ascontiguousarray(out[key][:, ::c, ::s, ::s])
            out[f"{key}_step"] = np.array([c, s])
    out["warp"] = warp[:, ::step, ::step].numpy()
    out["certainty"] = cert[:, ::step, ::step].numpy()
    out["warp_checksum"] = checksum(warp)
    out["certainty_checksum"] = checksum(cert)
    if isinstance(coarse, tuple):          # rectangular resolutions: (h, w) pairs
        out["res"] = np.array([*coarse, *(up or (0, 0))])
        out["meta"] = np.array([0, 0, int(symmetric), int(upsample_preds), batch, seed, step])
    else:
        out["meta"] = np.array([coarse, up or 0, int(symmetric), int(upsample_preds), batch, seed, step])
    if name == "small_sym_up":
        torch.manual_seed(123)
        m, c = model.sample(torch.from_numpy(out["warp"][0]), torch.from_numpy(out["certainty"][0]), num=500)
        out["sample_matches"], out["sample_certainty"] = m.numpy(), c.numpy()
    np.savez_compressed(os.path.join(HERE, f"{name}.npz"), **out)
    print(name, {k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    torch.set_num_threads(8)
    only = set(sys.argv[1:])                 # optional: names of the fixtures to (re)generate

    if only:
        _run, run = run, (lambda name, *a, **k: _run(name, *a, **k) if name in only else None)
    run("small_sym_up", 112, 168, step=3)
    run("small_nosym_up", 112, 168, symmetric=False, hooks=False)
    run("small_sym_noup", 112, None, upsample_preds=False, hooks=False)
    run("small_b2_sym_up", 112, 168, batch=2, seed=7, step=3, hooks=False)
    run("small_pil_sym_up", 112, 168, pil=True, hooks=False, seed=3)
    run("rect_sym_up", (112, 168), (168, 224), hooks=False, seed=5)
    run("full_sym_up", 560, 864, step=8, hooks=False)
    run("full_nosym_up", 560, 864, symmetric=False, step=8, hooks=False, seed=2)
    run("small_indoor_sym_up", 112, 168, hooks=False, seed=9, factory=roma_indoor)
