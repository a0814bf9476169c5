"""Pin the CPU oracle against outputs of the unmodified reference (tests/golden/*.npz).

The fixtures were produced by `tests/golden/make_golden.py` from `/root/reference` with the seeded
synthetic weights; the oracle must reproduce them (it is bit-exact in the build container; the
tolerance below allows for a different BLAS/thread count on another host).
"""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle.roma_oracle import RomaOracle
from roma_b200 import synthetic
from roma_b200.preprocess import pil_to_normalized

TOL = 2e-5


def _oracle(weights, g):
    coarse, up, sym, upp = (int(v) for v in g["meta"][:4])
    return RomaOracle(weights[0], weights[1], coarse, up or coarse, symmetric=bool(sym), upsample_preds=bool(upp))


def _check(warp, cert, g):
    """Max-abs error on the golden's pixels (every meta[6]-th row and column); over the whole tensors, the mean errors of the
    sum and the absolute sum (float64 checksums in the golden), which the max-abs error over all pixels bounds."""
    step = int(g["meta"][6])
    w = warp[:, ::step, ::step].numpy()
    c = cert[:, ::step, ::step].numpy()
    assert w.shape == g["warp"].shape and c.shape == g["certainty"].shape
    assert np.abs(w - g["warp"]).max() <= TOL
    assert np.abs(c - g["certainty"]).max() <= TOL
    for t, key in ((warp, "warp_checksum"), (cert, "certainty_checksum")):
        t = t.double()
        assert abs(t.sum().item() - g[key][0]) <= TOL * t.numel() and abs(t.abs().sum().item() - g[key][1]) <= TOL * t.numel()


def _stage(t, g, key):
    """The golden's subset of stage tensor `key` [B, C, H, W] (channel / spatial steps in `key_step`)."""
    c, s = (int(v) for v in g[f"{key}_step"])
    return t[:, ::c, ::s, ::s].numpy()


@pytest.mark.parametrize("name", ["small_sym_up", "small_nosym_up", "small_sym_noup", "small_b2_sym_up"])
def test_oracle_matches_reference_small(weights, name):
    g = load_golden(name)
    coarse, up, sym, upp, batch, seed, step = (int(v) for v in g["meta"])
    orc = _oracle(weights, g)
    A, B, Ah, Bh = synthetic.make_pair(batch, coarse, up if upp else None, seed)
    warp, cert = orc.match(A, B, Ah, Bh)
    h = up if upp else coarse
    assert warp.shape == (batch, h, h * (2 if sym else 1), 4) and cert.shape == warp.shape[:3]
    _check(warp, cert, g)
    assert warp.dtype == torch.float32 and cert.dtype == torch.float32


def test_oracle_matches_reference_rectangular(weights):
    """Non-square resolutions (112 x 168 -> 168 x 224): h and w differ in every grid, window and displacement scale."""
    g = load_golden("rect_sym_up")
    ch, cw, uh, uw = (int(v) for v in g["res"])
    orc = RomaOracle(weights[0], weights[1], (ch, cw), (uh, uw), symmetric=True, upsample_preds=True)
    A, B, Ah, Bh = synthetic.make_pair(1, (ch, cw), (uh, uw), int(g["meta"][5]))
    warp, cert = orc.match(A, B, Ah, Bh)
    _check(warp, cert, g)


def test_oracle_stage_tensors(weights):
    g = load_golden("small_sym_up")
    orc = _oracle(weights, g)
    orc.trace = {}
    A, B, Ah, Bh = synthetic.make_pair(1, 112, 168, 1)
    orc.match(A, B, Ah, Bh)
    t = orc.trace
    assert np.abs(_stage(t["gp.mu"], g, "gp_mu") - g["gp_mu"]).max() <= TOL
    # the kept classes are those of cls_and_cert but its last (certainty) channel
    assert np.abs(_stage(t["cls"], g, "cls_and_cert") - g["cls_and_cert"][:, :-1]).max() <= 1e-3     # logits are O(40)
    for s in (16, 8, 4, 2, 1):
        assert np.abs(_stage(t[f"lo.delta{s}"], g, f"delta{s}") - g[f"delta{s}"]).max() <= TOL * 10
        assert np.abs(_stage(t[f"lo.proj{s}.x"], g, f"proj{s}") - g[f"proj{s}"]).max() <= TOL


def test_oracle_pil_route(weights):
    """PIL inputs: host preprocessing of this repo + oracle == reference `match(PIL, PIL)`."""
    g = load_golden("small_pil_sym_up")
    coarse, up = int(g["meta"][0]), int(g["meta"][1])
    a, b = synthetic.make_pil_pair(int(g["meta"][5]))
    orc = _oracle(weights, g)
    A, B = pil_to_normalized(a, (coarse, coarse))[None], pil_to_normalized(b, (coarse, coarse))[None]
    Ah, Bh = pil_to_normalized(a, (up, up))[None], pil_to_normalized(b, (up, up))[None]
    warp, cert = orc.match(A, B, Ah, Bh)
    _check(warp, cert, g)


def test_oracle_sample_matches_reference(weights):
    g = load_golden("small_sym_up")
    orc = _oracle(weights, g)
    warp = torch.from_numpy(g["warp"])
    cert = torch.from_numpy(g["certainty"])
    torch.manual_seed(123)
    m, c = orc.sample(warp[0], cert[0], num=500)
    assert np.array_equal(m.numpy(), g["sample_matches"])
    assert np.array_equal(c.numpy(), g["sample_certainty"])


@pytest.mark.slow
def test_oracle_matches_reference_full(weights):
    """560 -> 864, the BASELINE.json config-2 workload (sub-sampled golden + full-tensor checksums)."""
    g = load_golden("full_sym_up")
    orc = _oracle(weights, g)
    A, B, Ah, Bh = synthetic.make_pair(1, 560, 864, 1)
    warp, cert = orc.match(A, B, Ah, Bh)
    _check(warp, cert, g)
    assert abs(warp.double().sum().item() - g["warp_checksum"][0]) <= 1e-3 * max(1.0, abs(g["warp_checksum"][0]))
    assert abs(cert.double().abs().sum().item() - g["certainty_checksum"][1]) <= 1e-4 * g["certainty_checksum"][1]
