"""CPU dry run of the engine in the parity mode: the stride-2 (C = 144) refiner blocks go through the fused
romab200_refiner_block_c144 with fp32 maps and the split weight planes, in place of the depthwise kernel + GEMM pair, and
nothing changes for the other widths or with the fused path switched off."""
import pytest
import torch

from roma_b200 import cabi, synthetic
from roma_b200.packing import PackedWeights

from test_host_logic import _Recorder, _tensors


def _dry_run(weights, monkeypatch, split, fused_c144_f32):
    import roma_b200.engine as engine_mod
    rec = _Recorder()
    log = []

    def record(fn, struct, **kw):
        rec(fn, struct, **kw)
        log.append((fn, kw))
    eng = engine_mod.Engine.__new__(engine_mod.Engine)
    eng.device = torch.device("cpu")
    eng.precision, eng.dtype, eng.dt = "fp32" if split else "fp32_simt", torch.float32, cabi.RB_F32
    eng.split, eng._lane, eng.generation = split, "main", 0
    eng.w = PackedWeights(weights[0], weights[1], eng.device, torch.float32, split=split)
    eng._buf, eng._const, eng.debug, eng.profile, eng.gemm_profile, eng.use_flash_attn, eng.gp_algo = {}, {}, None, None, None, True, (3 if split else 2)
    eng.overlap_cnn, eng._side, eng.gp_tensor_core, eng.fused_c144, eng.fused_small_f32 = False, None, True, True, True
    eng.lc_table16, eng.lc_tile_radii, eng.side_ctas = True, (2,), 0
    eng.fused_c144_f32 = fused_c144_f32
    for t in _tensors(eng.w):
        rec.track(t)
    orig_buf, orig_const = eng.buf, eng.const

    def buf(*a, **k):
        t = orig_buf(*a, **k); rec.track(t); return t

    def const(*a, **k):
        t = orig_const(*a, **k); rec.track(t); return t
    eng.buf, eng.const = buf, const
    monkeypatch.setattr(engine_mod, "call", record)
    A, B, Ah, Bh = synthetic.make_pair(1, 112, 168, 1)
    images = torch.cat((A, B)); rec.track(images)
    state, _, _ = eng.run_pass(images, 1, True, False, 112 / 560)
    hi = torch.cat((Ah, Bh)); rec.track(hi)
    eng.run_pass(hi, 1, True, True, 168 / 560, (state, 112, 112))
    return log


def _by_width(log):
    fused = [kw for fn, kw in log if fn == "romab200_refiner_block_c144"]
    dw = {}
    for fn, kw in log:
        if fn == "romab200_dwconv5x5_relu":
            dw[kw["c"]] = dw.get(kw["c"], 0) + 1
    pw = {}
    for fn, kw in log:
        if fn == "romab200_gemm" and kw["M"] > 0 and kw["N"] == kw["K"] and kw["N"] in (144, 569, 1137, 1377):
            pw[kw["N"]] = pw.get(kw["N"], 0) + 1
    return fused, dw, pw


@pytest.mark.parametrize("fused_c144_f32", [True, False])
def test_parity_mode_c144_blocks(weights, monkeypatch, fused_c144_f32):
    fused, dw, pw = _by_width(_dry_run(weights, monkeypatch, True, fused_c144_f32))
    # stride 2 is refined once per pass (coarse and upsample), 9 blocks each
    if fused_c144_f32:
        assert len(fused) == 18 and 144 not in dw and 144 not in pw
        for kw in fused:
            assert kw["dtype"] == cabi.RB_F32 and kw["c"] == 144
            assert kw["in"] is not kw["out"] and kw["in"].dtype == kw["out"].dtype == torch.float32
            assert kw["pw_weight"].dtype == kw["pw_weight_lo"].dtype == torch.float16
        # the blocks ping-pong between two maps
        assert all(a["out"] is b["in"] for a, b in zip(fused[:8], fused[1:9]))
    else:
        assert not fused and dw[144] == 18
    # the wide maps keep the depthwise kernel + split GEMM pair; the stride-1 maps keep their own fused kernel
    assert dw[569] == 18 and dw[1137] == 18 and dw[1377] == 9


def test_simt_backend_keeps_unfused_c144(weights, monkeypatch):
    fused, dw, _ = _by_width(_dry_run(weights, monkeypatch, False, True))
    assert not fused and dw[144] == 18
