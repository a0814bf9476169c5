"""End-to-end parity of the CUDA path (fp32 parity mode) against the CPU oracle and the golden fixtures
made from the unmodified reference.  North-star tolerance: 1e-4 max-abs on warp and certainty."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from conftest import load_golden  # noqa: E402
from roma_b200 import synthetic  # noqa: E402

TOL = 1e-4


BACKENDS = ["tcgen05", "simt"]       # GEMM back-ends of the fp32 parity mode: split-fp16 pairs on the tensor cores / CUDA-core FFMA


def build(weights, g, amp_dtype=torch.float32, backend="tcgen05"):
    from roma_b200 import model_zoo, roma_outdoor
    coarse, up, sym, upp = (int(v) for v in g["meta"][:4])
    model_zoo.fp32_backend = backend
    try:
        m = roma_outdoor("cuda", weights=weights[0], dinov2_weights=weights[1], coarse_res=coarse,
                         upsample_res=up or coarse, symmetric=bool(sym), upsample_preds=bool(upp), amp_dtype=amp_dtype)
    finally:
        model_zoo.fp32_backend = None
    if amp_dtype == torch.float32:
        assert m.engine.precision == ("fp32" if backend == "tcgen05" else "fp32_simt")
    return m


def mean_error(t, checksum):
    """Mean error of the sum and of the absolute sum of the whole tensor against the golden's float64 checksums: bounded
    by the max-abs error over all pixels, so it also covers the pixels the golden does not store."""
    t = t.double()
    return max(abs(t.sum().item() - checksum[0]), abs(t.abs().sum().item() - checksum[1])) / t.numel()


def report(name, warp, cert, g):
    """Max-abs errors on the golden's pixels (every meta[6]-th row and column), or the larger mean_error."""
    step = int(g["meta"][6])
    w = warp[:, ::step, ::step].float().cpu().numpy()
    c = cert[:, ::step, ::step].float().cpu().numpy()
    assert w.shape == g["warp"].shape and c.shape == g["certainty"].shape
    ew = max(np.abs(w - g["warp"]).max(), mean_error(warp, g["warp_checksum"]))
    ec = max(np.abs(c - g["certainty"]).max(), mean_error(cert, g["certainty_checksum"]))
    print(f"[{name}] warp max-abs err {ew:.3e}  certainty max-abs err {ec:.3e}")
    return ew, ec


def stage(t, g, key):
    """The golden's subset of stage tensor `key` [B, C, H, W] (channel / spatial steps in `key_step`)."""
    c, s = (int(v) for v in g[f"{key}_step"])
    return t[:, ::c, ::s, ::s]


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("name", ["small_sym_up", "small_nosym_up", "small_sym_noup", "small_b2_sym_up"])
def test_match_small_vs_reference_golden(weights, name, backend):
    g = load_golden(name)
    coarse, up, sym, upp, batch, seed, step = (int(v) for v in g["meta"])
    model = build(weights, g, backend=backend)
    A, B, Ah, Bh = synthetic.make_pair(batch, coarse, up if upp else None, seed)
    warp, cert = model.match(A.cuda(), B.cuda(), im_A_high_res=None if Ah is None else Ah.cuda(),
                             im_B_high_res=None if Bh is None else Bh.cuda())
    h = up if upp else coarse
    assert warp.shape == (batch, h, h * (2 if sym else 1), 4) and cert.shape == warp.shape[:3]
    assert warp.dtype == torch.float32 and cert.dtype == torch.float32 and warp.is_cuda
    ew, ec = report(name, warp, cert, g)
    assert ew <= TOL and ec <= TOL


@pytest.mark.parametrize("backend", BACKENDS)
def test_match_rectangular_vs_reference_golden(weights, backend):
    """Non-square resolutions (112 x 168 -> 168 x 224) against the unmodified reference."""
    from roma_b200 import model_zoo, roma_outdoor
    g = load_golden("rect_sym_up")
    ch, cw, uh, uw = (int(v) for v in g["res"])
    model_zoo.fp32_backend = backend
    try:
        model = roma_outdoor("cuda", weights=weights[0], dinov2_weights=weights[1], coarse_res=(ch, cw), upsample_res=(uh, uw), amp_dtype=torch.float32)
    finally:
        model_zoo.fp32_backend = None
    A, B, Ah, Bh = synthetic.make_pair(1, (ch, cw), (uh, uw), int(g["meta"][5]))
    warp, cert = model.match(A.cuda(), B.cuda(), im_A_high_res=Ah.cuda(), im_B_high_res=Bh.cuda())
    ew, ec = report(f"rect {backend}", warp, cert, g)
    assert ew <= TOL and ec <= TOL


@pytest.mark.parametrize("backend", BACKENDS)
def test_stagewise_vs_reference_hooks(weights, backend):
    """Stage tensors of the coarse pass against the tensors hooked out of the reference's own modules."""
    g = load_golden("small_sym_up")
    model = build(weights, g, backend=backend)
    model.engine.debug = {}
    A, B, Ah, Bh = synthetic.make_pair(1, 112, 168, 1)
    model.match(A.cuda(), B.cuda(), im_A_high_res=Ah.cuda(), im_B_high_res=Bh.cuda())
    dbg = model.engine.debug
    model.engine.debug = None

    def err(ours, key):
        return float((stage(ours, g, key).float().cpu() - torch.from_numpy(g[key])).abs().max())
    errs = {}
    for s in (16, 8, 4, 2, 1):
        errs[f"proj{s}"] = err(dbg[f"lo.proj{s}"].permute(0, 3, 1, 2), f"proj{s}")
        errs[f"delta{s}"] = err(dbg[f"lo{s}.delta"].permute(0, 3, 1, 2), f"delta{s}")
    errs["gp_mu"] = err(dbg["gp.mu"].transpose(1, 2).reshape(2, 512, 8, 8), "gp_mu")
    errs["cls"] = err(dbg["cls"].transpose(1, 2).reshape(2, 4097, 8, 8), "cls_and_cert")
    print({k: f"{v:.2e}" for k, v in errs.items()})
    assert errs["proj16"] < 2e-4 and errs["gp_mu"] < 1e-4 and errs["cls"] < 5e-3
    for s in (16, 8, 4, 2, 1):
        assert errs[f"proj{s}"] < 2e-4 and errs[f"delta{s}"] < 2e-3, (s, errs)


def test_match_pil_route(weights):
    g = load_golden("small_pil_sym_up")
    model = build(weights, g)
    a, b = synthetic.make_pil_pair(int(g["meta"][5]))
    warp, cert = model.match(a, b)
    ew, ec = report("pil", warp, cert, g)
    assert ew <= TOL and ec <= TOL


def test_api_errors_and_forward(weights):
    g = load_golden("small_sym_up")
    model = build(weights, g)
    A, B, Ah, Bh = synthetic.make_pair(1, 112, 168, 1)
    with pytest.raises(ValueError):
        model.match(A.cuda(), B.cuda(), batched=False)
    with pytest.raises(AssertionError):
        model.match(torch.zeros(1, 3, 100, 112).cuda(), B.cuda())
    with pytest.raises(AssertionError):          # tensors + upsample_preds need *_high_res (matcher.py:863-866)
        model.match(A.cuda(), B.cuda())
    with pytest.raises(ValueError):
        model.match(A.cuda(), B.cuda(), im_A_high_res=Ah.cuda())
    with pytest.raises(ValueError):          # mixed input types (matcher.py:828)
        model.match(A.cuda(), synthetic.make_pil_pair(3)[0])
    corr = model.forward_symmetric({"im_A": A.cuda(), "im_B": B.cuda()}, scale_factor=112 / 560)
    assert sorted(corr) == [1, 2, 4, 8, 16]
    assert corr[1]["flow"].shape == (2, 2, 112, 112) and corr[16]["certainty"].shape == (2, 1, 8, 8)
    model.symmetric = False
    model.upsample_preds = False
    warp, cert = model.match(A.cuda(), B.cuda(), 1, 2, 3)     # extra positional args are ignored
    assert warp.shape == (1, 112, 112, 4) and cert.shape == (1, 112, 112)
    assert model.get_output_resolution() == (112, 112)
    kp = model.to_pixel_coordinates(warp[0, :2, :2], 100, 200, 300, 400)
    assert kp[0].shape == (2, 2, 2)


def test_sample_statistics(weights):
    """sample(): shapes, membership in the warp and certainty thresholding, for the device sampler and the torch.multinomial route
    (the distribution itself is compared with the oracle in test_sample_distribution_vs_oracle)."""
    g = load_golden("small_sym_up")
    model = build(weights, g)
    warp = torch.from_numpy(g["warp"]).cuda()
    cert = torch.from_numpy(g["certainty"]).cuda()
    rows = {tuple(r) for r in warp[0].reshape(-1, 4).cpu().numpy().view("uint32").tolist()}
    for device_sampler in (True, False):
        model.device_sampler = device_sampler
        torch.manual_seed(0)
        m, c = model.sample(warp[0], cert[0], num=500)
        assert m.shape == (500, 4) and c.shape == (500,)
        # every sampled match is (bit-exactly) a row of the warp
        assert all(tuple(r) in rows for r in m.cpu().numpy().view("uint32").tolist())
        assert ((c == 1) | (c <= model.sample_thresh)).all()
        torch.manual_seed(0)
        m2, _ = model.sample(warp[0], cert[0], num=500)
        assert torch.equal(m2, m) or not device_sampler          # the device sampler is reproducible under torch.manual_seed


def test_sample_distribution_vs_oracle(weights):
    """Acceptance test of the device-side sampler (SURVEY 8f-1): RNG-stream parity with torch is impossible, so the sampled-match
    distribution of `model.sample` is compared with the oracle's `sample` (the reference's algorithm: two torch.multinomial draws
    around the fp16 KDE) over 60 seeds each: two-sample Kolmogorov-Smirnov on every coordinate and on the certainty, a chi-square
    test on a 6 x 6 histogram of the query position, and the agreement of the `density < 10` mask on a fixed first draw."""
    from scipy import stats
    from oracle.roma_oracle import RomaOracle
    g = load_golden("small_sym_up")
    model = build(weights, g)
    orc = RomaOracle(weights[0], weights[1], 112, 168)
    warp, cert = torch.from_numpy(g["warp"])[0], torch.from_numpy(g["certainty"])[0]
    wd, cd = warp.cuda(), cert.cuda()
    ours, ref = [], []
    for seed in range(60):
        torch.manual_seed(1000 + seed)
        m, c = model.sample(wd, cd, num=400)
        assert m.shape == (400, 4) and c.shape == (400,)
        ours.append(torch.cat((m, c[:, None]), 1).cpu())
        torch.manual_seed(5000 + seed)
        m, c = orc.sample(warp, cert, num=400)
        ref.append(torch.cat((m, c[:, None].float()), 1))
    ours, ref = torch.cat(ours).numpy(), torch.cat(ref).numpy()
    rows = {tuple(r) for r in warp.reshape(-1, 4).numpy().view("uint32").tolist()}
    assert all(tuple(r) in rows for r in np.ascontiguousarray(ours[:, :4]).view("uint32").tolist())      # every sample is a row of the warp
    for j in range(5):
        p = stats.ks_2samp(ours[:, j], ref[:, j]).pvalue
        assert p > 1e-3, (j, p)
    bins = np.linspace(-1, 1, 7)
    h_o, _, _ = np.histogram2d(ours[:, 0], ours[:, 1], bins=(bins, bins))
    h_r, _, _ = np.histogram2d(ref[:, 0], ref[:, 1], bins=(bins, bins))
    keep = (h_o + h_r) > 20
    chi2 = stats.chi2_contingency(np.stack((h_o[keep], h_r[keep])))
    assert chi2[1] > 1e-3, chi2[1]
    # density mask: the same first draw through both KDE implementations
    torch.manual_seed(7)
    good = warp.reshape(-1, 4)[torch.multinomial((cert.reshape(-1) > 0.05).float() + cert.reshape(-1) * (cert.reshape(-1) <= 0.05), 1600)]
    d_ref = RomaOracle.kde(good)
    d_ours = model.engine.kde(good.cuda(), std=0.1, half=True).to(torch.float16).cpu()
    mismatch = ((d_ref < 10) != (d_ours < 10)).float().mean().item()
    assert mismatch <= 2e-3, mismatch


@pytest.mark.slow
@pytest.mark.parametrize("backend", BACKENDS)
def test_match_full_vs_reference_golden(weights, backend):
    """560 -> 864 (BASELINE config 2 workload) against the sub-sampled reference output, for both GEMM back-ends of the
    parity mode; "tcgen05" (split-fp16 operand pairs on the tensor cores) is the mode bench.py reports."""
    g = load_golden("full_sym_up")
    model = build(weights, g, backend=backend)
    A, B, Ah, Bh = synthetic.make_pair(1, 560, 864, 1)
    warp, cert = model.match(A.cuda(), B.cuda(), im_A_high_res=Ah.cuda(), im_B_high_res=Bh.cuda())
    assert warp.shape == (1, 864, 1728, 4)
    ew, ec = report(f"full {backend}", warp, cert, g)
    assert ew <= TOL and ec <= TOL
    model.free_buffers()


@pytest.mark.slow
def test_match_full_one_direction_vs_reference_golden(weights):
    """560 -> 864 with symmetric=False (one-directional warp, `forward` instead of `forward_symmetric`, matcher.py:831-834)."""
    g = load_golden("full_nosym_up")
    model = build(weights, g)
    A, B, Ah, Bh = synthetic.make_pair(1, 560, 864, int(g["meta"][5]))
    warp, cert = model.match(A.cuda(), B.cuda(), im_A_high_res=Ah.cuda(), im_B_high_res=Bh.cuda())
    assert warp.shape == (1, 864, 864, 4)
    ew, ec = report("full one-direction", warp, cert, g)
    assert ew <= TOL and ec <= TOL
    model.free_buffers()


def test_roma_indoor_vs_reference_golden(weights):
    """`roma_indoor` (BASELINE config 4's factory, model_zoo/__init__.py:64-94) against the reference's roma_indoor."""
    from roma_b200 import roma_indoor
    g = load_golden("small_indoor_sym_up")
    coarse, up, sym, upp, batch, seed, step = (int(v) for v in g["meta"])
    model = roma_indoor("cuda", weights=weights[0], dinov2_weights=weights[1], coarse_res=coarse, upsample_res=up, amp_dtype=torch.float32)
    A, B, Ah, Bh = synthetic.make_pair(batch, coarse, up, seed)
    warp, cert = model.match(A.cuda(), B.cuda(), im_A_high_res=Ah.cuda(), im_B_high_res=Bh.cuda())
    ew, ec = report("indoor", warp, cert, g)
    assert ew <= TOL and ec <= TOL


@pytest.mark.parametrize("amp", [torch.float16, torch.bfloat16])
def test_match_fast_mode_small(weights, amp):
    """16-bit tensor-core mode (the reference's CUDA autocast regime).  Two fp16 implementations do not agree to
    1e-4 end to end (argmax flips of the coarse classifier move single pixels by a whole anchor, SURVEY §7.2), so
    the bar here is statistical: the bulk of the warp agrees closely and outliers are rare."""
    g = load_golden("small_sym_up")
    model = build(weights, g, amp_dtype=amp)
    A, B, Ah, Bh = synthetic.make_pair(1, 112, 168, 1)
    warp, cert = model.match(A.cuda(), B.cuda(), im_A_high_res=Ah.cuda(), im_B_high_res=Bh.cuda())
    step = int(g["meta"][6])
    ew = np.abs(warp[:, ::step, ::step].cpu().numpy() - g["warp"]).max(-1)
    ec = np.abs(cert[:, ::step, ::step].cpu().numpy() - g["certainty"])
    print(f"[fast {amp}] warp err: median {np.median(ew):.2e} p99 {np.percentile(ew, 99):.2e} max {ew.max():.2e} "
          f"frac>1e-2 {np.mean(ew > 1e-2):.4f}; cert err median {np.median(ec):.2e} max {ec.max():.2e}")
    assert np.isfinite(ew).all() and np.isfinite(ec).all()
    tol_med = 2e-3 if amp == torch.float16 else 1e-2
    assert np.median(ew) < tol_med and np.mean(ew > 5e-2) < 0.05


@pytest.mark.slow
def test_match_fast_mode_full(weights):
    """fp16 tensor-core mode at 560 -> 864 against the reference golden (sub-sampled)."""
    g = load_golden("full_sym_up")
    model = build(weights, g, amp_dtype=torch.float16)
    A, B, Ah, Bh = synthetic.make_pair(1, 560, 864, 1)
    warp, cert = model.match(A.cuda(), B.cuda(), im_A_high_res=Ah.cuda(), im_B_high_res=Bh.cuda())
    ew = np.abs(warp[:, ::8, ::8].cpu().numpy() - g["warp"]).max(-1)
    ec = np.abs(cert[:, ::8, ::8].cpu().numpy() - g["certainty"])
    print(f"[fast fp16 full] warp err: median {np.median(ew):.2e} p99 {np.percentile(ew, 99):.2e} max {ew.max():.2e} "
          f"frac>1e-3 {np.mean(ew > 1e-3):.4f}; cert err median {np.median(ec):.2e} p99 {np.percentile(ec, 99):.2e} max {ec.max():.2e}")
    assert np.median(ew) < 1e-3 and np.mean(ew > 5e-2) < 0.05
    model.free_buffers()


@pytest.mark.parametrize("amp,backend", [(torch.float32, "tcgen05"), (torch.float32, "simt"), (torch.float16, "tcgen05")])
def test_repeated_calls_and_cuda_graph_replay(weights, amp, backend):
    """Callers (and bench.py) use the path behind the first call: call 2 re-uses zero-initialised buffers that now hold
    stale data, call 3+ replays the captured CUDA graph (PDL edges, side-stream fork/join, baked-in tensor maps).  Ten
    calls alternating two input shapes and fresh inputs must equal an eager model (use_cuda_graph=False) exactly, and the
    fp32 modes must stay on the goldens; free_buffers() between calls must not leave a graph pointing at freed memory."""
    g = load_golden("small_sym_up")
    graph_model = build(weights, g, amp_dtype=amp, backend=backend)
    eager_model = build(weights, g, amp_dtype=amp, backend=backend)
    eager_model.use_cuda_graph = False
    shapes = [(112, 168), (168, 224)]
    for call_idx in range(10):
        coarse, up = shapes[call_idx % 2]
        seed = 1 if call_idx in (4, 8) else 10 + call_idx        # call 4: graph replay of the golden input; call 8: re-capture after free_buffers()
        A, B, Ah, Bh = synthetic.make_pair(1, coarse, up, seed)
        for m in (graph_model, eager_model):
            m.upsample_res = (up, up)
            m.h_resized = m.w_resized = coarse
        args = (A.cuda(), B.cuda())
        kw = dict(im_A_high_res=Ah.cuda(), im_B_high_res=Bh.cuda())
        w1, c1 = graph_model.match(*args, **kw)
        w2, c2 = eager_model.match(*args, **kw)
        assert torch.isfinite(w1).all() and torch.isfinite(c1).all()
        dw, dc = (w1 - w2).abs().max().item(), (c1 - c2).abs().max().item()
        assert dw <= 1e-6 and dc <= 1e-6, (call_idx, dw, dc)
        if seed == 1 and coarse == 112 and amp == torch.float32:
            ew, ec = report(f"call {call_idx}", w1, c1, g)
            assert ew <= TOL and ec <= TOL
        if call_idx == 5:
            graph_model.engine.free_buffers()        # what user code can do: graphs recorded so far must not be replayed
    assert any(e["graph"] is not None for e in graph_model._graphs.values())
