"""CPU tests of the host side: C-ABI library loads and exports what the header declares, weight packing
(BN folding) is right, and a dry run of the whole engine with a recording fake of `cabi.call` checks every
kernel call's argument names, dtypes and that every pointer range stays inside an allocated buffer."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from roma_b200 import arch, cabi, synthetic
from roma_b200.packing import PackedWeights, fold_bn, pad8


def test_library_exports_every_declared_symbol():
    lib = cabi.load_library()
    assert lib.romab200_abi_version() == 4
    assert len(cabi.FUNCTIONS) >= 20
    for fn in cabi.FUNCTIONS:
        assert hasattr(lib, fn), fn
    assert ctypes.sizeof(cabi.STRUCTS["rb_gemm_args"]) == 368


def test_fold_bn_matches_batchnorm(weights):
    sd = weights[0]
    x = torch.randn(2, 64, 9, 9)
    w, b = sd["encoder.cnn.layers.3.weight"], sd["encoder.cnn.layers.3.bias"]
    ref = F.batch_norm(F.conv2d(x, w, b, padding=1), sd["encoder.cnn.layers.4.running_mean"], sd["encoder.cnn.layers.4.running_var"],
                       sd["encoder.cnn.layers.4.weight"], sd["encoder.cnn.layers.4.bias"], False, 0.0, 1e-5)
    w2, b2 = fold_bn(w, b, sd, "encoder.cnn.layers.4")
    assert (F.conv2d(x, w2, b2, padding=1) - ref).abs().max() < 2e-5


def test_packing_layouts(weights):
    pw = PackedWeights(weights[0], weights[1], torch.device("cpu"), torch.float32)
    assert pw.vgg[0]["w"].shape == (64, 27) and pw.vgg[1]["w"].shape == (64, 576)
    # 3x3 weights are (ky, kx, cin)-major
    w, _ = fold_bn(weights[0]["encoder.cnn.layers.3.weight"], weights[0]["encoder.cnn.layers.3.bias"], weights[0], "encoder.cnn.layers.4")
    assert torch.equal(pw.vgg[1]["w"].reshape(64, 3, 3, 64)[5, 1, 2], w[5, :, 1, 2])
    R = pw.refiner[16]
    assert R["c"] == 1377 and R["cp"] == 1384 and R["blocks"][0]["dw_w"].shape == (25, 1384)
    assert R["blocks"][0]["pw_w"].shape == (1377, 1384) and (R["blocks"][0]["pw_w"][:, 1377:] == 0).all()
    assert pw.vit_patch_w.shape == (1024, 592)
    with pytest.raises(RuntimeError):
        bad = dict(weights[0]); bad.pop("decoder.gps.16.pos_conv.bias")
        PackedWeights(bad, weights[1], torch.device("cpu"), torch.float32)


class _Recorder:
    """Stands in for cabi.call: validates field names and that pointer ranges lie inside live tensors."""

    def __init__(self):
        self.calls = []
        self.allocs = {}

    def track(self, t):
        self.allocs[t.data_ptr()] = t.numel() * t.element_size()

    def _inside(self, ptr, nbytes, what):
        if isinstance(ptr, torch.Tensor):
            ptr = ptr.data_ptr()
        for base, size in self.allocs.items():
            if base <= ptr and ptr + nbytes <= base + size:
                return
        raise AssertionError(f"{what}: pointer range [{ptr}, +{nbytes}) not inside any tracked buffer")

    def __call__(self, fn, struct, **kw):
        valid = {f for f, _ in cabi.STRUCT_FIELDS[struct]}
        assert set(kw) <= valid, (fn, set(kw) - valid)
        self.calls.append(fn)
        es = {0: 4, 1: 2, 2: 2, 3: 2}
        if fn == "romab200_gemm":
            if kw["dtype_ab"] == cabi.RB_F16S:        # split pairs: the second planes have the same geometry
                assert kw.get("A_lo") is not None and kw.get("B_lo") is not None
                lo = dict(kw, A=kw["A_lo"], B=kw["B_lo"], A_lo=None, B_lo=None, dtype_ab=cabi.RB_F16)
                if kw["dtype_c"] == cabi.RB_F16S:
                    lo.update(C=kw["C_lo"], dtype_c=cabi.RB_F16)
                self.calls.pop()
                self(fn, struct, **{k: v for k, v in lo.items() if v is not None})
            if kw["dtype_c"] == cabi.RB_F16S:
                assert kw.get("C_lo") is not None
            b0, b1 = kw.get("batch0", 1), kw.get("batch1", 1)
            M, N, K = kw["M"], kw["N"], kw["K"]
            ea, ec = es[kw["dtype_ab"]], es[kw["dtype_c"]]
            nt = kw.get("ntaps", 1)
            kt = K // nt
            off = (b0 - 1) * kw.get("sa0", 0) + (b1 - 1) * kw.get("sa1", 0)
            if nt == 1:
                self._inside(kw["A"], (off + (M - 1) * kw["lda"] + kt) * ea, f"{fn}.A")
            else:
                assert kw["a_rows"] == M
                self._inside(kw["A"], ((kw["a_rows"] - 1) * kw["lda"] + kt) * ea, f"{fn}.A")
            offb = (b0 - 1) * kw.get("sb0", 0) + (b1 - 1) * kw.get("sb1", 0)
            if kw.get("trans_b", 0):
                self._inside(kw["B"], (offb + (K - 1) * kw["ldb"] + N) * ea, f"{fn}.B")
            else:
                self._inside(kw["B"], (offb + (N - 1) * kw["ldb"] + K) * ea, f"{fn}.B")
            offc = (b0 - 1) * kw.get("sc0", 0) + (b1 - 1) * kw.get("sc1", 0)
            rows_out = M
            if kw.get("rowmap", 0) == cabi.ROWMAP_PAD_TO_COMPACT:
                rows_out = M // (kw["pad_h"] * kw["pad_w"]) * (kw["pad_h"] - 2) * (kw["pad_w"] - 2)
            self._inside(kw["C"], (offc + (rows_out - 1) * kw["ldc"] + N) * ec, f"{fn}.C")
            assert kw["lda"] % 4 == 0 and kw["ldb"] % 4 == 0, "vector path wants 16-byte pitches"
            if ea == 2:
                assert kw["lda"] % 8 == 0 and kw["ldb"] % 8 == 0, "TMA wants 16-byte pitches"
        for k, v in kw.items():
            if isinstance(v, torch.Tensor):
                assert v.is_contiguous(), (fn, k)
                self._inside(v, 1, f"{fn}.{k}")


@pytest.mark.parametrize("symmetric,upsample,split", [(True, True, True), (True, True, False), (False, True, True), (True, False, False)])
def test_engine_dry_run(weights, monkeypatch, symmetric, upsample, split):
    import roma_b200.engine as engine_mod
    rec = _Recorder()
    eng = engine_mod.Engine.__new__(engine_mod.Engine)
    eng.device = torch.device("cpu")
    eng.precision, eng.dtype, eng.dt = "fp32" if split else "fp32_simt", torch.float32, cabi.RB_F32
    eng.split, eng._lane, eng.generation = split, "main", 0
    eng.w = PackedWeights(weights[0], weights[1], eng.device, torch.float32, split=split)
    eng._buf, eng._const, eng.debug, eng.profile, eng.gemm_profile, eng.use_flash_attn, eng.gp_algo = {}, {}, None, None, None, True, (3 if split else 2)
    eng.overlap_cnn, eng._side, eng.gp_tensor_core, eng.fused_c144, eng.fused_small_f32 = False, None, True, True, True
    eng.lc_table16, eng.lc_tile_radii, eng.side_ctas = True, (2,), 0
    for t in _tensors(eng.w):
        rec.track(t)
    orig_buf, orig_const = eng.buf, eng.const

    def buf(*a, **k):
        t = orig_buf(*a, **k); rec.track(t); return t

    def const(*a, **k):
        t = orig_const(*a, **k); rec.track(t); return t
    eng.buf, eng.const = buf, const
    monkeypatch.setattr(engine_mod, "call", rec)
    b, coarse, up = 1, 112, 168
    A, B, Ah, Bh = synthetic.make_pair(b, coarse, up, 1)
    images = torch.cat((A, B)); rec.track(images)
    state, states, sizes = eng.run_pass(images, b, symmetric, False, coarse / 560)
    assert sizes == {1: (112, 112), 2: (56, 56), 4: (28, 28), 8: (14, 14), 16: (8, 8)}
    D = 2 * b if symmetric else b
    assert state.shape == (D, 112, 112, 3) and states[16].shape == (D, 8, 8, 3)
    if upsample:
        hi = torch.cat((Ah, Bh)); rec.track(hi)
        state, _, sizes = eng.run_pass(hi, b, symmetric, True, up / 560, (state, 112, 112))
        assert state.shape == (D, 168, 168, 3)
    n_gemm = rec.calls.count("romab200_gemm")
    per_pass_refiner = 9 * (5 if not upsample else 5 + 4)
    # refiner pointwise GEMMs (the stride-1 blocks are fused kernels) + 24 ViT blocks x 4 linears (+ 2 attention GEMMs un-fused)
    assert n_gemm > per_pass_refiner * 4 // 5 + 24 * 4
    assert rec.calls.count("romab200_gp_solve") == 1
    assert rec.calls.count("romab200_refiner_prologue") == (9 if upsample else 5)


def _tensors(obj):
    if isinstance(obj, torch.Tensor):
        yield obj
    elif isinstance(obj, dict):
        for v in obj.values():
            yield from _tensors(v)
    elif isinstance(obj, (list, tuple)):
        for v in obj:
            yield from _tensors(v)
    elif hasattr(obj, "hi") and hasattr(obj, "lo"):          # packing.Split (RB_F16S pair)
        yield from _tensors([obj.hi, obj.lo])
    elif hasattr(obj, "__dict__"):
        yield from _tensors(vars(obj))


def test_layout_product_never_imports_oracle():
    """The shipped package must not route through the oracle (or the reference) anywhere."""
    import os
    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "roma_b200")
    for dirpath, _, files in os.walk(root):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text and "romatch import" not in text, f


def test_cabi_call_validates_tensors():
    """The ctypes shim refuses tensors whose device / dtype / layout / size contradict the call's description (a raw pointer of
    the wrong kind would be silent garbage on the device)."""
    a = torch.zeros(8, 8)
    with pytest.raises(RuntimeError, match="expected the current CUDA device"):
        cabi.call("romab200_gemm", "rb_gemm_args", A=a, B=a, C=a, M=8, N=8, K=8, lda=8, ldb=8, ldc=8, dtype_ab=cabi.RB_F32, dtype_c=cabi.RB_F32)
    with pytest.raises(TypeError):
        cabi.call("romab200_gemm", "rb_gemm_args", not_a_field=1)
    # dtype / contiguity / size rules, exercised on the validator itself with the device check satisfied by a stand-in
    # (on the current CUDA device when there is one)
    index = torch.cuda.current_device() if torch.cuda.is_available() else None

    class FakeCuda(torch.Tensor):
        is_cuda = True

        @property
        def device(self):
            return type("D", (), {"index": index})()
    def fake(t):
        return t.as_subclass(FakeCuda)
    half, f32 = fake(torch.zeros(8, 8, dtype=torch.float16)), fake(torch.zeros(8, 8))
    kw = dict(A=half, B=half, C=f32, M=8, N=8, K=8, lda=8, ldb=8, ldc=8, dtype_ab=cabi.RB_F32, dtype_c=cabi.RB_F32)
    with pytest.raises(RuntimeError, match="dtype"):
        cabi._validate("romab200_gemm", "rb_gemm_args", kw)
    kw.update(A=f32, B=f32, M=16)
    with pytest.raises(RuntimeError, match="needs"):
        cabi._validate("romab200_gemm", "rb_gemm_args", kw)
    kw.update(M=8, A=fake(torch.zeros(8, 16)[:, :8]))
    with pytest.raises(RuntimeError, match="contiguous"):
        cabi._validate("romab200_gemm", "rb_gemm_args", kw)
    kw.update(A=f32)
    cabi._validate("romab200_gemm", "rb_gemm_args", kw)


def test_romatch_import_shim():
    """`import romatch` through shim/ gives the reference's import surface backed by this package (romatch/__init__.py:2-8)."""
    import importlib
    import os
    import sys
    shim = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "shim")
    sys.path.insert(0, shim)
    try:
        for m in [k for k in sys.modules if k == "romatch" or k.startswith("romatch.")]:
            del sys.modules[m]
        romatch = importlib.import_module("romatch")
        import roma_b200
        assert romatch.roma_outdoor is roma_b200.roma_outdoor and romatch.roma_indoor is roma_b200.roma_indoor
        assert romatch.tiny_roma_v1_outdoor is roma_b200.tiny_roma_v1_outdoor
        assert (romatch.DEBUG_MODE, romatch.GLOBAL_STEP, romatch.STEP_SIZE, romatch.LOCAL_RANK) == (False, 0, 1, -1) and isinstance(romatch.RANK, int)
        zoo = importlib.import_module("romatch.models.model_zoo")
        assert "outdoor" in zoo.weight_urls["romatch"] and zoo.roma_model is roma_b200.model_zoo.roma_model
        assert importlib.import_module("romatch.models.matcher").RegressionMatcher is roma_b200.matcher.RegressionMatcher
    finally:
        sys.path.remove(shim)
        for m in [k for k in sys.modules if k == "romatch" or k.startswith("romatch.")]:
            del sys.modules[m]


def test_prologue_tiles_matches_kernel_geometry():
    """cabi.prologue_tiles (the size of the `tile_done` workspace callers allocate) follows the tile shapes compiled into the kernels."""
    import os, re
    text = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "roma_b200", "csrc", "refiner_common.cuh")).read()
    generic = re.search(r"template <int R> struct LcTile \{ static constexpr int TQX = (\d+), TQY = (\d+)", text)
    r7 = re.search(r"struct LcTile<7> \{ static constexpr int TQX = (\d+), TQY = (\d+)", text)
    r2 = re.search(r"struct LcTile<2> \{ static constexpr int TQX = (\d+), TQY = (\d+)", text)
    shapes = {3: tuple(map(int, generic.groups())), 7: tuple(map(int, r7.groups())), 2: tuple(map(int, r2.groups()))}
    for r, (tx, ty) in shapes.items():
        for h, w in ((40, 40), (70, 70), (108, 108), (13, 9), (1, 1)):
            assert cabi.prologue_tiles(r, h, w) == -(-h // ty) * -(-w // tx), (r, h, w)
