#!/usr/bin/env python
"""bench.py — pairs/s of RoMa dense match() (+ sample()) at 560 -> 864 on B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision fp32|fp32_simt|fp16|bf16] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch of synthetic input: `roma_outdoor(...).match()` on
`--pairs-per-gpu` symmetric 560x560 pairs with 864x864 high-res tensors, followed by `.sample()` of each pair
(BASELINE.json configs[1]; with N > 1 every rank runs the same per-GPU batch on its own pairs: weak scaling,
no data-path collective — pairs are independent, SURVEY §8e).  Prints ONE JSON line (rank 0).

  value      whole-job pairs/s, inputs resident in HBM, CUDA-event timed per step, max over ranks
  e2e        the same through the public API with HOST buffers: pinned inputs -> H2D inside match(), and the
             step's results (warp, certainty, sampled matches) read back D2H inside the timed region
  roofline   the dominant kernel (the GEMM back-end: tcgen05 in the 16-bit modes), algorithmic FLOPs of every
             launch / its CUDA-event time, both collected live during the timed steps
  parity     max-abs error of this run's warp / certainty against tests/golden/full_sym_up.npz (the UNMODIFIED reference's
             fp32 output for the seed-1 pair, every 8th pixel), computed live; the default precision is the one that meets
             the 1e-4 bar: "fp32" = fp32-class GEMMs on tcgen05 from split-fp16 operand pairs (DESIGN.md §2)
  fast_mode  the same workload in the reference's CUDA autocast regime (fp16 operands), reported beside it with its error
  cpu_baseline  the CPU oracle (a port of the reference's fp32 CPU path) on this box's host cores, one pair
--dump-outputs DIR writes what the last timed step returned to its caller on rank 0 as float32 .npy files: warp and certainty
(rank 0's match() results; the whole gathered batch when N > 1 scatters it) and sample_matches, sample_certainty (only the pairs
rank 0 sampled itself, so fewer pairs than warp when the batch is sharded).  Inputs are seeded and torch's generator is seeded
before the timed steps, so two builds run with the same arguments can be compared file by file.  The samples are reproducible
with one pair per step (the default): sample() calls share one pinned seed buffer, so with several pairs per step an earlier
call can read a later call's seeds.  Above DUMP_LIMIT bytes in all, every file keeps the same seeded subset of its rows (pixels
of warp / certainty, samples), flattened to [rows] or [rows, 4].
--impl reference times that CPU path alone (the reference itself is pure Python/PyTorch and does not travel
to the GPU box; `oracle/` is its validated restatement, bit-exact against it in the build container).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

COARSE, UPSAMPLE = 560, 864
FLOP_PER_PAIR = 6.58e12          # SURVEY §6 (FlopCounterMode + analytic attention/solves)
DUMP_LIMIT = 64 * 10 ** 6       # bytes of --dump-outputs in all


def dump_outputs(path, outputs):
    """Writes {name: tensor} as path/<name>.npy in float32.  When the total exceeds DUMP_LIMIT, each array is cut to the same
    fraction of its rows (a 4-vector of warp / sample_matches, one value of the certainties), drawn with a fixed seed: arrays
    with the same row count (warp and certainty; the two sample outputs) keep the same rows."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    arrays = {k: v.detach().float().cpu().numpy() for k, v in outputs.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        frac = (DUMP_LIMIT - 4096 * len(arrays)) / total                 # room for the .npy headers
        for k, a in arrays.items():
            rows = a.reshape(-1, 4) if k in ("warp", "sample_matches") else a.reshape(-1)
            keep = np.sort(np.random.default_rng(0).choice(len(rows), int(len(rows) * frac), replace=False))
            arrays[k] = rows[keep]
    for k, a in arrays.items():
        np.save(os.path.join(path, f"{k}.npy"), a)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_burst=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons every 200 ms while the timed region runs."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        rows = [r for r in self.rows if len(r) >= 8]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[1]) for r in rows if r[1].replace(".", "").isdigit())
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(rows[0][2]) if rows[0][2].isdigit() else None,
                "power_w_max": max((float(r[3]) for r in rows if r[3].replace(".", "").isdigit()), default=None),
                "samples": len(rows), "reasons": sorted(reasons)}


def cpu_reference_time(steps, warmup, budget_s=240.0, with_sample=True):
    """Times the CPU oracle on one symmetric 560->864 pair per step. Returns (seconds per pair list, threads)."""
    import torch
    from oracle.roma_oracle import RomaOracle
    from roma_b200 import synthetic
    # measured on the 128-core GPU box (scripts/cpu_threads_probe.py): 16 thr 40 s, 32 thr 28 s, 64 thr 32 s, 128 thr 59 s for
    # the coarse pass -> the oracle (like the reference: torch CPU ops) is fastest at ~32 threads; more only add contention
    threads = int(os.environ.get("ROMA_CPU_THREADS", "0")) or min(os.cpu_count() or 1, 32)
    torch.set_num_threads(threads)
    mw, dw = synthetic.make_weights(0)
    orc = RomaOracle(mw, dw, COARSE, UPSAMPLE)
    if warmup > 0:                                   # warm the thread pool / allocator on a tiny problem
        small = RomaOracle(mw, dw, 112, 168)
        a, b, ah, bh = synthetic.make_pair(1, 112, 168, 1)
        for _ in range(warmup):
            small.match(a, b, ah, bh)
    A, B, Ah, Bh = synthetic.make_pair(1, COARSE, UPSAMPLE, 1)
    times, t_begin = [], time.perf_counter()
    for _ in range(steps):
        t0 = time.perf_counter()
        warp, cert = orc.match(A, B, Ah, Bh)
        if with_sample:
            torch.manual_seed(0)
            orc.sample(warp[0], cert[0], num=10000)
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_begin > budget_s:
            break
    return times, torch.get_num_threads()


def local_corr_flow_sweep(dev, precision, mode="engine"):
    """The local-correlation prologue launches alone, on smooth flow (identity + 0.5 pixel of noise: neighbouring pixels share their
    windows) and on random flow (uniform over the image: no sharing, what the seeded synthetic weights produce): ms per launch and the
    compulsory HBM bytes of SURVEY 8d (read f0 + f1 + flow, write the window) per second, for the five launches of one direction pair.
    mode "engine" = what the parity mode runs (stride 16: split + two all-pairs tcgen05 GEMMs + the gathering prologue, replayed from a
    CUDA graph; stride 4: tile-cooperative pass + per-pixel kernel for the tiles it declines; stride 8: per-pixel kernel);
    "per_pixel" = the per-pixel kernel everywhere; "tile_all" = the tile-cooperative pass at every scale."""
    import torch
    from roma_b200 import arch, cabi
    from roma_b200.cabi import call
    dt = torch.float32 if precision.startswith("fp32") else (torch.float16 if precision == "fp16" else torch.bfloat16)
    if dt != torch.float32:
        mode = "per_pixel"
    code = cabi.DTYPE_CODE[dt]
    es = 4 if dt == torch.float32 else 2
    g = torch.Generator(device="cpu").manual_seed(0)
    out = {}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for kind in ("smooth", "random"):
        tot_ms, tot_bytes, per = 0.0, 0.0, {}
        for res, scales in ((COARSE, (16, 8, 4)), (UPSAMPLE, (8, 4))):
            for sc in scales:
                spec = arch.REFINERS[sc]
                h = w = res // sc if sc != 16 else res // 14
                D = E = 2
                n = h * w
                ldf = (spec.feat + 7) // 8 * 8
                cp = (spec.channels + 7) // 8 * 8
                feat = torch.randn(E, h, w, ldf, generator=g).to(dev, dt)
                ys, xs = torch.linspace(-1 + 1 / h, 1 - 1 / h, h), torch.linspace(-1 + 1 / w, 1 - 1 / w, w)
                gy, gx = torch.meshgrid(ys, xs, indexing="ij")
                ident = torch.stack((gx, gy), -1)[None].expand(D, h, w, 2)
                flow = ident + torch.randn(D, h, w, 2, generator=g) * (1.0 / w) if kind == "smooth" else torch.rand(D, h, w, 2, generator=g) * 2 - 1
                state = torch.cat((flow, torch.zeros(D, h, w, 1)), -1).contiguous().to(dev)
                d = torch.zeros(D * h * w, cp, dtype=dt, device=dev)
                r = spec.radius
                wx = torch.linspace(-2 * r / w, 2 * r / w, 2 * r + 1).to(dev)
                wy = torch.linspace(-2 * r / h, 2 * r / h, 2 * r + 1).to(dev)
                R = dict(emb_w=torch.randn(spec.emb, 2).to(dev), emb_b=torch.randn(spec.emb).to(dev))
                kw = dict(feat=feat, ldf=ldf, n_img=E, y_shift=1, state=state, d=d, ldd=cp, D=D, h=h, w=w, cf=spec.feat, emb=spec.emb, radius=r, dtype=code,
                          emb_weight=R["emb_w"], emb_bias=R["emb_b"], disp_scale=1.25, grid_x=xs.to(dev), grid_y=ys.to(dev), win_x=wx, win_y=wy)
                how = "per-pixel kernel"
                pre = []                                   # launches before the prologue (table path)
                if mode == "tile_all" or (mode == "engine" and r == 2):
                    tiles = torch.zeros(D * cabi.prologue_tiles(r, h, w), dtype=torch.uint8, device=dev)
                    kw.update(tile_done=tiles, tile_done_len=tiles.numel())
                    how = "tile-cooperative pass + per-pixel kernel for declined tiles"
                elif mode == "engine" and sc == 16:
                    cf = spec.feat
                    hi, lo = torch.empty(E * n, cf, dtype=torch.float16, device=dev), torch.empty(E * n, cf, dtype=torch.float16, device=dev)
                    ldt = (n + 7) // 8 * 8
                    table = torch.zeros(D, n, ldt, device=dev)
                    pre.append(lambda feat=feat, hi=hi, lo=lo, n=n, cf=cf: call("romab200_split_f16s", "rb_split_pair_args", x=feat, hi=hi, lo=lo, rows=E * n, cols=cf, ldx=cf, ldd=cf))
                    for i0, y0 in ((0, 1), (1, 0)):
                        pre.append(lambda i0=i0, y0=y0, hi=hi, lo=lo, table=table, n=n, cf=cf, ldt=ldt: call(
                            "romab200_gemm", "rb_gemm_args", A=hi[i0 * n:], A_lo=lo[i0 * n:], B=hi[y0 * n:], B_lo=lo[y0 * n:], C=table[i0], M=n, N=n, K=cf, lda=cf,
                            ldb=cf, ldc=ldt, dtype_ab=cabi.RB_F16S, dtype_c=cabi.RB_F32, batch0=1, batch1=1, ntaps=1, alpha=float(cf) ** -0.5))
                    kw.update(corr_table=table, ld_corr_table=ldt)
                    how = "split + 2 all-pairs tcgen05 GEMMs + gathering prologue (CUDA graph of the 4 launches)"

                def launches():
                    for f in pre:
                        f()
                    call("romab200_refiner_prologue", "rb_refiner_prologue_args", **kw)
                side = torch.cuda.Stream()
                with torch.cuda.stream(side):
                    for _ in range(2):
                        launches()
                torch.cuda.synchronize()
                run = launches
                if pre:                                    # several short launches: replay them from a graph so that host launch latency is not timed
                    graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(graph):
                        launches()
                    run = graph.replay
                ts = []
                for _ in range(5):
                    flush.zero_()
                    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    s.record(); run(); e.record()
                    torch.cuda.synchronize()
                    ts.append(s.elapsed_time(e))
                ms = sorted(ts)[2]
                nbytes = D * h * w * ((2 * spec.feat + spec.k) * es + 8)        # f0 + f1 read once, window written once, flow read
                per[f"stride{sc}@{res}"] = {"ms": round(ms, 4), "gbs": round(nbytes / ms / 1e6, 1), "how": how}
                tot_ms += ms; tot_bytes += nbytes
        out[kind] = {"ms_per_pair": round(tot_ms, 4), "hbm_gbs": round(tot_bytes / tot_ms / 1e6, 1), "launches": per}
    return out


def allpairs_kernel_leg(dev, reps=20):
    """The all-pairs CosKernel launches of one pair exactly as the engine issues them (K_AA | K_BB batched into the Cholesky workspace,
    K_AB and K_BA as split pairs for mu = K_xy alpha; 1600 x 1600 x 512 each, split-fp16 operands on tcgen05), `reps` times in ONE CUDA
    graph so that host launch latency (3 launches of ~30 us each) is not in the timed region; inputs are L2-resident as in the step
    (the split kernel that produces them runs right before)."""
    import torch
    from roma_b200 import arch, cabi
    from roma_b200.cabi import call
    n, cf, E = (COARSE // 14) ** 2, arch.PROJ[16][1], 2
    ldw = (n + 7) // 8 * 8
    g = torch.Generator().manual_seed(0)
    x = torch.randn(E * n, cf, generator=g).to(dev)
    norms = torch.empty(E * n, device=dev)
    call("romab200_row_norms", "rb_rownorm_args", x=x, out=norms, rows=E * n, cols=cf, ldx=cf, dtype=cabi.RB_F32)
    hi, lo = torch.empty(E * n, cf, dtype=torch.float16, device=dev), torch.empty(E * n, cf, dtype=torch.float16, device=dev)
    call("romab200_split_f16s", "rb_split_pair_args", x=x, hi=hi, lo=lo, rows=E * n, cols=cf, ldx=cf, ldd=cf, row_norm=norms)
    stride_w = (n + arch.GP_DIM) * ldw
    Wk = torch.zeros(E, n + arch.GP_DIM, ldw, device=dev)
    kxy_hi, kxy_lo = torch.zeros(E, n, ldw, dtype=torch.float16, device=dev), torch.zeros(E, n, ldw, dtype=torch.float16, device=dev)
    common = dict(M=n, N=n, K=cf, lda=cf, ldb=cf, ldc=ldw, dtype_ab=cabi.RB_F16S, ntaps=1, alpha=1.0, epi=cabi.EPI_COSKERNEL, sna0=n, snb0=n,
                  eps=arch.GP_COS_EPS, inv_t=1.0 / arch.GP_TEMPERATURE, cos_normalized=1)

    def three():
        call("romab200_gemm", "rb_gemm_args", A=hi, A_lo=lo, B=hi, B_lo=lo, C=Wk, dtype_c=cabi.RB_F32, batch0=E, batch1=1, sa0=n * cf, sb0=n * cf, sc0=stride_w,
             norm_a=norms, norm_b=norms, diag_add=arch.GP_SIGMA_NOISE, **common)
        for i0, y0 in ((0, 1), (1, 0)):
            call("romab200_gemm", "rb_gemm_args", A=hi[i0 * n:], A_lo=lo[i0 * n:], B=hi[y0 * n:], B_lo=lo[y0 * n:], C=kxy_hi[i0], C_lo=kxy_lo[i0], dtype_c=cabi.RB_F16S,
                 batch0=1, batch1=1, sa0=n * cf, sb0=n * cf, sc0=n * ldw, norm_a=norms[i0 * n:], norm_b=norms[y0 * n:], diag_add=0.0, **common)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        for _ in range(3):
            three()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(reps):
            three()
    ts = []
    for _ in range(7):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); graph.replay(); e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e) / reps)
    return {"ms_per_pair": sorted(ts)[3], "launches_per_pair": 3, "flops_per_pair_reference": 4 * 2.0 * n * n * cf, "flops_per_pair_computed": 4 * 2.0 * n * n * cf,
            "reps_in_graph": reps}


def preprocess_leg(dev, reps=5):
    """Input preprocessing of the PIL route (utils.py:164-173) for one 12-megapixel frame -> 560x560 and 864x864: the CUDA path (raw bytes
    H2D + romab200_preprocess_rgb8, CUDA events incl. the copy) beside Pillow + numpy on one host core, and whether the results are the same bits."""
    import numpy as np
    import torch
    from PIL import Image
    from roma_b200 import preprocess
    rng = np.random.default_rng(0)
    pil = Image.fromarray(rng.integers(0, 256, (3000, 4000, 3), dtype=np.uint8), "RGB")
    pre = preprocess.DevicePreprocessor(dev)
    sizes = ((COARSE, COARSE), (UPSAMPLE, UPSAMPLE))
    outs = [pre.resize_normalize(pre.upload(pil), s) for s in sizes]            # warm-up, tables cached
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        raw = pre.upload(pil)
        for s in sizes:
            pre.resize_normalize(raw, s)
    e1.record()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    host = [preprocess.pil_to_normalized(pil, s) for s in sizes]
    host_ms = (time.perf_counter() - t0) * 1e3
    same = all(torch.equal(o.cpu(), h) for o, h in zip(outs, host))
    return {"image": "3000x4000 RGB -> 560x560 + 864x864", "device_ms": e0.elapsed_time(e1) / reps, "pillow_host_ms": host_ms,
            "bit_exact_vs_pillow": bool(same), "h2d_bytes": 3000 * 4000 * 3}


def torch_cuda_baseline(dev, steps=5, warmup=2, with_sample=True):
    """The "existing Blackwell kernels" bar (SURVEY 2, BASELINE.md 3): the same graph through stock PyTorch on this GPU — the oracle's
    torch.nn.functional restatement of the reference with weights and inputs on `cuda`, i.e. cuDNN convolutions, cuBLAS GEMMs, SDPA
    attention, cuSOLVER Cholesky, ATen grid_sample — once in fp32 (TF32 off) and once under fp16 autocast with the GP kept in fp32
    (the reference's CUDA regime, utils.py:639-653, approximately).  A comparison leg only: nothing of the product runs here."""
    import torch
    from oracle.roma_oracle import RomaOracle
    from roma_b200 import synthetic
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    mw, dw = synthetic.make_weights(0)
    orc = RomaOracle(mw, dw, COARSE, UPSAMPLE, device=dev)
    A, B, Ah, Bh = (t.to(dev) for t in synthetic.make_pair(1, COARSE, UPSAMPLE, seed=1))
    stage_ev = {}

    def wrap(name, fn):
        def inner(*a, **k):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            out = fn(*a, **k)
            e.record()
            stage_ev.setdefault(name, []).append((s, e))
            return out
        return inner
    gp_fp32 = orc.gp

    def gp_no_autocast(x, y):
        with torch.autocast("cuda", enabled=False):
            return gp_fp32(x.float(), y.float())
    orc.gp = wrap("gp", gp_no_autocast)
    orc.vgg, orc.dinov2 = wrap("vgg", orc.vgg), wrap("dinov2", orc.dinov2)
    orc.embedding_decoder = wrap("decoder transformer", orc.embedding_decoder)
    ref_fn = orc.conv_refiner
    orc.conv_refiner = lambda s, *a, **k: wrap(f"refine{s}", ref_fn)(s, *a, **k)
    out = {}
    for label, ctx in (("fp32", lambda: torch.autocast("cuda", enabled=False)), ("fp16_autocast", lambda: torch.autocast("cuda", dtype=torch.float16))):
        def step():
            with torch.inference_mode(), ctx():
                w, c = orc.match(A, B, Ah, Bh)
            if with_sample:
                orc.sample(w[0].float(), c[0].float(), num=10000)
        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        stage_ev.clear()
        ev = []
        for _ in range(steps):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(); step(); e.record()
            ev.append((s, e))
        torch.cuda.synchronize()
        ms = sum(s.elapsed_time(e) for s, e in ev) / steps
        out[label] = {"value": 1e3 / ms, "unit": "pairs/s", "ms_per_step": ms,
                      "stage_ms_per_step": {k: round(sum(s.elapsed_time(e) for s, e in v) / steps, 3) for k, v in stage_ev.items()}}
    out["what"] = ("stock PyTorch " + torch.__version__ + " on the same GPU: oracle/roma_oracle.py (torch.nn.functional restatement of the reference, "
                   "bit-exact vs it on CPU) with weights and inputs on cuda: cuDNN / cuBLAS / SDPA / cuSOLVER / ATen kernels; 1 pair per step, "
                   "CUDA events, TF32 off; fp16_autocast keeps the GP in fp32")
    del orc
    torch.cuda.empty_cache()
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    times, threads = cpu_reference_time(args.steps, args.warmup)
    sec = sum(times) / len(times)
    v = 1.0 / sec
    sample = f"{len(times)} x (1 symmetric pair 560->864 match()+sample(10000)) on {threads} host threads" + \
             ("" if len(times) == args.steps else f"; stopped after {len(times)} of {args.steps} steps (240 s budget)")
    line = {
        "impl": "reference", "metric": "image-pairs/sec match()+sample() 560->864", "value": v, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": len(times), "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "roma_outdoor 560->864 single pair, symmetric, full match()+sample() [BASELINE configs[1]]",
                   "pairs_per_step": 1, "weights": "seeded synthetic (no network)"},
        "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def run_ours(args):
    import torch
    import torch.distributed as dist
    from roma_b200 import cabi, roma_indoor, roma_outdoor, sharding, synthetic

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # stdout must carry the single JSON line only: NCCL prints its version banner to stdout when NCCL_DEBUG=VERSION comes
        # from the environment or from an nccl.conf (seen on the GPU boxes), so the level is pinned unless the caller asked for
        # more, and communicator creation (init + first collective) runs with fd 1 pointed at stderr
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        # the data path is point-to-point (scatter of inputs, gather of results): measured at N=2 with NCCL's default one or two P2P
        # channels it moved 17-49 GB/s; more channels per peer use the NVLink bandwidth (770 GB/s per direction measured)
        os.environ.setdefault("NCCL_MIN_P2P_NCHANNELS", "16")
        os.environ.setdefault("NCCL_MAX_P2P_NCHANNELS", "32")
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    from roma_b200 import model_zoo
    amp = {"fp16": torch.float16, "bf16": torch.bfloat16, "fp32": torch.float32, "fp32_simt": torch.float32}[args.precision]
    factory, wseed = (roma_indoor, 1) if args.model == "indoor" else (roma_outdoor, 0)      # same graph, different checkpoint (model_zoo/__init__.py:8-9)
    mw, dw = synthetic.make_weights(wseed)
    model_zoo.fp32_backend = "simt" if args.precision == "fp32_simt" else "tcgen05"
    model = factory(dev, weights=mw, dinov2_weights=dw, coarse_res=COARSE, upsample_res=UPSAMPLE, amp_dtype=amp)
    assert model.engine.precision == args.precision
    P = args.pairs_per_gpu                       # pairs per match() call on one GPU
    G = args.global_pairs or P * world           # pairs per step over the whole job
    # N > 1: rank 0 owns the batch of a step; the inputs are scattered and the warps / certainties gathered over NCCL INSIDE the
    # timed region (SURVEY 8e).  --no-scatter keeps every rank on its own resident pairs (no collective on the data path).
    sharded = world > 1 and not args.no_scatter
    if sharded or world == 1:
        lo, hi = sharding.shard_bounds(G, world)[rank]
        src_pairs = synthetic.make_pair(G, COARSE, UPSAMPLE, seed=1) if rank == 0 else None
    else:
        lo, hi = 0, G // world
        src_pairs = synthetic.make_pair(hi, COARSE, UPSAMPLE, seed=1 + rank)
    host = [t.pin_memory() for t in src_pairs] if src_pairs is not None else None
    devt = [t.to(dev) for t in src_pairs] if src_pairs is not None else None
    del src_pairs
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)        # > 126 MB L2
    out_host = None
    d2h_samples = [0]
    sample_calls = [0]

    sample_host = {}                                  # pinned read-back buffers of the samples, per pair slot of a step
    dump_step = {}                                    # --dump-outputs: this rank's results of the current headline step

    def sample_batch(warp, cert, to_host=False):
        if args.no_sample:
            return
        for i in range(warp.shape[0]):
            m, c = model.sample(warp[i], cert[i], num=10000)
            if "samples" in dump_step:
                dump_step["samples"].append((m, c))
            if to_host:
                # asynchronous read-back into pinned memory on the step's stream: no host synchronisation inside a step, so the host
                # queues the next step while this one runs (a blocking .cpu() here exposed ~0.2 ms of launch latency per step)
                slot = (sample_calls[0], tuple(m.shape), tuple(c.shape), c.dtype)
                sample_calls[0] += 1
                if slot not in sample_host:
                    sample_host[slot] = (torch.empty(m.shape, dtype=m.dtype).pin_memory(), torch.empty(c.shape, dtype=c.dtype).pin_memory())
                sample_host[slot][0].copy_(m, non_blocking=True)
                sample_host[slot][1].copy_(c, non_blocking=True)
                d2h_samples[0] += m.numel() * 4 + c.numel() * c.element_size()

    def run_pairs(inputs, to_host=False):
        """match() (+ sample()) of the step's pairs: sharded over the ranks from rank 0's tensors, or local sub-batches of P pairs."""
        if sharded:
            return sharding.match_sharded(model, *(inputs if rank == 0 else (None, None, None, None)), n_pairs=G, max_batch=P,
                                          on_batch=lambda w, c: sample_batch(w, c, to_host))
        outs = []
        for a in range(0, inputs[0].shape[0], P):
            w, c = model.match(inputs[0][a:a + P], inputs[1][a:a + P], im_A_high_res=inputs[2][a:a + P], im_B_high_res=inputs[3][a:a + P])
            sample_batch(w, c, to_host)
            outs.append((w, c))
        return outs[0] if len(outs) == 1 else (torch.cat([o[0] for o in outs]), torch.cat([o[1] for o in outs]))

    def step_device():
        return run_pairs(devt)

    d2h_stream = torch.cuda.Stream(device=dev)
    h2d_stream = torch.cuda.Stream(device=dev)
    out_hosts = [None, None]
    stage_in = [None, None]                           # device staging of a step's inputs, filled by the upload stream one step ahead
    e2e_state = {"k": 0, "done": None, "uploaded": [None, None], "consumed": [None, None]}

    def upload(slot):
        """Pinned host inputs -> device staging buffer `slot` on the upload stream (after the step that last read the buffer)."""
        if stage_in[slot] is None:
            stage_in[slot] = [torch.empty(t.shape, dtype=t.dtype, device=dev) for t in host]
        with torch.cuda.stream(h2d_stream):
            if e2e_state["consumed"][slot] is not None:
                h2d_stream.wait_event(e2e_state["consumed"][slot])
            for d, h in zip(stage_in[slot], host):
                d.copy_(h, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
        e2e_state["uploaded"][slot] = ev

    def step_e2e():
        """The same step from HOST buffers: pinned inputs -> H2D, results (warp, certainty, samples) -> pinned host memory.  Nothing in a
        step synchronises the host.  At N = 1 the read-back of warp / certainty runs on a copy stream into one of two pinned buffers, so
        that it overlaps the NEXT step's upload and compute (PCIe is full duplex); every step still copies its inputs in and its results
        out inside the timed region, and the tail of the last read-back is added to the total (see `e2e_tail_ms`)."""
        nonlocal out_host
        d2h_samples[0] = 0
        sample_calls[0] = 0
        if sharded:
            if rank == 0:
                for d, h in zip(devt, host):
                    d.copy_(h, non_blocking=True)
            res = run_pairs(devt, to_host=True)
        else:
            # software pipeline a serving loop would run: the upload of step k+1 (pinned host -> device, on its own stream) is issued
            # before step k's kernels and overlaps them; step k itself starts from the buffer uploaded during step k-1.  Every step's
            # inputs still cross PCIe inside the timed region (the upload issued in the last timed step belongs to the step after it,
            # the first timed step's was issued in the last warm-up step: K uploads in K steps).
            slot = e2e_state["k"] & 1
            if e2e_state["uploaded"][slot] is None:
                upload(slot)                                   # very first step: nothing was prefetched
            torch.cuda.current_stream().wait_event(e2e_state["uploaded"][slot])
            upload(slot ^ 1)
            res = run_pairs(stage_in[slot], to_host=True)
            consumed = torch.cuda.Event()
            consumed.record()
            e2e_state["consumed"][slot] = consumed
            e2e_state["uploaded"][slot] = None
        d2h = d2h_samples[0]
        if res is not None:
            warp, cert = res
            d2h += warp.numel() * 4 + cert.numel() * 4
            if sharded:
                if out_host is None:
                    out_host = (torch.empty(warp.shape, dtype=warp.dtype).pin_memory(), torch.empty(cert.shape, dtype=cert.dtype).pin_memory())
                out_host[0].copy_(warp, non_blocking=True)
                out_host[1].copy_(cert, non_blocking=True)
            else:
                k = e2e_state["k"] & 1
                e2e_state["k"] += 1
                if out_hosts[k] is None:
                    out_hosts[k] = (torch.empty(warp.shape, dtype=warp.dtype).pin_memory(), torch.empty(cert.shape, dtype=cert.dtype).pin_memory())
                ready = torch.cuda.Event()
                ready.record()
                with torch.cuda.stream(d2h_stream):
                    d2h_stream.wait_event(ready)
                    out_hosts[k][0].copy_(warp, non_blocking=True)
                    out_hosts[k][1].copy_(cert, non_blocking=True)
                    warp.record_stream(d2h_stream); cert.record_stream(d2h_stream)
                    done = torch.cuda.Event(enable_timing=True)
                    done.record()
                e2e_state["done"] = done
        return d2h

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, profile=False, tail=None):
        ev = []
        barrier()
        for _ in range(steps):
            flush.zero_()                                       # evict L2 between timed iterations
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            ev.append((s, e))
        last = tail() if tail else None                         # event that ends work the last step left on another stream
        barrier()
        out = [s.elapsed_time(e) for s, e in ev]
        if last is not None:
            out[-1] += max(0.0, ev[-1][1].elapsed_time(last))   # the last step's read-back ends after its stream-side end event
        return out

    for _ in range(max(args.warmup, 3)):
        step_device()
    torch.cuda.synchronize()
    eng = model.engine
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)

    def dump_step_device():
        dump_step["samples"] = []
        dump_step["out"] = step_device()
    if args.dump_outputs:
        torch.manual_seed(0)                                  # sample() draws its seeds from torch's CPU generator
    launches0 = cabi.kernel_launches() + model.graph_launches
    ms = timed(dump_step_device if args.dump_outputs else step_device, args.steps)      # headline: device side replayed as a CUDA graph
    launches = cabi.kernel_launches() + model.graph_launches - launches0
    if args.dump_outputs:
        if rank == 0:
            outputs = dict(zip(("warp", "certainty"), dump_step["out"]))
            if dump_step["samples"]:
                outputs["sample_matches"] = torch.cat([m for m, _ in dump_step["samples"]])
                outputs["sample_certainty"] = torch.cat([c for _, c in dump_step["samples"]])
            dump_outputs(args.dump_outputs, outputs)
        dump_step.clear()
    # second timed region, same workload, eager launches with a CUDA-event pair around every GEMM launch and every
    # pipeline stage (events cannot be read back from inside a replayed graph): feeds `roofline` and the stage table
    eng.gemm_profile, eng.profile = [], {}
    ms_prof = timed(step_device, args.steps)
    gemm_prof, stage_prof = eng.gemm_profile, eng.profile
    eng.gemm_profile, eng.profile = None, None
    h2d = sum(t.numel() * 4 for t in host) if host is not None else 0
    d2h_box = [0]
    for _ in range(2):
        step_e2e()

    def e2e_fn():
        d2h_box[0] = step_e2e()
    ms_e2e = timed(e2e_fn, args.steps, tail=lambda: e2e_state["done"])
    clocks = sampler.stop()

    def golden_errors(m):
        """max-abs / percentile errors of m.match() on the seed-1 pair against the unmodified reference's output."""
        import numpy as np
        g = dict(np.load(os.path.join(ROOT, "tests", "golden", "full_sym_up.npz")))
        ga, gb, gah, gbh = (t.to(dev) for t in synthetic.make_pair(1, COARSE, UPSAMPLE, seed=1))
        w, c = m.match(ga, gb, im_A_high_res=gah, im_B_high_res=gbh)
        ew = np.abs(w[:, ::8, ::8].float().cpu().numpy() - g["warp"]).max(-1)
        ec = np.abs(c[:, ::8, ::8].float().cpu().numpy() - g["certainty"])
        return ew, ec

    parity = fast = None
    if rank == 0 and args.model != "outdoor":
        parity = {"ok": None, "tol": 1e-4,
                  "note": "the 560->864 golden is the reference's output for the outdoor (seed-0) weights; roma_indoor (same graph, seed-1 weights) is pinned "
                          "against the reference at 112->168 by tests/test_e2e_gpu.py::test_roma_indoor_vs_reference_golden"}
    elif rank == 0:
        ew, ec = golden_errors(model)
        parity = {"warp": float(ew.max()), "certainty": float(ec.max()), "tol": 1e-4, "ok": bool(ew.max() <= 1e-4 and ec.max() <= 1e-4),
                  "reference": "tests/golden/full_sym_up.npz = output of the unmodified reference (CPU fp32) for the seed-1 560->864 pair, every 8th pixel",
                  "precision": args.precision}
    if rank == 0 and world == 1 and args.precision == "fp32" and not args.no_fast_mode:
        # the reference's CUDA regime (fp16 autocast) next to the parity mode: same workload, same timing method
        import numpy as np
        model.free_buffers()
        model_zoo.fp32_backend = None
        fmodel = roma_outdoor(dev, weights=mw, dinov2_weights=dw, coarse_res=COARSE, upsample_res=UPSAMPLE, amp_dtype=torch.float16)
        main_model, model = model, fmodel
        for _ in range(3):
            step_device()
        fms = timed(step_device, args.steps)
        ew, ec = golden_errors(fmodel)
        model = main_model
        fast = {"precision": "fp16 operands / f32 accumulate (the reference's CUDA autocast regime)", "value": G * args.steps / (sum(fms) / 1e3),
                "unit": "pairs/s", "ms_per_step": sum(fms) / args.steps,
                "parity": {"warp_median": float(np.median(ew)), "warp_p99": float(np.percentile(ew, 99)), "warp_max": float(ew.max()),
                           "certainty_median": float(np.median(ec)), "certainty_p99": float(np.percentile(ec, 99)), "certainty_max": float(ec.max()),
                           "tol": 1e-4, "ok": bool(ew.max() <= 1e-4 and ec.max() <= 1e-4)},
                "note": "16-bit operands cannot meet 1e-4 end to end (coarse-classifier argmax flips, SURVEY 7.2); not the headline"}
        fmodel.free_buffers()
        del fmodel
    del mw, dw
    library = None
    if rank == 0 and world == 1 and not args.no_library_baseline:
        model.free_buffers()
        torch.cuda.empty_cache()
        try:
            library = torch_cuda_baseline(dev, steps=min(args.steps, 5), with_sample=not args.no_sample)
        except Exception as exc:                      # a comparison leg must never take the product's line down
            library = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    total_ms, total_ms_e2e = sum(ms), sum(ms_e2e)
    if world > 1:
        t = torch.tensor([total_ms, total_ms_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, total_ms_e2e = t.tolist()
        tb = torch.tensor([float(h2d), float(d2h_box[0])], device=dev, dtype=torch.float64)      # host<->device bytes of all ranks
        dist.all_reduce(tb)
        h2d, d2h_box[0] = int(tb[0].item()), int(tb[1].item())
    pairs = G * args.steps
    value = pairs / (total_ms / 1e3)
    e2e_value = pairs / (total_ms_e2e / 1e3)

    if rank == 0:
        peaks = load_peaks()
        by = {}
        shapes = {}
        cos_ms, cos_flops, cos_n, cos_backend = 0.0, 0.0, 0, None
        for backend, flops, s, e, shape, epi in gemm_prof:
            t = s.elapsed_time(e)
            if epi == cabi.EPI_COSKERNEL:
                cos_ms += t; cos_flops += flops; cos_n += 1; cos_backend = backend
            d = by.setdefault(backend, [0.0, 0.0, 0])
            d[0] += flops; d[1] += t; d[2] += 1
            sh = shapes.setdefault((backend,) + shape, [0.0, 0.0, 0])
            sh[0] += flops; sh[1] += t; sh[2] += 1
        dom = max(by, key=lambda k: by[k][1]) if by else None
        roofline = None
        if dom:
            fl, t_ms, n = by[dom]
            ach = fl / (t_ms / 1e3) / 1e12
            # dram__bytes_read+write of one named launch of this kernel, measured by `ncu --set full` on this same command
            # (scripts/gpu_profile.sh writes the side-car next to the ncu summary it comes from); null when not captured
            traffic = None
            tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
            if os.path.exists(tpath):
                traffic = json.load(open(tpath)).get(dom)
            passes = 3.0 if dom == "tcgen05-split" else 1.0
            roofline = {"kernel": f"romab200_gemm[{dom}]", "bound": "tensor", "achieved": ach * passes, "peak": peaks["bf16_sustained"],
                        "unit": "TFLOP/s", "frac": ach * passes / peaks["bf16_sustained"],
                        "flops_definition": ("tensor-core FLOPs of the algorithm as it runs on the f16 pipe: an fp32-class product from split-fp16 operand pairs is THREE "
                                             "f16 MMAs per k-step (hi.hi, hi.lo, lo.hi; 22 significand bits), i.e. 3 x 2MNK per launch - each term is needed, none is a "
                                             "recomputation; ncu's sm__pipe_tensor_cycles_active of the same kernel (profiles/r02_ncu_gemm_fc1_qkv_tcgen05_split_final.txt: "
                                             "46-53 %) is the independent check" if passes > 1 else "2MNK per launch"),
                        "fp32_equivalent": {"achieved": ach, "frac": ach / peaks["bf16_sustained"],
                                            "note": "2MNK per launch (the FLOPs of the fp32 contraction the reference performs) against the same bf16 peak: "
                                                    "bounded by 1/3 in the split mode"} if passes > 1 else None,
                        "passes": passes,
                        "traffic": traffic["dram_bytes"] if traffic else None,
                        "traffic_launch": traffic["launch"] if traffic else None,
                        "peak_source": peaks["source"] + ", sustained bf16 cuBLAS figure (kernel timed inside a long step)",
                        "launches_timed": n, "share_of_step": t_ms / sum(ms_prof),
                        "measured_in": "second timed region of the same K steps, eager launches (per-kernel events cannot be read "
                                       "from a replayed CUDA graph); headline value uses graph replay",
                        "eager_ms_per_step": sum(ms_prof) / args.steps,
                        "flops_per_launch_avg": fl / n, "avg_launch_ms": t_ms / n}
        stages = {k: sum(s.elapsed_time(e) for s, e in v) / args.steps for k, v in stage_prof.items()}
        # the two kernels BASELINE.json's north_star names, measured live in the same eager region
        from roma_b200 import arch
        extra = []
        if cos_n:
            # executed FLOPs: the 16-bit modes run the contraction on split-fp16 operands (K' = 3K) for fp32-class accuracy;
            # the algorithmic count is the fp32 contraction the reference performs (matcher.py:191-200)
            # (fp16 mode: K' = 3K operand trick -> flops recorded are 3x; split mode: flops recorded are algorithmic, 3 MMAs each)
            split = 3.0 if cos_backend == "tcgen05" else 1.0
            executed = 3.0 if cos_backend == "tcgen05-split" else 1.0
            ach = cos_flops / split / (cos_ms / 1e3) / 1e12
            pk = peaks["bf16_sustained"] if cos_backend.startswith("tcgen05") else 72.0
            entry = {"kernel": f"all-pairs CosKernel (romab200_gemm, RB_EPI_COSKERNEL, {cos_backend})", "bound": "tensor" if cos_backend.startswith("tcgen05") else "fp32",
                     "achieved": ach, "achieved_executed": cos_flops * executed / (cos_ms / 1e3) / 1e12, "peak": pk, "unit": "TFLOP/s", "frac": ach / pk,
                     "launches_per_step": cos_n / args.steps, "ms_per_step": cos_ms / args.steps,
                     "measured_in": "eager launches of the step, CUDA events around each launch (includes the host's launch latency: ~100 us for a ~30 us kernel)",
                     "note": "four 1600x1600x512 problems per pair (2.6 GFLOP each, 1.5 us at peak): size-limited, see DESIGN.md"}
            if cos_backend == "tcgen05-split" and world == 1:
                try:
                    leg = allpairs_kernel_leg(dev)
                    ach = leg["flops_per_pair_reference"] / (leg["ms_per_pair"] / 1e3) / 1e12
                    entry.update({"eager": {k: entry[k] for k in ("achieved", "achieved_executed", "frac", "ms_per_step", "measured_in")},
                                  "achieved": 3.0 * ach, "frac": 3.0 * ach / pk, "achieved_executed": 3.0 * ach,
                                  "fp32_equivalent": {"achieved": ach, "frac": ach / pk, "note": "2MNK of the four matrices the reference computes per pair"},
                                  "flops_definition": "3 x 2MNK per matrix: split-fp16 operand pairs, three f16 MMAs per k-step (see roofline.flops_definition)",
                                  "ms_per_step": leg["ms_per_pair"] * P,
                                  "measured_in": f"the engine's 3 launches per pair, {leg['reps_in_graph']} pairs replayed from one CUDA graph (device time only, "
                                                 "operands L2-resident as in the step)"})
                except Exception as exc:
                    entry["graph_leg_error"] = f"{type(exc).__name__}: {exc}"[:200]
            extra.append(entry)
        lc_fma, lc_bytes = 0.0, 0.0
        try:
            lc_sweep = local_corr_flow_sweep(dev, args.precision)
        except Exception as exc:
            lc_sweep = {"error": f"{type(exc).__name__}: {exc}"[:200]}
        esz = 4 if args.precision.startswith("fp32") else 2
        for res, scales in ((COARSE, arch.SCALES), (UPSAMPLE, arch.UPSAMPLE_SCALES)):
            for sc in scales:
                spec = arch.REFINERS[sc]
                if spec.radius:
                    px = 2 * P * (res // sc) ** 2
                    lc_fma += px * (2 * spec.radius + 2) ** 2 * spec.feat
                    lc_bytes += px * (2 * spec.feat + spec.k) * esz          # f0 + f1 read once, window written once
        lc_ms = sum(v for k, v in stages.items() if (k.strip().startswith("prologue") and arch.REFINERS[int(k.strip()[8:].split(".")[0])].radius) or k.strip() == "gp.corr16")
        lc_pp = None
        if world == 1 and args.precision == "fp32":
            try:
                lc_pp = {m: {k: {"ms_per_pair": v["ms_per_pair"], "hbm_gbs": v["hbm_gbs"], "ms": {a: b["ms"] for a, b in v["launches"].items()}}
                             for k, v in local_corr_flow_sweep(dev, args.precision, m).items()} for m in ("per_pixel", "tile_all")}
            except Exception as exc:
                lc_pp = {"error": f"{type(exc).__name__}: {exc}"[:200]}
        if lc_ms > 0:
            extra.append({"kernel": "local correlation (stride 16: all-pairs tcgen05 table + gather; stride 8: refiner_prologue_kernel<3>; stride 4: "
                                    "refiner_prologue_tile_kernel<2> + refiner_prologue_kernel<2>) incl. the x / grid_sample / embedding part of the prologue",
                          "bound": "hbm", "achieved": lc_bytes / (lc_ms / 1e3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": lc_bytes / (lc_ms / 1e3) / 1e9 / peaks["hbm_gbs"],
                          "fp32_fma_tflops": 2 * lc_fma / (lc_ms / 1e3) / 1e12, "fp32_fma_frac_of_nominal_72": 2 * lc_fma / (lc_ms / 1e3) / 1e12 / 72.0,
                          "ms_per_step": lc_ms, "measured_in": "eager launches of the step (the flow of the seeded synthetic weights is random: no window sharing)",
                          "flow_sweep": lc_sweep, "flow_sweep_hbm_frac": ({k: round(v["hbm_gbs"] / peaks["hbm_gbs"], 4) for k, v in lc_sweep.items()} if lc_sweep and "error" not in lc_sweep else None),
                          "flow_sweep_other_kernels": lc_pp,
                          "note": "algorithmic bytes = SURVEY 8d (f0 + f1 + flow read once, window written once).  The windows of neighbouring pixels overlap, so f1 "
                                  "is served from L1/L2, not HBM; the CUDA-core kernels are bound by the 4 bytes of L1/shared-memory bandwidth each fp32 FMA "
                                  "needs (floor 0.29 ms per pair = 0.24 of the HBM roofline, DESIGN.md 4); only stride 16, where the table is small, goes "
                                  "through the tensor cores"})
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            times, threads = cpu_reference_time(1, 1, with_sample=not args.no_sample)
            cpu = {"value": 1.0 / (sum(times) / len(times)), "unit": "pairs/s", "cores": threads, "kind": "port",
                   "sample": f"{len(times)} symmetric pair 560->864 match()" + ("" if args.no_sample else "+sample(10000)") +
                             " through oracle/roma_oracle.py (fp32 restatement of the reference, bit-exact vs it in the build container)"}
        prep = None
        if world == 1:
            try:
                prep = preprocess_leg(dev)
            except Exception as exc:
                prep = {"error": f"{type(exc).__name__}: {exc}"[:200]}
        cfg_name = "configs[1]"
        if args.global_pairs == 64 and world == 8 and args.model == "outdoor":
            cfg_name = "configs[2]"
        elif args.global_pairs == 32 and world == 4 and args.model == "indoor":
            cfg_name = "configs[3]"
        workload = (f"roma_{args.model} 560->864, symmetric, full match()" + ("" if args.no_sample else "+sample(10000)") +
                    (f", batch {G} synthetic pairs sharded over {world} GPU(s) [BASELINE {cfg_name}]" if args.global_pairs else
                     f", {G} pair(s) per step [BASELINE configs[1] per GPU]"))
        in_b = 2 * (3 * COARSE * COARSE + 3 * UPSAMPLE * UPSAMPLE) * 4
        out_b = UPSAMPLE * 2 * UPSAMPLE * 5 * 4
        wire = sharding.wire_bytes(G, world, in_b, out_b)
        line = {
            "metric": "image-pairs/sec match()+sample() 560->864", "value": value, "unit": "pairs/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if args.global_pairs else "weak", "vs_baseline": None,
            "dtype": {"fp16": "f16 operands / f32 accumulate (reference CUDA autocast regime)", "bf16": "bf16 operands / f32 accumulate",
                      "fp32": "f32 (activations f32; GEMM operands as split-f16 pairs hi + 2^-11 lo on tcgen05, f32 accumulate: fp32-class)",
                      "fp32_simt": "f32 (CUDA-core FFMA GEMMs)"}[args.precision],
            "data": "synthetic",
            "config": {"workload": workload,
                       "pairs_per_match_call": P, "global_pairs_per_step": G,
                       "parallelism": (f"dp{world}: rank 0 holds the {G} pairs of a step, NCCL scatter of the inputs + gather of warp/certainty inside the "
                                       f"timed region, {P} pairs per match() call" if sharded else
                                       (f"dp{world} (every rank on its own resident pairs, no collective)" if world > 1 else "1 GPU")),
                       "nccl_bytes_per_step": {"scatter": wire[0], "gather": wire[1]} if sharded else None,
                       "precision": args.precision, "weights": "seeded synthetic (no network)",
                       "l2": "256 MiB buffer written between timed steps; per-step activations also exceed the 126 MB L2"},
            "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_box[0],
                    "ms_per_step": total_ms_e2e / args.steps,
                    "how": ("every step's inputs go from pinned host memory to the device and its warp, certainty and samples back into pinned host memory, "
                            "all through roma_outdoor().match() / .sample(); no host synchronisation inside a step; " +
                            ("software-pipelined like a serving loop: the upload of step k+1 (own stream, two device staging buffers) and the warp / "
                             "certainty read-back of step k-1 (own stream, two pinned buffers) overlap step k's kernels; K uploads and K read-backs in K "
                             "timed steps, the tail of the last read-back is added to the total" if not sharded else "upload and read-back on the step's stream"))},
            "parity": parity, "fast_mode": fast, "gpu_library_baseline": library, "preprocess": prep,
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "roofline_kernels": extra, "cpu_baseline": cpu,
            "stage_ms_per_step": {k: round(v, 3) for k, v in sorted(stages.items(), key=lambda kv: -kv[1])},
            "gemm_backends": {k: {"tflops": v[0] / (v[1] / 1e3) / 1e12, "ms_per_step": v[1] / args.steps, "launches_per_step": v[2] / args.steps}
                              for k, v in by.items()},
            "whole_path_tflops": FLOP_PER_PAIR * pairs / (total_ms / 1e3) / 1e12,
            "top_gemm_shapes": [{"backend": k[0], "MxNxK,batch": list(k[1:]), "ms_per_step": round(v[1] / args.steps, 3),
                                 "launches_per_step": v[2] / args.steps, "tflops": round(v[0] / (v[1] / 1e3) / 1e12, 1)}
                                for k, v in sorted(shapes.items(), key=lambda kv: -kv[1][1])[:16]],
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch_cuda"])
    ap.add_argument("--no-library-baseline", action="store_true", help="skip the stock-PyTorch-CUDA comparison leg (gpu_library_baseline)")
    ap.add_argument("--precision", default=os.environ.get("ROMA_B200_PRECISION", "fp32"), choices=["fp32", "fp32_simt", "fp16", "bf16"])
    ap.add_argument("--no-fast-mode", action="store_true", help="skip the fp16 fast-mode leg reported beside the parity mode")
    ap.add_argument("--pairs-per-gpu", type=int, default=1, help="pairs per match() call on one GPU")
    ap.add_argument("--global-pairs", type=int, default=0, help="total pairs per step held by rank 0 and sharded over the GPUs (strong scaling; "
                    "BASELINE configs[2]: --gpus 8 --global-pairs 64 --pairs-per-gpu 8; configs[3]: --model indoor --gpus 4 --global-pairs 32 --pairs-per-gpu 8)")
    ap.add_argument("--model", default="outdoor", choices=["outdoor", "indoor"])
    ap.add_argument("--no-scatter", action="store_true", help="N > 1: every rank on its own resident pairs (no NCCL scatter / gather in the timed region)")
    ap.add_argument("--no-sample", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's warp, certainty and samples to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "torch_cuda":
        import torch
        if int(os.environ.get("RANK", "0")) == 0:
            torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
            lib = torch_cuda_baseline(torch.device("cuda", torch.cuda.current_device()), steps=args.steps, warmup=max(args.warmup, 2), with_sample=not args.no_sample)
            print(json.dumps({"impl": "torch_cuda", "metric": "image-pairs/sec match()+sample() 560->864", "unit": "pairs/s", "n_gpus": 1,
                              "value": lib["fp16_autocast"]["value"], "value_fp32": lib["fp32"]["value"], "gpu_library_baseline": lib}))
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
