"""ctypes binding of libromab200.so — the thin shim between PyTorch (device memory, streams) and the C ABI.

The argument structs are generated from `include/romab200.h` itself at import time, so the Python side
cannot drift from the header.  Every wrapper passes raw device pointers (`tensor.data_ptr()`) and the
current CUDA stream; a non-zero return code becomes a `RuntimeError` carrying `romab200_last_error()`.
There is no fallback: if the library is missing or the device is not a B200, calls fail loudly.
"""
from __future__ import annotations

import ctypes
import os
import re
from typing import Dict

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(os.path.dirname(HERE), "include", "romab200.h")
LIB_PATH = os.path.join(HERE, "lib", "libromab200.so")

RB_F32, RB_F16, RB_BF16, RB_F16S = 0, 1, 2, 3
ACT_NONE, ACT_RELU, ACT_GELU = 0, 1, 2
ROWMAP_NONE, ROWMAP_PAD_KEEP, ROWMAP_PAD_TO_COMPACT, ROWMAP_SEGMENT = 0, 1, 2, 3
EPI_LINEAR, EPI_COSKERNEL = 0, 1
BACKEND_AUTO, BACKEND_SIMT, BACKEND_TCGEN05 = 0, 1, 2
SAMPLE_IDENTITY, SAMPLE_THRESHOLD, SAMPLE_BALANCE = 0, 1, 2

DTYPE_CODE = {torch.float32: RB_F32, torch.float16: RB_F16, torch.bfloat16: RB_BF16}

_CTYPES = {
    "int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64, "uint64_t": ctypes.c_uint64, "float": ctypes.c_float,
}


def _parse_header(path: str):
    """Returns ({struct_name: [(field, ctype)]}, [function names]) parsed from the C header."""
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    structs: Dict[str, list] = {}
    for body, name in re.findall(r"typedef\s+struct\s*\{(.*?)\}\s*(\w+)\s*;", text, flags=re.S):
        fields = []
        for decl in body.split(";"):
            decl = decl.strip()
            if not decl:
                continue
            m = re.match(r"(const\s+)?(\w+)\s*(\*?)\s*(.*)$", decl, flags=re.S)
            base, ptr, names = m.group(2), m.group(3), m.group(4)
            first = True
            for part in names.split(","):
                part = part.strip()
                is_ptr = bool(ptr) if first else part.startswith("*")
                first = False
                part = part.lstrip("*").strip()
                arr = re.match(r"(\w+)\[(\d+)\]$", part)
                if is_ptr:
                    fields.append((part, ctypes.c_void_p))
                elif arr:
                    fields.append((arr.group(1), _CTYPES[base] * int(arr.group(2))))
                else:
                    fields.append((part, _CTYPES[base]))
        structs[name] = fields
    funcs = re.findall(r"\b(romab200_\w+)\s*\(", text)
    return structs, sorted(set(funcs))


STRUCT_FIELDS, FUNCTIONS = _parse_header(HEADER)
STRUCTS = {name: type(name, (ctypes.Structure,), {"_fields_": fields}) for name, fields in STRUCT_FIELDS.items()}

_lib = None


def load_library(path: str = LIB_PATH) -> ctypes.CDLL:
    """dlopen the in-tree library and type its entry points.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(path):
        raise RuntimeError(f"{path} not found: build it with `python -m roma_b200.build` "
                           "(there is no CPU or PyTorch fallback for the CUDA path)")
    lib = ctypes.CDLL(path)
    lib.romab200_last_error.restype = ctypes.c_char_p
    lib.romab200_abi_version.restype = ctypes.c_int
    lib.romab200_device_ok.restype = ctypes.c_int
    lib.romab200_launch_count.restype = ctypes.c_ulonglong
    for fn in FUNCTIONS:
        getattr(lib, fn)            # AttributeError if the header declares a symbol the library lacks
    _lib = lib
    return lib


def _ptr(t):
    if t is None:
        return None
    if isinstance(t, int):
        return t
    return t.data_ptr()


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


launch_count = 0      # number of C-ABI calls made (bench.py reports kernel launches from it)

# ---- argument validation: the C ABI takes raw pointers, so a tensor of the wrong dtype / device / layout would be silent garbage.
# For every struct: tensor field -> the field that carries its dtype code (or a fixed torch dtype, or a function of the call's fields).
_CODE_DTYPE = {RB_F32: torch.float32, RB_F16: torch.float16, RB_BF16: torch.bfloat16, RB_F16S: torch.float16}
_F32 = torch.float32
_FIELD_DTYPES = {
    "rb_gemm_args": {"A": "dtype_ab", "B": "dtype_ab", "A_lo": torch.float16, "B_lo": torch.float16, "C": "dtype_c", "C_lo": torch.float16,
                     "R": "dtype_r", "bias": _F32, "col_scale": _F32, "norm_a": _F32, "norm_b": _F32},
    "rb_layernorm_args": {"x": "dtype_x", "y": "dtype_y", "y_lo": torch.float16, "gamma": _F32, "beta": _F32},
    "rb_softmax_args": {"s": "dtype", "out_hi": torch.float16, "out_lo": torch.float16},
    "rb_flash_attn_args": {"qkv": "dtype", "out": "dtype", "qkv_lo": torch.float16, "out_lo": torch.float16},
    "rb_rownorm_args": {"x": "dtype", "out": _F32},
    "rb_copy2d_args": {"src": "dtype_src", "dst": "dtype_dst", "row_scale": _F32},
    "rb_split_pair_args": {"x": _F32, "hi": torch.float16, "lo": torch.float16, "row_norm": _F32},
    "rb_conv_first_args": {"image": _F32, "out": "dtype_out", "out_lo": torch.float16, "weight": _F32, "bias": _F32},
    "rb_maxpool_args": {"in": "dtype", "out": "dtype", "in_lo": torch.float16, "out_lo": torch.float16},
    "rb_im2col_args": {"image": _F32, "out": "dtype_out"},
    "rb_tokens_args": {"patch": _F32, "cls": _F32, "pos": _F32, "tokens": _F32},
    "rb_gp_solve_args": {"W": _F32},
    "rb_cls_args": {"logits": "dtype", "state": _F32},
    "rb_refiner_prologue_args": {"feat": "dtype", "state": _F32, "d": "dtype", "emb_weight": _F32, "emb_bias": _F32, "grid_x": _F32, "grid_y": _F32,
                                 "win_x": _F32, "win_y": _F32, "tile_done": torch.uint8, "corr_table": _F32},
    "rb_local_corr_args": {"f0": "dtype_f", "f1": "dtype_f", "flow": _F32, "out": "dtype_out", "win_x": _F32, "win_y": _F32},
    "rb_local_corr_warp_args": {"f0": _F32, "f1": _F32, "warp": _F32, "out": _F32},
    "rb_dwconv_args": {"in": "dtype", "weight": _F32, "bias": _F32, "out_lo": torch.float16},
    "rb_refiner_block_small_args": {"in": "dtype", "out": "dtype", "dw_weight": _F32, "dw_bias": _F32},
    "rb_refiner_block_c144_args": {"in": "dtype", "out": "dtype", "dw_weight": _F32, "dw_bias": _F32, "pw_bias": _F32, "pw_weight_lo": torch.float16,
                                   # fp32 maps take the pointwise weights as an RB_F16S pair (pw_weight = hi plane)
                                   "pw_weight": lambda kw: torch.float16 if kw.get("dtype") == RB_F32 else _CODE_DTYPE.get(kw.get("dtype"))},
    "rb_refiner_tail_args": {"d": "dtype", "weight": _F32, "bias": _F32, "state": _F32, "delta_out": _F32},
    "rb_resize_args": {"in": _F32, "out": _F32},
    "rb_match_epilogue_args": {"state": _F32, "coarse_state": _F32, "warp": _F32, "cert": _F32, "grid_x": _F32, "grid_y": _F32},
    "rb_kde_args": {"x": _F32, "density": _F32, "workspace": _F32},
    "rb_preprocess_args": {"in": torch.uint8, "tmp": torch.uint8, "out_u8": torch.uint8, "out": _F32, "bounds_x": torch.int32, "kk_x": torch.int32,
                           "bounds_y": torch.int32, "kk_y": torch.int32},
    "rb_sample_args": {"values": _F32, "out_idx": torch.int32, "out_weights": _F32, "keys": _F32, "scratch": torch.int32, "seed_dev": torch.int64},
}


def _gemm_min_elems(kw):
    """(field, minimum number of elements) of the GEMM operands for the given geometry."""
    b0, b1 = kw.get("batch0", 1) or 1, kw.get("batch1", 1) or 1
    M, N, K, nt = kw["M"], kw["N"], kw["K"], kw.get("ntaps", 1) or 1
    offa = (b0 - 1) * kw.get("sa0", 0) + (b1 - 1) * kw.get("sa1", 0)
    offb = (b0 - 1) * kw.get("sb0", 0) + (b1 - 1) * kw.get("sb1", 0)
    offc = (b0 - 1) * kw.get("sc0", 0) + (b1 - 1) * kw.get("sc1", 0)
    a = offa + ((kw.get("a_rows") or M) - 1) * kw["lda"] + K // nt
    b = offb + ((K - 1) * kw["ldb"] + N if kw.get("trans_b", 0) else (N - 1) * kw["ldb"] + K)
    rows_out = M
    if kw.get("rowmap", 0) == ROWMAP_PAD_TO_COMPACT:
        rows_out = M // (kw["pad_h"] * kw["pad_w"]) * (kw["pad_h"] - 2) * (kw["pad_w"] - 2)
    elif kw.get("rowmap", 0) == ROWMAP_SEGMENT:
        rows_out = (M - 1) // kw["seg_in"] * kw["seg_out"] + (M - 1) % kw["seg_in"] + kw.get("seg_off", 0) + 1
    c = offc + (rows_out - 1) * kw["ldc"] + N
    return {"A": a, "A_lo": a, "B": b, "B_lo": b, "C": c, "C_lo": c}


def _validate(fn_name, struct_name, kw):
    table = _FIELD_DTYPES.get(struct_name, {})
    cur = torch.cuda.current_device() if torch.cuda.is_available() else None
    mins = _gemm_min_elems(kw) if struct_name == "rb_gemm_args" else {}
    for k, v in kw.items():
        if not isinstance(v, torch.Tensor):
            continue
        if not v.is_cuda or (cur is not None and v.device.index != cur):
            raise RuntimeError(f"{fn_name}: argument `{k}` lives on {v.device}, expected the current CUDA device cuda:{cur}")
        if not v.is_contiguous():
            raise RuntimeError(f"{fn_name}: argument `{k}` is not contiguous (shape {tuple(v.shape)}, strides {v.stride()})")
        want = table.get(k)
        if isinstance(want, str):
            want = _CODE_DTYPE.get(kw.get(want))
        elif callable(want) and not isinstance(want, torch.dtype):
            want = want(kw)
        if want is not None and v.dtype != want:
            raise RuntimeError(f"{fn_name}: argument `{k}` has dtype {v.dtype}, the call describes it as {want}")
        if k in mins and v.numel() < mins[k]:
            raise RuntimeError(f"{fn_name}: argument `{k}` holds {v.numel()} elements, the described geometry needs {mins[k]}")


def call(fn_name: str, struct_name: str, **kw) -> None:
    """Fill `struct_name` from keyword arguments (tensors become device pointers) and call `fn_name`."""
    global launch_count
    lib = load_library()
    args = STRUCTS[struct_name]()
    valid = {f for f, _ in STRUCT_FIELDS[struct_name]}
    for k in kw:
        if k not in valid:
            raise TypeError(f"{struct_name} has no field {k}")
    _validate(fn_name, struct_name, kw)
    for k, v in kw.items():
        if isinstance(v, torch.Tensor) or v is None:
            setattr(args, k, _ptr(v))
        elif isinstance(v, (list, tuple)):
            arr = getattr(args, k)
            for i, x in enumerate(v):
                arr[i] = x
        else:
            setattr(args, k, v)
    rc = getattr(lib, fn_name)(ctypes.byref(args), _stream())
    launch_count += 1
    if rc != 0:
        raise RuntimeError(f"{fn_name} failed: {lib.romab200_last_error().decode()}")


def prologue_tiles(radius: int, h: int, w: int) -> int:
    """Tiles per map of the tile-cooperative refiner prologue (`tile_done` bytes per decoder item; include/romab200.h)."""
    ty = 2 if radius == 7 else 4
    return ((h + ty - 1) // ty) * ((w + 7) // 8)


def kernel_launches() -> int:
    """Kernels launched by libromab200 in this process so far."""
    return int(load_library().romab200_launch_count())


def device_ok() -> bool:
    return bool(load_library().romab200_device_ok())
