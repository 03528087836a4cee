"""ctypes binding of the C-ABI shared library (``include/b200q.h``) and its in-tree build.

The library is built with plain ``nvcc`` for sm_100a (no torch headers) into
``convnet_quantization_b200/libb200q.so``; there is deliberately NO CPU fallback:
if the library is missing, or no CUDA device is present, product calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC = PKG_DIR / "csrc"
LIB_PATH = PKG_DIR / "libb200q.so"
# Development build (-DB200Q_DEV): the product sources plus the experiments that are kept for their analysis but do not
# ship - the fused conv1+conv2 kernel (measured slower), the CUDA-core bring-up convolution, and the environment
# switches that disable kernel roles / select alternate instantiations for timing.  Only tests and A-B scripts load it.
DEV_LIB_PATH = PKG_DIR / "libb200q_dev.so"
BUILD_DIR = PKG_DIR / "build"
SOURCES = ("runtime.cu", "elementwise.cu", "simt.cu", "igemm_tc.cu", "conv_halo.cu", "conv_halo2.cu", "conv_pair.cu", "conv_small.cu", "conv1_tc.cu",
           "linear_dynamic_tc.cu", "net.cu")
DEV_SOURCES = SOURCES + ("conv12_fused.cu",)
# -fmad=false: the requantisation is specified as separately rounded fp32 add / mul (SURVEY.md Appendix A); ptxas was
# seen contracting even explicit mul.rn.f32x2 + add.rn.f32x2 pairs into FFMA2, which changes the rounding.
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false",
              "-Xcompiler", "-fPIC"]

EXPORTS = (
    "b200q_last_error", "b200q_abi_version", "b200q_launch_count", "b200q_quantize_nchw_to_nhwc", "b200q_quantize_flat",
    "b200q_dequantize", "b200q_relu_q", "b200q_max_pool2x2_nhwc", "b200q_minmax", "b200q_aminmax", "b200q_histc",
    "b200q_lut_u8", "b200q_conv3x3_first", "b200q_quantize_conv3x3_first", "b200q_u8_conv3x3_first", "b200q_conv3x3_tc",
    "b200q_linear_tc", "b200q_linear_simt", "b200q_linear_dequant", "b200q_linear_dynamic",
    "b200q_static_workspace_bytes", "b200q_static_forward", "b200q_static_forward_u8", "b200q_graph_create",
    "b200q_graph_create_u8", "b200q_graph_launch", "b200q_graph_destroy", "b200q_static_num_stages", "b200q_static_stage_name",
    "b200q_static_forward_profiled", "b200q_static_evaluate", "b200q_static_evaluate_u8",
)
DEV_EXPORTS = EXPORTS + ("b200q_conv12_fused", "b200q_conv3x3_simt")
REDUCE_SCRATCH_BYTES = 8256    # B200Q_REDUCE_SCRATCH_BYTES
REDUCE_QPARAMS_OFFSET = 8224   # B200Q_REDUCE_QPARAMS_OFFSET
GRAPH_PDL = 1                  # B200Q_GRAPH_PDL
EVAL_COUNTERS = 5              # B200Q_EVAL_COUNTERS, in the order of B200Q_EVAL_TOP1 .. B200Q_EVAL_TOP5_TIED
EVAL_COUNTER_NAMES = ("top1", "top5", "images", "top1_tied", "top5_tied")


class B200QError(RuntimeError):
    pass


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    raise B200QError("nvcc not found")


def _stale(path: Path = LIB_PATH) -> bool:
    if not path.exists():
        return True
    t = path.stat().st_mtime
    deps = list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [PKG_DIR.parent / "include" / "b200q.h"]
    return any(p.stat().st_mtime > t for p in deps)


def build(force: bool = False, verbose: bool = False, dev: bool = False) -> Path:
    """Compile every CUDA source for sm_100a and link ``libb200q.so`` (``dev``: ``libb200q_dev.so``) in-tree."""
    lib_path = DEV_LIB_PATH if dev else LIB_PATH
    if not force and not _stale(lib_path):
        return lib_path
    build_dir = BUILD_DIR / "dev" if dev else BUILD_DIR
    build_dir.mkdir(exist_ok=True, parents=True)
    nvcc = _nvcc()
    flags = NVCC_FLAGS + (["-DB200Q_DEV"] if dev else [])
    sources = DEV_SOURCES if dev else SOURCES

    def compile_one(src: str) -> Path:
        obj = build_dir / (src[:-3] + ".o")
        cmd = [nvcc, *flags, "-c", str(CSRC / src), "-o", str(obj)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise B200QError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose and r.stderr.strip():
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(sources)) as ex:
        objs = list(ex.map(compile_one, sources))
    tmp = lib_path.with_suffix(".so.tmp")
    cmd = [nvcc, "-shared", "-o", str(tmp), *map(str, objs), "-gencode", "arch=compute_100a,code=sm_100a",
           "-cudart", "static"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise B200QError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, lib_path)
    return lib_path


# ------------------------------------------------------------------ C structs (mirror include/b200q.h)
class Requant(C.Structure):
    _fields_ = [("mult", C.c_void_p), ("bdiv", C.c_void_p), ("zp_out", C.c_int32), ("relu", C.c_int32),
                ("flags", C.c_int32), ("reserved", C.c_int32), ("mult_host", C.c_void_p), ("bdiv_host", C.c_void_p)]


RQ_BOUNDED = 1  # B200Q_RQ_BOUNDED
RQ_ACC22 = 2    # B200Q_RQ_ACC22


class Conv3x3(C.Structure):
    _fields_ = [("cin", C.c_int32), ("cout", C.c_int32), ("img", C.c_int32), ("zp_x", C.c_int32),
                ("w", C.c_void_p), ("corr", C.c_void_p), ("corr_host", C.c_void_p), ("rq", Requant)]


class Linear(C.Structure):
    _fields_ = [("k", C.c_int32), ("n", C.c_int32), ("zp_x", C.c_int32),
                ("w", C.c_void_p), ("corr", C.c_void_p), ("corr_host", C.c_void_p), ("rq", Requant)]


class StaticNet(C.Structure):
    _fields_ = [("in_inv_scale", C.c_float), ("in_zp", C.c_int32), ("conv", Conv3x3 * 6),
                ("fc1", Linear), ("fc2", Linear), ("out_scale", C.c_float)]


_P, _I, _L, _F = C.c_void_p, C.c_int, C.c_int64, C.c_float
_SIGNATURES = {
    "b200q_quantize_nchw_to_nhwc": [_P, _P, _L, _I, _I, _I, _I, _F, _I, _P],
    "b200q_quantize_flat": [_P, _P, _L, _F, _I, _P],
    "b200q_dequantize": [_P, _P, _L, _F, _I, _P],
    "b200q_relu_q": [_P, _P, _L, _I, _P],
    "b200q_max_pool2x2_nhwc": [_P, _P, _L, _I, _I, _I, _P],
    "b200q_minmax": [_P, _L, _P, _P, _P],
    "b200q_aminmax": [_P, _L, _P, _P, _P],
    "b200q_histc": [_P, _L, _F, _F, _I, _P, _P],
    "b200q_lut_u8": [_P, _P, _L, _P, _P],
    "b200q_graph_create": [C.POINTER(StaticNet), _P, _P, _L, _P, _L, _I, _P, C.POINTER(C.c_void_p)],
    "b200q_graph_create_u8": [C.POINTER(StaticNet), _P, _P, _P, _L, _P, _L, _I, _P, C.POINTER(C.c_void_p)],
    "b200q_graph_launch": [_P, _P],
    "b200q_graph_destroy": [_P],
    "b200q_conv3x3_first": [_P, _P, _L, C.POINTER(Conv3x3), _P],
    "b200q_quantize_conv3x3_first": [_P, _P, _L, _F, C.POINTER(Conv3x3), _P],
    "b200q_u8_conv3x3_first": [_P, _P, _L, _P, C.POINTER(Conv3x3), _P],
    "b200q_static_forward_u8": [C.POINTER(StaticNet), _P, _P, _P, _L, _P, _L, _P],
    "b200q_static_evaluate": [C.POINTER(StaticNet), _P, _P, _L, _P, _P, _P, _P, _L, _P],
    "b200q_static_evaluate_u8": [C.POINTER(StaticNet), _P, _P, _P, _L, _P, _P, _P, _P, _L, _P],
    "b200q_conv3x3_tc": [_P, _P, _L, C.POINTER(Conv3x3), _I, _P],
    "b200q_linear_tc": [_P, _P, _L, C.POINTER(Linear), _P],
    "b200q_linear_simt": [_P, _P, _L, C.POINTER(Linear), _P],
    "b200q_linear_dequant": [_P, _P, _L, C.POINTER(Linear), _F, _P],
    "b200q_linear_dynamic": [_P, _P, _L, _I, _I, _P, _P, _F, _P, _I, _P, _L, _P],
    "b200q_static_forward": [C.POINTER(StaticNet), _P, _P, _L, _P, _L, C.POINTER(C.c_void_p), _P],
    "b200q_static_forward_profiled": [C.POINTER(StaticNet), _P, _P, _L, _P, _L, C.POINTER(C.c_float), _P],
    "b200q_static_num_stages": [],
}

_DEV_SIGNATURES = {
    "b200q_conv12_fused": [_P, _P, _L, _F, C.POINTER(Conv3x3), C.POINTER(Conv3x3), _P],
    "b200q_conv3x3_simt": [_P, _P, _L, C.POINTER(Conv3x3), _P],
}

_lib = None
_dev_lib = None


def _open(path: Path, exports, signatures) -> C.CDLL:
    if not path.exists():
        raise B200QError(f"{path} is not built; run `python -c 'import __graft_entry__ as g; g.build()'` "
                         "(there is no CPU fallback for the CUDA path)")
    lib = C.CDLL(str(path))
    for name in exports:
        if not hasattr(lib, name):
            raise B200QError(f"{path} does not export {name}")
    lib.b200q_last_error.restype = C.c_char_p
    lib.b200q_last_error.argtypes = []
    lib.b200q_abi_version.restype = C.c_int
    lib.b200q_launch_count.restype = C.c_uint64
    lib.b200q_launch_count.argtypes = []
    lib.b200q_static_workspace_bytes.restype = C.c_int64
    lib.b200q_static_workspace_bytes.argtypes = [C.c_int64]
    lib.b200q_static_stage_name.restype = C.c_char_p
    lib.b200q_static_stage_name.argtypes = [C.c_int]
    for name, args in signatures.items():
        fn = getattr(lib, name)
        fn.restype = C.c_int
        fn.argtypes = args
    return lib


def load(build_if_missing: bool = False) -> C.CDLL:
    """dlopen ``libb200q.so`` and attach signatures.  Raises ``B200QError`` if it is not built."""
    global _lib
    if _lib is None:
        if build_if_missing and _stale():
            build()
        # B200Q_LIB: A-B timing of two builds of the PRODUCT library (development only)
        _lib = _open(Path(os.environ.get("B200Q_LIB", LIB_PATH)), EXPORTS, _SIGNATURES)
    return _lib


def load_dev(build_if_missing: bool = False) -> C.CDLL:
    """The development library (``-DB200Q_DEV``): product exports + ``DEV_EXPORTS``.  Tests and A-B scripts only."""
    global _dev_lib
    if _dev_lib is None:
        if build_if_missing and _stale(DEV_LIB_PATH):
            build(dev=True)
        _dev_lib = _open(DEV_LIB_PATH, DEV_EXPORTS, {**_SIGNATURES, **_DEV_SIGNATURES})
    return _dev_lib


def check(rc: int, what: str = "", lib: C.CDLL | None = None) -> None:
    """Turn a negative status into a Python exception (the reference's error convention is exceptions only)."""
    if rc != 0:
        msg = (lib or load()).b200q_last_error().decode(errors="replace")
        raise B200QError(f"{what or 'b200q call'} failed with status {rc}: {msg}")
