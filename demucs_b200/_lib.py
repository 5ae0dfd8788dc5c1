"""ctypes binding of libdemucs_b200.so (the C ABI declared in include/demucs_b200.h).

There is NO fallback: if the shared library is missing or a kernel call fails, an exception
is raised.  ``build()`` compiles the library in-tree with nvcc for sm_100a.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import typing as tp

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.path.join(HERE, "libdemucs_b200.so")
SOURCES = ["api.cu", "spectral.cu", "gemm_simt.cu", "gemm_tc.cu", "gemm_tc_b16x3.cu", "gemm_tc_b16x3_smem.cu", "gemm_tc_b16.cu", "norm.cu", "dconv.cu", "attention.cu", "attention_tc.cu", "attention_b16.cu",
           "ola.cu", "audio.cu", "hdemucs.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--use_fast_math=false"]

BD_MAX_TAPS = 9
A_NONE, A_GN_GELU, A_ITEM_AFFINE = 0, 1, 2
ACT_NONE, ACT_GELU, ACT_GLU = 0, 1, 2
MATH_FP32, MATH_TF32, MATH_TF32X3, MATH_BF16X3, MATH_BF16 = 0, 1, 2, 3, 4


class KernelError(RuntimeError):
    pass


class GemmDesc(C.Structure):
    """Mirror of ``bd_gemm_desc`` (include/demucs_b200.h)."""
    _fields_ = [
        ("M", C.c_int), ("N", C.c_int), ("K", C.c_int),
        ("Cin", C.c_int), ("taps", C.c_int),
        ("I1", C.c_int), ("I0", C.c_int),
        ("m1", C.c_int), ("m0", C.c_int), ("J1", C.c_int), ("J0", C.c_int),
        ("d1", C.c_int * BD_MAX_TAPS), ("d0", C.c_int * BD_MAX_TAPS),
        ("xs_b", C.c_longlong), ("xs_1", C.c_longlong), ("xs_0", C.c_longlong), ("xs_c", C.c_longlong),
        ("x", C.c_void_p), ("w", C.c_void_p), ("bias", C.c_void_p),
        ("a_mode", C.c_int), ("a_stats", C.c_void_p), ("a_stats_stride", C.c_int),
        ("a_gamma", C.c_void_p), ("a_beta", C.c_void_p),
        ("e_stats", C.c_void_p), ("e_gamma", C.c_void_p), ("e_beta", C.c_void_p),
        ("act", C.c_int), ("rowbias", C.c_void_p), ("rowbias_period", C.c_int),
        ("resid", C.c_void_p), ("scale", C.c_void_p), ("addend", C.c_void_p),
        ("out", C.c_void_p), ("os_b", C.c_longlong), ("os_1", C.c_longlong), ("os_0", C.c_longlong),
        ("convt", C.c_int), ("O0", C.c_int), ("oc_split", C.c_int), ("oc_stride", C.c_longlong),
        ("stats_out", C.c_void_p), ("stat_div", C.c_int), ("stat_mul", C.c_int), ("stat_mod", C.c_int),
        ("math", C.c_int), ("w16_hi", C.c_void_p), ("w16_lo", C.c_void_p), ("x_bf16", C.c_int), ("out_bf16", C.c_int),
    ]


_P, _I, _LL, _D, _F = C.c_void_p, C.c_int, C.c_longlong, C.c_double, C.c_float
SIGNATURES: tp.Dict[str, tp.List] = {
    "bd_stft_cac": [_P, _P, _P, _P, _P, _I, _I, _I, _P],
    "bd_finalize_item_norm": [_P, _P, _I, _D, _D, _P],
    "bd_istft_frames": [_P, _P, _P, _P, _P, _I, _I, _I, _P],
    "bd_istft_ola": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "bd_ola_combine": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "bd_conv_gemm": [C.POINTER(GemmDesc), _P],
    "bd_conv_gemm_arm": [C.POINTER(GemmDesc)],
    "bd_finalize_group_stats": [_P, _P, _I, _D, _P],
    "bd_dconv_tail": [_P, _P, _P, _P, _P, _P, _LL, _I, _LL, _I, _P],
    "bd_encoder_conv0": [_P, _I, _P, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P],
    "bd_dconv_conv3": [_P, _P, _P, _P, _I, _P, _LL, _I, _I, _LL, _I, _I, _I, _P],
    "bd_dconv_expand_stats": [_P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _LL, _I, _LL, _I, _P],
    "bd_dconv_expand_update": [_P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _LL, _I, _LL, _I, _I, _P],
    "bd_gn_gelu_apply": [_P, _P, _P, _P, _LL, _I, _LL, _I, _P],
    "bd_layer_norm": [_P, _P, _P, _P, _P, _I, _LL, _I, _I, _P],
    "bd_attention_bf16": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "bd_item_stats": [_P, _P, _I, _LL, _P],
    "bd_group_norm_apply": [_P, _P, _P, _P, _I, _LL, _I, _P],
    "bd_attention_workspace": [_I, _I, _I, _I, _I],
    "bd_attention": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P],
    "bd_overlap_add": [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _LL, _LL, _LL, _LL, _LL, _P, _F, _I, _P],
    "bd_gather_segments": [_P, _P, _I, _I, _LL, _LL, _LL, _I, _I, _I, _I, _I, _P],
    "bd_gn_stats": [_P, _P, _I, _LL, _I, _I, _P],
    "bd_gn_act": [_P, _P, _P, _P, _P, _P, _I, _LL, _LL, _LL, _I, _I, _I, _LL, _P],
    "bd_lstm_frame": [_P, _P, _I, _LL, _I, _I, _I, _I, _P],
    "bd_lstm_unframe_add": [_P, _P, _P, _I, _LL, _I, _I, _I, _I, _P],
    "bd_lstm_bidir": [_P, _P, _P, _P, _I, _I, _I, _P],
    "bd_local_state": [_P, _P, _P, _I, _I, _I, _I, _P],
    "bd_convert_channels": [_P, _P, _I, _I, _I, _LL, _P],
    "bd_resample_frac": [_P, _P, _P, _I, _I, _I, _LL, _LL, _I, _I, _I, _P],
    "bd_absmax": [_P, _P, _LL, _P],
    "bd_clip_pcm": [_P, _P, _I, _LL, _I, _P, _I, _P],
}
VALUE_CALLS = {"bd_attention_workspace"}          # entry points that return a value, not a status
EXPORTS = ["bd_last_error", "bd_version"] + list(SIGNATURES)

_lib: tp.Optional[C.CDLL] = None


def build(verbose: bool = False, force: bool = False) -> str:
    """Compile csrc/*.cu into libdemucs_b200.so for sm_100a (cross-compiles without a GPU).

    Every source becomes its own object file (compiled in parallel, cached under csrc/.obj by the content
    hash of the source, the shared headers and the flags), then one link step."""
    import hashlib
    from concurrent.futures import ThreadPoolExecutor
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    headers = [os.path.join(os.path.dirname(HERE), "include", "demucs_b200.h")]
    headers += sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh"))
    flags = [f for f in NVCC_FLAGS if not f.startswith("--use_fast_math")]
    flags += os.environ.get("BD_NVCC_DEFS", "").split()     # experiment knobs, e.g. -DBD_TC_PIPE_BYTES=196608
    base = hashlib.sha256(" ".join(flags).encode())
    for dep in headers:
        with open(dep, "rb") as f:
            base.update(f.read())
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objdir = os.path.join(CSRC, ".obj")
    os.makedirs(objdir, exist_ok=True)
    total = base.copy()
    jobs = []
    for src in srcs:
        d = base.copy()
        with open(src, "rb") as f:
            data = f.read()
        d.update(data)
        total.update(data)
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        jobs.append((src, obj, d.hexdigest()))
    stamp_path = LIB_PATH + ".stamp"
    stamp = total.hexdigest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(stamp_path):
        with open(stamp_path) as f:
            if f.read().strip() == stamp:       # content hash: file times do not survive a snapshot
                return LIB_PATH

    def compile_one(job):
        src, obj, digest = job
        if not force and os.path.exists(obj) and os.path.exists(obj + ".stamp"):
            with open(obj + ".stamp") as f:
                if f.read().strip() == digest:
                    return ""
        cmd = [nvcc] + flags + (["-Xptxas=-v"] if verbose else []) + ["-c", "-o", obj, src]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise KernelError(f"nvcc failed on {src}:\n{res.stdout}\n{res.stderr}")
        with open(obj + ".stamp", "w") as f:
            f.write(digest)
        return res.stderr

    with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as pool:
        logs = list(pool.map(compile_one, jobs))
    if verbose:
        print("\n".join(logs))
    res = subprocess.run([nvcc] + flags + ["-shared", "-o", LIB_PATH] + [j[1] for j in jobs], capture_output=True, text=True)
    if res.returncode != 0:
        raise KernelError(f"link failed:\n{res.stdout}\n{res.stderr}")
    with open(stamp_path, "w") as f:
        f.write(stamp)
    return LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise KernelError(
                f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(demucs_b200 has no CPU or PyTorch fallback path)")
        handle = C.CDLL(LIB_PATH)
        handle.bd_last_error.restype = C.c_char_p
        handle.bd_last_error.argtypes = []
        handle.bd_version.restype = C.c_int
        for name, args in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = C.c_longlong if name in VALUE_CALLS else C.c_int
            fn.argtypes = args
        _lib = handle
    return _lib


# Test seam: tests/abi_emulator.py installs a numpy restatement of the C ABI here so that the HOST
# logic (descriptor construction, weight packing, batching, sharding) can be checked on a machine
# without a GPU.  Product code never sets it; with it unset every call goes to the CUDA library.
TEST_HOOK: tp.Optional[tp.Callable] = None


def call(name: str, *args) -> None:
    if TEST_HOOK is not None:
        return TEST_HOOK(name, *args)
    rc = getattr(lib(), name)(*args)
    if rc != 0:
        raise KernelError(f"{name} failed ({rc}): {lib().bd_last_error().decode()}")


def call_value(name: str, *args) -> int:
    """Entry points that return a size rather than a status code."""
    if TEST_HOOK is not None:
        return TEST_HOOK(name, *args)
    return int(getattr(lib(), name)(*args))


def ptr(t) -> tp.Optional[int]:
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()
