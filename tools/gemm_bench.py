"""Micro-benchmark of bd_conv_gemm on the transformer / U-Net shapes (CUDA events, L2 flushed by size).

    python tools/gemm_bench.py [shape,shape,...|all] [tf32,tf32x3,strict]

`strict` is the default mode's arithmetic (bf16 hi/lo operands, three products).  Each strict shape is timed
alternately with the default kernels ("tmem-A": split A operand in tensor memory, exact 96 / 192-column tiles) and
with BD_TC_SMEM_A=1 BD_TC_NO_EXACT=1 (A split in place in shared memory, power-of-two tiles); both switches are read
per call.  Every line carries the kernel template <TBK,TBN> the launch ran.
"""
import ctypes as C
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from demucs_b200 import _lib  # noqa: E402
from demucs_b200._lib import GemmDesc, ptr  # noqa: E402

_lib.build()
DEV = "cuda:0"
B, T = 16, 336                                      # one 16-segment forward of htdemucs: 336 frames per segment
TAPS9 = tuple((kt - 1, kf - 1) for kf in range(3) for kt in range(3))
# name, M, N, Cin, act, taps, F (frequency rows of a 3x3 decoder convolution; None: plain GEMM over M rows)
SHAPES = [("ffn1+gelu", 43008, 2048, 512, _lib.ACT_GELU, ((0, 0),), None),
          ("ffn2", 43008, 512, 2048, 0, ((0, 0),), None),
          ("qkv", 43008, 1536, 512, 0, ((0, 0),), None),
          ("proj", 43008, 512, 512, 0, ((0, 0),), None),
          ("proj_t", 21504, 512, 512, 0, ((0, 0),), None),
          ("ffn2_t", 21504, 512, 2048, 0, ((0, 0),), None),
          ("thin_glu", 2752512, 96, 48, _lib.ACT_GLU, ((0, 0),), None),
          ("dec3x3_n96", B * T * 512, 96, 48, _lib.ACT_GLU, TAPS9, 512),
          ("dec3x3_n192", B * T * 128, 192, 96, _lib.ACT_GLU, TAPS9, 128),
          ("dec3x3_n384", B * T * 32, 384, 192, _lib.ACT_GLU, TAPS9, 32)]
MATHS = {"tf32": _lib.MATH_TF32, "tf32x3": _lib.MATH_TF32X3, "strict": _lib.MATH_BF16X3}
OLD_PATH = {"BD_TC_SMEM_A": "1", "BD_TC_NO_EXACT": "1"}
ONLY = sys.argv[1].split(",") if len(sys.argv) > 1 and sys.argv[1] != "all" else None
MODES = sys.argv[2].split(",") if len(sys.argv) > 2 else ["tf32", "tf32x3", "strict"]
REPEATS = 5


def make(M, N, Cin, act, taps, F, math_mode):
    K = len(taps) * Cin
    n_out = N // 2 if act == _lib.ACT_GLU else N
    x = torch.randn(M, Cin, device=DEV)
    w = torch.randn(N, K, device=DEV) / K ** 0.5
    b = torch.randn(N, device=DEV)
    out = torch.empty(M, n_out, device=DEV)
    d = GemmDesc()
    d.M, d.N, d.K, d.Cin, d.taps, d.m1, d.m0 = M, N, K, Cin, len(taps), 1, 1
    for i, (d1, d0) in enumerate(taps):
        d.d1[i], d.d0[i] = d1, d0
    if F is None:
        d.I1, d.I0, d.J1, d.J0 = 1, M, 1, M
        d.xs_b, d.xs_1, d.xs_0, d.os_b, d.os_1, d.os_0 = M * Cin, 0, Cin, M * n_out, 0, n_out
    else:                                           # [B, T, F, Cin] channels-last, zero padding at the borders
        d.I1, d.I0, d.J1, d.J0 = T, F, T, F
        d.xs_b, d.xs_1, d.xs_0 = T * F * Cin, F * Cin, Cin
        d.os_b, d.os_1, d.os_0 = T * F * n_out, F * n_out, n_out
    d.xs_c = 1
    d.stat_div, d.stat_mul, d.stat_mod = d.I0, 1, 1
    d.x, d.w, d.bias, d.out, d.act, d.math = ptr(x), ptr(w), ptr(b), ptr(out), act, math_mode
    keep = [x, w, b, out]
    if math_mode == _lib.MATH_BF16X3:               # pre-split bf16 weight planes, as the engine makes them
        w_hi = w.to(torch.bfloat16)
        w_lo = (w - w_hi.float()).to(torch.bfloat16)
        d.w16_hi, d.w16_lo = ptr(w_hi), ptr(w_lo)
        keep += [w_hi, w_lo]
    return d, keep


def set_env(env):
    for k in OLD_PATH:
        os.environ.pop(k, None)
    os.environ.update(env)


def time_ms(d, n=10):
    for _ in range(3):
        _lib.call("bd_conv_gemm", C.byref(d), 0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        _lib.call("bd_conv_gemm", C.byref(d), 0)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def label(d):
    code = _lib.lib().bd_conv_gemm_arm(C.byref(d))
    return f"<{code // 1000},{code % 1000}>"


props = torch.cuda.get_device_properties(0)
print(f"device: {props.name}, {props.multi_processor_count} SMs; BD_TC_NO_WIDE={os.environ.get('BD_TC_NO_WIDE', '')}",
      flush=True)
for mname in MODES:
    variants = [("tmem-A", {}), ("smem-A", OLD_PATH)] if mname == "strict" else [("", {})]
    for name, M, N, Cin, act, taps, F in SHAPES:
        if ONLY and name not in ONLY:
            continue
        d, keep = make(M, N, Cin, act, taps, F, MATHS[mname])
        flops = 2.0 * M * N * d.K
        times = {v: [] for v, _ in variants}
        labels = {}
        for _ in range(REPEATS):                    # the variants alternate, so drifting clocks hit both alike
            for v, env in variants:
                set_env(env)
                labels[v] = label(d)
                times[v].append(time_ms(d))
        set_env({})
        for v, _ in variants:
            ms = statistics.median(times[v])
            print(f"{mname:7s} {v:7s} {name:12s} {labels[v]:9s} M={M} N={N} K={d.K} taps={len(taps)}: {ms:7.3f} ms "
                  f"(min {min(times[v]):.3f} max {max(times[v]):.3f})  {flops / ms / 1e9:7.1f} TF/s", flush=True)
        del keep
