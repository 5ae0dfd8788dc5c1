"""The implicit GEMM (bd_conv_gemm) against a float64 statement of bd_gemm_desc, descriptor by descriptor.

``ref_conv_gemm`` restates include/demucs_b200.h in torch float64, in the header's order: the A gather with its zero
taps and prologues, bias, the epilogue GroupNorm, the activation, the row bias, LayerScale + residual, the skip addend,
the output index (transposed-conv phases and crop, channel-group planes) and the statistics of the stored values.
It is pinned on the CPU to the numpy ABI emulator and to torch's own convolutions on the engine's weight packings.

``Shadow`` wraps demucs_b200._lib.call.  For every bd_conv_gemm / bd_attention(_bf16) launch it computes each operand's
extent from the header's index arithmetic, checks that the extent lies inside one live allocation (before the launch,
so that a descriptor reaching outside its tensors is reported instead of run), snapshots the operands, runs the
launch and compares its output with the float64 statement of the snapshots:
- rel-L2 of the written elements within the arm's bound, the worst 128-row block (rows m) within 4x that bound;
- every element of the output range the header does not write (pitch padding, cropped transposed-conv positions,
  channel-group gaps) bitwise unchanged;
- the stats_out increments equal to the float64 sums of the values actually stored, and to the reference sums.
It checks every GEMM and attention launch of real forwards (htdemucs in every mode, htdemucs_6s, hdemucs_mmi), and a
matrix of synthetic descriptors that switches each fused feature on in every arithmetic and reaches every kernel
template the dispatcher can instantiate.

Largest rel-L2 per call over the forwards and the matrix below, measured on one NVIDIA B200 (1000 W power limit), by
mode and feature (the arm that ran in brackets; "bf16" mode runs the U-Net convolutions in tf32):
    fp32    [fp32]    1.2e-6 worst (taps3 / stats_item); convt1 5.3e-7, oc_split 1.8e-7, e_stats 1.7e-7, rowbias 1.0e-7,
                      a_item_affine 1.3e-7, addend 6.9e-7, N%4 2.2e-7; attention 7.7e-7
    tf32    [tf32]    9.5e-4 worst (gelu); convt2 8.8e-4, oc_split 7.4e-4, e_stats 8.1e-4, rowbias 5.8e-4; attention 7.2e-4
    tf32x3  [tf32x3]  2.6e-5 worst (3x3 rewrite, K = 3456); convt2 5.8e-6, e_stats 3.4e-7, rowbias 2.6e-7; attention 1.4e-5
    strict  [bf16x3]  1.7e-5 worst (K = 4608); convt2 5.4e-6, oc_split 4.5e-6, e_stats 4.8e-6, rowbias 3.1e-6;
                      attention 4.4e-6
    bf16    [bf16]    2.5e-3 worst (x16 / out16 GELU); resid 2.5e-4; bf16-tensor attention 1.7e-3
The worst 128-row block was at most 1.7x the whole call.  The split arms (tf32x3, bf16x3) lose accuracy linearly in K
(7.6e-9 * K and 3.9e-9 * K at K >= 3456, against a sqrt(K) growth for the CUDA-core arm): the tensor core's fp32
accumulation is not round-to-nearest, so its error does not average out.  Their bound is therefore the fixed one of
test_gpu_gemm.py up to K = 770 and 3x the measured slope above (K_SLOPE).  The BF16 bound is 3x its measured worst; the
FP32 and TF32 bounds stay those of test_gpu_gemm.py (2.4x and 2.1x the measured worst).
"""
import contextlib
import ctypes as C
import math
import sys
from collections import namedtuple

import pytest
import torch
import torch.nn.functional as F

import abi_emulator as E
from _fixtures import forward_fixture_inputs, golden, htdemucs_config, init_weights, small_config, synth_mix
from demucs_b200 import _lib
from demucs_b200._lib import GemmDesc
from demucs_b200.engine import MODES, Engine, _interleave_glu, conv_w, convtr_w, convtr_w3

F64, F32, BF16 = torch.float64, torch.float32, torch.bfloat16
ES = {F32: 4, BF16: 2, F64: 8}
INT_OF = {F32: torch.int32, BF16: torch.int16, F64: torch.int64}
CHUNK = 1 << 23                      # elements of the float64 im2col per row chunk
# rel-L2 bound of one call, by the arithmetic that ran (a descriptor the tensor-core arm declines runs in fp32)
BOUND = {_lib.MATH_FP32: 3e-6, _lib.MATH_TF32X3: 2e-5, _lib.MATH_BF16X3: 2e-5, _lib.MATH_TF32: 2e-3,
         _lib.MATH_BF16: 7e-3}
K_SLOPE = {_lib.MATH_TF32X3: 2.3e-8, _lib.MATH_BF16X3: 1.2e-8}   # split arms: error linear in K (module docstring)
OUT16_ROUNDING = 2.0 ** -9           # bf16 output: one rounding, 2^-9 relative at most (1.7e-3 rms measured)


def gemm_bound(math_, K, out16=False):
    return max(BOUND[math_], K_SLOPE.get(math_, 0.0) * K) + (OUT16_ROUNDING if out16 else 0.0)
ATT_BOUND = {_lib.MATH_FP32: 3e-6, _lib.MATH_TF32: 2e-3, _lib.MATH_TF32X3: 3e-5, _lib.MATH_BF16X3: 3e-5,
             _lib.MATH_BF16: 8e-3, "bf16-tensor": 6e-3}
MATH_NAME = {_lib.MATH_FP32: "fp32", _lib.MATH_TF32: "tf32", _lib.MATH_TF32X3: "tf32x3", _lib.MATH_BF16X3: "bf16x3",
             _lib.MATH_BF16: "bf16"}


# ---------------------------------------------------------------------------------------------------------------------
# raw memory
class _CudaBytes:
    def __init__(self, p, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "|u1", "data": (p, False), "version": 2}


def raw_bytes(p, nbytes, device):
    """uint8 view of nbytes of device (or host) memory at address p."""
    if torch.device(device).type == "cuda":
        return torch.as_tensor(_CudaBytes(p, nbytes), device=device)
    return torch.frombuffer((C.c_uint8 * nbytes).from_address(p), dtype=torch.uint8)


def host_read(p, n, dtype):
    return raw_bytes(p, n * ES[dtype], "cpu").view(dtype)


# ---------------------------------------------------------------------------------------------------------------------
# float64 statement of bd_gemm_desc
Ext = namedtuple("Ext", "name ptr lo hi dtype")          # elements [lo, hi] of `dtype` after ptr
Ref = namedtuple("Ref", "vals idx rows stats")            # stored values, their flat output indices, their rows m,
#                                                           per-slab (sum, sumsq) increments (None without stats_out)


def n_out(d):
    """Channels per output position."""
    return d.N // 2 if d.act == _lib.ACT_GLU else (d.N // 4 if d.convt else d.N)


def _cols(d, dev):
    """(output channel, transposed-conv phase) of each epilogue column: N/2 columns after GLU, n = phase*Cout + channel
    for a transposed conv."""
    if d.act == _lib.ACT_GLU:
        n = torch.arange(d.N // 2, device=dev)
        return n, torch.zeros_like(n)
    n = torch.arange(d.N, device=dev)
    if d.convt:
        return n % (d.N // 4), n // (d.N // 4)
    return n, torch.zeros_like(n)


def _coords(d, m):
    """Row m = (b * I1 + i1) * I0 + i0."""
    t = m // d.I0
    return t // d.I1, t % d.I1, m % d.I0


def slab_of(d, m):
    return (m // d.stat_div) * d.stat_mul + m % d.stat_mod


def _tap_offsets(d, m, tap):
    """Offset of x[b, j1, j0, 0] for rows m and whether the tap lies inside [0, J1) x [0, J0)."""
    b, i1, i0 = _coords(d, m)
    j1, j0 = i1 * d.m1 + d.d1[tap], i0 * d.m0 + d.d0[tap]
    ok = (j1 >= 0) & (j1 < d.J1) & (j0 >= 0) & (j0 < d.J0)
    return b * d.xs_b + j1 * d.xs_1 + j0 * d.xs_0, ok, b


def _out_index(d, m, ch, ph):
    """Flat output index [rows, columns] and whether it is written (transposed conv: 0 <= o0 < O0)."""
    b, i1, i0 = _coords(d, m)
    colofs = ch if not d.oc_split else (ch // d.oc_split) * d.oc_stride + ch % d.oc_split
    if d.convt:
        o0 = 4 * i0[:, None] + ph[None, :] - (2 if d.convt == 1 else 0)
        ok = (o0 >= 0) & (o0 < d.O0)
    else:
        o0 = i0[:, None].expand(-1, ch.numel())
        ok = torch.ones_like(o0, dtype=torch.bool)
    return (b * d.os_b + i1 * d.os_1)[:, None] + o0 * d.os_0 + colofs[None, :], ok


def _row_chunks(d, dev, width):
    step = max(1, CHUNK // max(1, width))
    for m0 in range(0, d.M, step):
        yield torch.arange(m0, min(d.M, m0 + step), device=dev)


def extents(d, dev="cpu"):
    """Every operand the descriptor reads or writes, as element ranges derived from the header's index arithmetic."""
    N, K, no = d.N, d.K, n_out(d)
    ch, ph = _cols(d, dev)
    ci = torch.arange(d.Cin, device=dev) * d.xs_c
    big = 1 << 62
    xlo, xhi, olo, ohi, smax = big, -1, big, -1, -1
    slabs = d.stats_out or d.e_stats or d.a_mode == _lib.A_GN_GELU
    for m in _row_chunks(d, dev, N + d.taps):
        for tap in range(d.taps):
            base, ok, _ = _tap_offsets(d, m, tap)
            if ok.any():
                xlo = min(xlo, int(base[ok].min() + ci.min()))
                xhi = max(xhi, int(base[ok].max() + ci.max()))
        idx, ok = _out_index(d, m, ch, ph)
        if ok.any():
            olo, ohi = min(olo, int(idx[ok].min())), max(ohi, int(idx[ok].max()))
        if slabs:
            smax = max(smax, int(slab_of(d, m).max()))
    items = d.M // (d.I1 * d.I0)
    ext = []

    def add(name, p, lo, hi, dt=F32):
        if p:
            ext.append(Ext(name, p, lo, hi, dt))
    add("x", d.x, xlo, xhi, BF16 if d.x_bf16 else F32)
    add("w", d.w, 0, N * K - 1)
    add("w16_hi", d.w16_hi, 0, N * K - 1, BF16)
    add("w16_lo", d.w16_lo, 0, N * K - 1, BF16)
    add("bias", d.bias, 0, N - 1)
    if d.a_mode == _lib.A_ITEM_AFFINE:
        add("a_stats", d.a_stats, 0, (items - 1) * d.a_stats_stride + 2)
    elif d.a_mode == _lib.A_GN_GELU:
        add("a_stats", d.a_stats, 0, 2 * smax + 1)
        add("a_gamma", d.a_gamma, 0, d.Cin - 1)
        add("a_beta", d.a_beta, 0, d.Cin - 1)
    if d.e_stats:
        add("e_stats", d.e_stats, 0, 2 * smax + 1)
        add("e_gamma", d.e_gamma, 0, N - 1)
        add("e_beta", d.e_beta, 0, N - 1)
    if d.rowbias:
        add("rowbias", d.rowbias, 0, min(d.rowbias_period, d.M) * no - 1)
    if d.resid:
        add("resid", d.resid, olo, ohi)
        add("scale", d.scale, 0, no - 1)
    add("addend", d.addend, olo, ohi)
    add("out", d.out, olo, ohi, BF16 if d.out_bf16 else F32)
    add("stats_out", d.stats_out, 0, 2 * smax + 1, F64)
    return ext


def ref_conv_gemm(d, read, dev="cpu"):
    """float64 bd_conv_gemm of descriptor d; read(ptr, n, dtype) returns n elements at ptr (device or host memory)."""
    ext = {e.name: e for e in extents(d, dev)}

    def load(name):
        e = ext[name]
        return read(e.ptr + e.lo * ES[e.dtype], e.hi - e.lo + 1, e.dtype).to(dev), e.lo

    def vec(name):
        return load(name)[0].to(F64)
    N, K = d.N, d.K
    ch, ph = _cols(d, dev)
    ci = torch.arange(d.Cin, device=dev) * d.xs_c
    X, xlo = load("x")
    W = vec("w").view(N, K)
    bias = vec("bias") if d.bias else None
    if d.a_mode != _lib.A_NONE:
        ast = vec("a_stats")
    if d.a_mode == _lib.A_GN_GELU:
        ast, ag, ab = ast.view(-1, 2), vec("a_gamma"), vec("a_beta")
    if d.e_stats:
        est, eg, eb = vec("e_stats").view(-1, 2), vec("e_gamma"), vec("e_beta")
    rb = vec("rowbias").view(-1, n_out(d)) if d.rowbias else None
    if d.resid:
        res, olo = load("resid")
        sc = vec("scale")[ch] if d.scale else 1.0
    if d.addend:
        add, olo = load("addend")
    stats = None
    if d.stats_out:
        stats = torch.zeros(ext["stats_out"].hi // 2 + 1, 2, dtype=F64, device=dev)
    vals, idxs, rows = [], [], []
    for m in _row_chunks(d, dev, K + N):
        # 1. A(m, tap, ci), zero outside [0,J1) x [0,J0), prologue transforms before the zero padding
        A = torch.zeros(m.numel(), d.taps, d.Cin, dtype=F64, device=dev)
        for tap in range(d.taps):
            base, ok, b = _tap_offsets(d, m, tap)
            a = X[base[ok][:, None] + ci[None, :] - xlo].to(F64)
            if d.a_mode == _lib.A_GN_GELU:
                sl = slab_of(d, m[ok])
                a = F.gelu((a - ast[sl, :1]) * ast[sl, 1:] * ag + ab)
            elif d.a_mode == _lib.A_ITEM_AFFINE:
                bo = b[ok] * d.a_stats_stride
                a = (a - ast[bo][:, None]) * ast[bo + 2][:, None]
            A[:, tap][ok] = a
        # 2. acc + bias
        v = A.view(m.numel(), K) @ W.t()
        if bias is not None:
            v = v + bias
        # 3. GroupNorm of the pre-activation output on the slab map
        if d.e_stats:
            sl = slab_of(d, m)
            v = (v - est[sl, :1]) * est[sl, 1:] * eg + eb
        # 4. activation; GLU = value[2c] * sigmoid(gate[2c + 1])
        if d.act == _lib.ACT_GELU:
            v = F.gelu(v)
        elif d.act == _lib.ACT_GLU:
            v = v[:, 0::2] * torch.sigmoid(v[:, 1::2])
        # 5. row bias [(m % period) * Nout + channel]
        if rb is not None:
            v = v + rb[m % d.rowbias_period][:, ch]
        # 8. output index (needed by 6 / 7, which read at it)
        idx, ok = _out_index(d, m, ch, ph)
        # 6. resid + scale * v, 7. + addend
        if d.resid:
            v = res[torch.where(ok, idx, olo) - olo].to(F64) + sc * v
        if d.addend:
            v = v + add[torch.where(ok, idx, olo) - olo].to(F64)
        vals.append(v[ok])
        idxs.append(idx[ok])
        rows.append(m[:, None].expand_as(idx)[ok])
        # 9. statistics of the stored values
        if stats is not None:
            z = torch.where(ok, v, 0.0)
            stats.index_add_(0, slab_of(d, m), torch.stack([z.sum(1), (z * z).sum(1)], 1))
    return Ref(torch.cat(vals), torch.cat(idxs), torch.cat(rows), stats)


# ---------------------------------------------------------------------------------------------------------------------
# live allocations
def cuda_blocks():
    """(address, size) of every active block of the caching allocator."""
    out = []
    for seg in torch.cuda.memory_snapshot():
        addr = seg["address"]
        for blk in seg["blocks"]:
            a = blk.get("address", addr)
            if blk["state"] == "active_allocated":
                out.append((a, blk["size"]))
            addr = a + blk["size"]
    return out


def _tensors(obj, seen, depth=0):
    if torch.is_tensor(obj):
        yield obj
        return
    if depth > 5 or id(obj) in seen:
        return
    seen.add(id(obj))
    if isinstance(obj, dict):
        items = list(obj.values())
    elif isinstance(obj, (list, tuple)):
        items = obj
    elif type(obj).__module__.startswith(("demucs_b200", __name__)) and hasattr(obj, "__dict__"):
        items = list(vars(obj).values())
    else:
        return
    for v in items:
        yield from _tensors(v, seen, depth + 1)


def host_blocks(*roots):
    """Storages of every tensor reachable from roots (host memory: the CPU stand-in for the allocator's blocks)."""
    def blocks():
        out = {}
        for t in _tensors(list(roots), set()):
            s = t.untyped_storage()
            out[s.data_ptr()] = s.nbytes()
        return list(out.items())
    return blocks


# ---------------------------------------------------------------------------------------------------------------------
def features(d):
    f = []
    if d.taps > 1:
        f.append(f"taps{d.taps}")
    if d.m0 == 4:
        f.append("stride4")
    if d.convt:
        f.append(f"convt{d.convt}")
    if d.oc_split:
        f.append("oc_split")
    if d.a_mode:
        f.append({_lib.A_GN_GELU: "a_gn_gelu", _lib.A_ITEM_AFFINE: "a_item_affine"}[d.a_mode])
    if d.xs_c != 1:
        f.append("channel_major")
    if d.e_stats:
        f.append("e_stats")
    if d.act:
        f.append({_lib.ACT_GELU: "gelu", _lib.ACT_GLU: "glu"}[d.act])
    if d.rowbias:
        f.append("rowbias")
    if d.resid:
        f.append("resid_in_place" if d.resid == d.out else "resid")
    if d.addend:
        f.append("addend")
    if not d.out:
        f.append("stats_only")
    if d.stats_out:
        f.append("stats_freq" if d.stat_mod > 1 else "stats_item")
    if d.x_bf16:
        f.append("x16")
    if d.out_bf16:
        f.append("out16")
    if d.I1 > 1 and d.I0 < 128:
        f.append("R0<128")
    if d.N % 4:
        f.append("N%4")
    return f or ["plain"]


class Shadow:
    """Stand-in for demucs_b200._lib.call that checks every GEMM and attention launch against float64 (see module
    docstring).  ``blocks()`` lists the live allocations; failures are collected, not raised, unless an operand lies
    outside its allocation (then the launch is not made)."""

    def __init__(self, device, blocks, real=None, tag=""):
        self.dev = torch.device(device)
        self.blocks = blocks
        self.real = real or _lib.call
        self.tag = tag
        self.site, self.label = "", ""
        self.records, self.failures = [], []
        self.worst = {}
        self.quiet = False

    # -- plumbing
    def __call__(self, name, *args):
        if name == "bd_conv_gemm":
            return self.gemm(*args)
        if name in ("bd_attention", "bd_attention_bf16"):
            return self.attention(name, *args)
        return self.forward(name, *args)

    def forward(self, name, *args):
        if self.dev.type == "cpu" and _host_bf16(self.real, name, args):
            return None
        return self.real(name, *args)

    def sync(self):
        if self.dev.type == "cuda":
            torch.cuda.synchronize(self.dev)

    def check_inside(self, ext):
        live = self.blocks()
        for e in ext:
            lo, hi = e.ptr + e.lo * ES[e.dtype], e.ptr + (e.hi + 1) * ES[e.dtype]
            if not any(a <= lo and hi <= a + n for a, n in live):
                raise AssertionError(f"{self.site} {self.label}: operand {e.name} [{lo:#x}, {hi:#x}) is not inside one live "
                                     f"allocation")

    def snapshot(self, ext):
        regions = [(e.ptr + e.lo * ES[e.dtype], (e.hi - e.lo + 1) * ES[e.dtype]) for e in ext]
        snaps = [(p, n, raw_bytes(p, n, self.dev).clone()) for p, n in regions]

        def read(p, n, dtype):
            nb = n * ES[dtype]
            for q, qn, buf in snaps:
                if q <= p and p + nb <= q + qn:
                    return buf[p - q:p - q + nb].view(dtype)
            raise AssertionError(f"reference read outside the snapshots: {p:#x} + {nb}")
        return read, snaps

    def note(self, key, err, line, problems):
        self.records.append(line)
        if not self.quiet:
            print(line + ("  <-- " + "; ".join(problems) if problems else ""))
        for k in key:
            self.worst[k] = max(self.worst.get(k, 0.0), err)
        if problems:
            self.failures.append(f"{line}: {'; '.join(problems)}")

    # -- bd_conv_gemm
    def gemm(self, dref, stream):
        d = dref._obj
        self.sync()
        ext = extents(d, self.dev)
        self.check_inside(ext)
        by = {e.name: e for e in ext}
        read, _ = self.snapshot(ext)
        arm = _lib.lib().bd_conv_gemm_arm(dref) if self.dev.type == "cuda" else 0
        rc = self.forward("bd_conv_gemm", dref, stream)
        self.sync()
        ref = ref_conv_gemm(d, read, self.dev)
        math_ = d.math if arm else _lib.MATH_FP32
        bound = gemm_bound(math_, d.K, d.out_bf16)
        err, problems = self.compare_gemm(d, by, read, ref, bound)
        feats = features(d)
        line = (f"{self.tag} {self.site:<16} {self.label:<24} arm={MATH_NAME[math_]}:{arm:<5} M={d.M} N={d.N} K={d.K} "
                f"[{','.join(feats)}] rel-L2 {err[0]:.2e} block {err[1]:.2e} stats {err[2]:.1e}")
        self.note([(self.tag, MATH_NAME[math_], f) for f in feats], err[0], line, problems)
        self.last = dict(arm=arm, math=math_, err=err, ref=ref, bound=bound)
        return rc

    def compare_gemm(self, d, by, read, ref, bound):
        problems = []
        e_rel = e_blk = e_st = 0.0
        got = None
        if d.out:
            eo = by["out"]
            n = eo.hi - eo.lo + 1
            before = read(eo.ptr + eo.lo * ES[eo.dtype], n, eo.dtype)
            after = raw_bytes(eo.ptr + eo.lo * ES[eo.dtype], n * ES[eo.dtype], self.dev).view(eo.dtype)
            got = after[ref.idx - eo.lo].to(F64)
            if not torch.isfinite(got).all():
                problems.append(f"{int((~torch.isfinite(got)).sum())} written elements not finite")
            diff = torch.nan_to_num(got - ref.vals, nan=1e30, posinf=1e30, neginf=1e30)
            e_rel = float(diff.norm() / ref.vals.norm().clamp_min(1e-30))
            blk = ref.rows // 128
            nb = int(blk.max()) + 1
            err2 = torch.zeros(nb, dtype=F64, device=self.dev).index_add_(0, blk, diff * diff)
            ref2 = torch.zeros(nb, dtype=F64, device=self.dev).index_add_(0, blk, ref.vals * ref.vals)
            e_blk = float((err2 / ref2.clamp_min(1e-60)).sqrt().max())
            written = torch.zeros(n, dtype=torch.bool, device=self.dev)
            written[ref.idx - eo.lo] = True
            it = INT_OF[eo.dtype]
            moved = (before.view(it) != after.view(it)) & ~written
            if moved.any():
                problems.append(f"{int(moved.sum())} elements the header does not write changed "
                                f"(first at offset {int(moved.nonzero()[0]) + eo.lo})")
            if e_rel > bound:
                problems.append(f"rel-L2 {e_rel:.2e} > {bound:.1e}")
            if e_blk > 4 * bound:
                problems.append(f"worst 128-row block rel-L2 {e_blk:.2e} > {4 * bound:.1e}")
        if d.stats_out:
            es = by["stats_out"]
            nsl = es.hi // 2 + 1
            before = read(es.ptr, 2 * nsl, F64).view(nsl, 2)
            after = raw_bytes(es.ptr, 16 * nsl, self.dev).view(F64).view(nsl, 2).clone()
            delta = after - before
            sl = slab_of(d, ref.rows)
            cnt = torch.zeros(nsl, dtype=F64, device=self.dev).index_add_(0, sl, torch.ones_like(ref.vals))
            q = ref.stats[:, 1]
            tol_s, tol_q = (cnt * q).sqrt(), q
            dv = (delta - ref.stats).abs()
            e_st = float(torch.maximum(dv[:, 0] / tol_s.clamp_min(1e-30), dv[:, 1] / tol_q.clamp_min(1e-30)).max())
            if (dv[:, 0] > 4 * bound * tol_s + 1e-9).any() or (dv[:, 1] > 8 * bound * tol_q + 1e-9).any():
                problems.append(f"stats_out increments off the reference sums by {e_st:.1e} (bound {4 * bound:.1e})")
            if got is not None:
                stored = torch.zeros(nsl, 2, dtype=F64, device=self.dev)
                stored.index_add_(0, sl, torch.stack([got, got * got], 1))
                rt = 2.0 ** -8 if d.out_bf16 else 1e-6
                ds = (delta - stored).abs()
                if (ds[:, 0] > rt * (cnt * stored[:, 1]).sqrt() + 1e-9).any() or (ds[:, 1] > 2 * rt * stored[:, 1] + 1e-9).any():
                    problems.append(f"stats_out increments are not the sums of the stored values ({float(ds.max()):.2e})")
        return (e_rel, e_blk, e_st), problems

    # -- attention
    def attention(self, name, *args):
        bf = name == "bd_attention_bf16"
        q, k, v, o, B, H, Tq, Tk, ldq, ldk, ldv, ldo = args[:12]
        math_ = "bf16-tensor" if bf else args[12]
        D, dt = 64 * H, (BF16 if bf else F32)
        ext = [Ext("q", q, 0, (B * Tq - 1) * ldq + D - 1, dt), Ext("k", k, 0, (B * Tk - 1) * ldk + D - 1, dt),
               Ext("v", v, 0, (B * Tk - 1) * ldv + D - 1, dt), Ext("o", o, 0, (B * Tq - 1) * ldo + D - 1, dt)]
        if not bf:
            nws = _lib.call_value("bd_attention_workspace", B, H, Tq, Tk, math_)
            if nws:
                ext.append(Ext("ws", args[13], 0, nws - 1, F32))
        self.sync()
        self.check_inside(ext)
        read, _ = self.snapshot(ext[:3])
        rc = self.forward(name, *args)
        self.sync()

        def heads(p, T, ld, mem=None):
            t = read(p, (B * T - 1) * ld + D, dt) if mem is None else mem
            return t.as_strided((B, T, H, 64), (T * ld, ld, 64, 1)).to(F64).transpose(1, 2)
        Q, Kh, V = heads(q, Tq, ldq), heads(k, Tk, ldk), heads(v, Tk, ldv)
        Oraw = raw_bytes(o, ((B * Tq - 1) * ldo + D) * ES[dt], self.dev).view(dt)
        got = heads(o, Tq, ldo, Oraw)
        num = den = 0.0
        for b in range(B):
            want = torch.softmax(Q[b] @ Kh[b].transpose(-1, -2) / 8.0, dim=-1) @ V[b]
            num += float(((got[b] - want) ** 2).sum())
            den += float((want ** 2).sum())
        err = math.sqrt(num / max(den, 1e-60))
        bound = ATT_BOUND[math_]
        problems = [] if err <= bound else [f"rel-L2 {err:.2e} > {bound:.1e}"]
        mname = math_ if bf else MATH_NAME[math_]
        line = f"{self.tag} {self.site:<16} {name:<24} arm={mname} B={B} H={H} Tq={Tq} Tk={Tk} rel-L2 {err:.2e}"
        self.note([(self.tag, mname, "attention")], err, line, problems)
        return rc


def _host_bf16(real, name, args):
    """Host stand-ins for the bf16-tensor entry points the numpy emulator keeps in fp32: convert, run the fp32 entry
    point, round the output back.  Returns whether the call was handled."""
    if name == "bd_layer_norm" and args[8]:
        x, y, g, b, pos, period, M, Cc, _, st = args
        tmp = torch.empty(M * Cc)
        real(name, x, tmp.data_ptr(), g, b, pos, period, M, Cc, 0, st)
        host_read(y, M * Cc, BF16).copy_(tmp.to(BF16))
        return True
    if name == "bd_attention_bf16":
        q, k, v, o, B, H, Tq, Tk, ldq, ldk, ldv, ldo, st = args
        D = 64 * H
        qf, kf, vf = (host_read(p, (B * T - 1) * ld + D, BF16).float() for p, T, ld in ((q, Tq, ldq), (k, Tk, ldk), (v, Tk, ldv)))
        ob = host_read(o, (B * Tq - 1) * ldo + D, BF16)
        of = ob.float()
        real("bd_attention", qf.data_ptr(), kf.data_ptr(), vf.data_ptr(), of.data_ptr(), B, H, Tq, Tk, ldq, ldk, ldv, ldo,
             _lib.MATH_FP32, None, st)
        ob.copy_(of.to(BF16))
        return True
    if name == "bd_conv_gemm" and (args[0]._obj.x_bf16 or args[0]._obj.out_bf16):
        d = args[0]._obj
        by = {e.name: e for e in extents(d)}
        d2 = GemmDesc.from_buffer_copy(d)
        d2.x_bf16 = d2.out_bf16 = 0
        if d.x_bf16:
            e = by["x"]
            xf = host_read(e.ptr + 2 * e.lo, e.hi - e.lo + 1, BF16).float()
            d2.x = xf.data_ptr() - 4 * e.lo
        if d.out_bf16:
            e = by["out"]
            ob = host_read(e.ptr + 2 * e.lo, e.hi - e.lo + 1, BF16)
            of = ob.float()
            d2.out = of.data_ptr() - 4 * e.lo
        real(name, C.byref(d2), args[1])
        if d.out_bf16:
            ob.copy_(of.to(BF16))
        return True
    return False


@contextlib.contextmanager
def shadowed(monkeypatch, shadow):
    """Route the engines' launches through ``shadow``; name each call after the engine method that issued it."""
    orig_k = Engine._k

    def k(self, name, *args, **kw):
        f = sys._getframe(1)
        if f.f_code.co_name == "_gemm":
            f = f.f_back
        shadow.site, shadow.label = f.f_code.co_name, kw.get("label") or name
        return orig_k(self, name, *args, **kw)
    monkeypatch.setattr(Engine, "_k", k)
    monkeypatch.setattr(_lib, "call", shadow)
    yield shadow


# ---------------------------------------------------------------------------------------------------------------------
# synthetic descriptors
class Case:
    """One bd_conv_gemm launch with every tensor it needs.  The output region sits between two guard regions of a
    NaN-filled buffer; `resid` (in place) fills the region with data first."""
    GUARD = 64

    def __init__(self, dev, math_, *, B=2, I1=1, I0=300, Cin=32, N=64, taps=((0, 0),), m0=1, J0=None, act=_lib.ACT_NONE,
                 bias=True, e_stats=False, rowbias=0, resid=False, addend=False, convt=0, O0=None, oc_split=0,
                 stats=None, stat=None, store=True, a_mode=_lib.A_NONE, channel_major=False, x16=False, out16=False,
                 pitch=0, seed=0):
        g = torch.Generator().manual_seed(seed)

        def rnd(*shape, s=1.0):
            return (s * torch.randn(*shape, generator=g)).to(dev)
        J0 = (I0 * m0 if not convt else (I0 - 1 if convt == 1 else I0)) if J0 is None else J0
        J1 = I1
        K = len(taps) * Cin
        d = self.d = GemmDesc()
        d.M, d.N, d.K, d.Cin, d.taps = B * I1 * I0, N, K, Cin, len(taps)
        d.I1, d.I0, d.m1, d.m0, d.J1, d.J0 = I1, I0, 1, m0, J1, J0
        for i, (a, b) in enumerate(taps):
            d.d1[i], d.d0[i] = a, b
        if channel_major:
            self.x = rnd(B, Cin, J1 * J0)
            d.xs_b, d.xs_1, d.xs_0, d.xs_c = Cin * J1 * J0, J0, 1, J1 * J0
        else:
            self.x = rnd(B, J1, J0, Cin).to(BF16 if x16 else F32)
            d.xs_b, d.xs_1, d.xs_0, d.xs_c = J1 * J0 * Cin, J0 * Cin, Cin, 1
        self.w = rnd(N, K, s=K ** -0.5)
        self.bias = rnd(N) if bias else None
        if math_ in (_lib.MATH_BF16X3, _lib.MATH_BF16):
            self.w_hi = self.w.to(BF16)
            self.w_lo = (self.w - self.w_hi.float()).to(BF16)
            d.w16_hi, d.w16_lo = self.w_hi.data_ptr(), self.w_lo.data_ptr()
        no = N // 2 if act == _lib.ACT_GLU else (N // 4 if convt else N)
        O0 = (4 * J0 - 2 if convt == 1 else 4 * I0) if (convt and O0 is None) else (O0 or 0)
        P = O0 if convt else I0
        Pp = P + pitch
        if oc_split:
            d.os_b, d.os_1, d.os_0, d.oc_split, d.oc_stride = I1 * no * Pp, no * Pp, oc_split, oc_split, Pp * oc_split
        else:
            d.os_b, d.os_1, d.os_0 = I1 * Pp * no, Pp * no, no
        d.convt, d.O0 = convt, O0
        nreg = B * I1 * Pp * no
        odt = BF16 if out16 else F32
        self.buf = torch.full((nreg + 2 * self.GUARD,), float("nan"), dtype=odt, device=dev)
        self.region = self.buf[self.GUARD:self.GUARD + nreg]
        if resid:
            self.region.copy_(rnd(nreg))
            self.scale = rnd(no)
            d.resid, d.scale = self.region.data_ptr(), self.scale.data_ptr()
        if addend:
            self.addend = rnd(nreg)
            d.addend = self.addend.data_ptr()
        d.out = self.region.data_ptr() if store else None
        rows_per_item = I1 * I0
        d.stat_div, d.stat_mul, d.stat_mod = stat or (rows_per_item, 1, 1)
        nsl = int(slab_of(d, torch.arange(d.M)).max()) + 1
        if e_stats:
            self.e_stats = torch.stack([rnd(nsl, s=0.3), 0.5 + torch.rand(nsl, generator=g).to(dev)], 1).contiguous()
            self.e_gamma, self.e_beta = rnd(N), rnd(N)
            d.e_stats, d.e_gamma, d.e_beta = (t.data_ptr() for t in (self.e_stats, self.e_gamma, self.e_beta))
        if rowbias:
            self.rowbias = rnd(rowbias, no)
            d.rowbias, d.rowbias_period = self.rowbias.data_ptr(), rowbias
        if stats:
            self.stats = rnd(nsl, 2).double()            # the increments add to whatever is there
            d.stats_out = self.stats.data_ptr()
        if a_mode == _lib.A_ITEM_AFFINE:
            self.a_stats = torch.zeros(B, 8)
            self.a_stats[:, 0] = 0.1 * torch.randn(B, generator=g)
            self.a_stats[:, 2] = 1.0 + 0.2 * torch.rand(B, generator=g)
            self.a_stats = self.a_stats.to(dev)
            d.a_mode, d.a_stats, d.a_stats_stride = a_mode, self.a_stats.data_ptr(), 8
        elif a_mode == _lib.A_GN_GELU:
            self.a_stats = torch.stack([rnd(nsl, s=0.3), 0.5 + torch.rand(nsl, generator=g).to(dev)], 1).contiguous()
            self.a_gamma, self.a_beta = rnd(Cin), rnd(Cin)
            d.a_mode, d.a_stats = a_mode, self.a_stats.data_ptr()
            d.a_gamma, d.a_beta = self.a_gamma.data_ptr(), self.a_beta.data_ptr()
        d.act, d.x, d.w, d.bias = act, self.x.data_ptr(), self.w.data_ptr(), (self.bias.data_ptr() if bias else None)
        d.math, d.x_bf16, d.out_bf16 = math_, int(x16), int(out16)

    def arm(self):
        return _lib.lib().bd_conv_gemm_arm(C.byref(self.d))

    def run(self, shadow):
        """Launch through the shadow checker; check the guard regions and what is written."""
        before = self.buf.clone()
        shadow.gemm(C.byref(self.d), 0)
        it = INT_OF[self.buf.dtype]
        G = self.GUARD
        for sl in (slice(0, G), slice(self.buf.numel() - G, None)):
            assert torch.equal(self.buf[sl].view(it), before[sl].view(it)), "a guard region changed"
        return shadow.last


TAPS8 = tuple((0, k - 2) for k in range(8))
TAPS9 = tuple((kt - 1, kf - 1) for kf in range(3) for kt in range(3))
TAPS_CT1, TAPS_CT3 = ((0, 0), (0, -1)), ((0, -1), (0, 0), (0, 1))
WAVE = 148 * 128                      # one 128-row tile per SM: exact / wide tiles win the wave-efficiency test

# feature matrix: every case in every arithmetic unless `maths` says otherwise
FEATURES = {
    "convt1_gelu_addend_cout12": dict(convt=1, taps=TAPS_CT1, I0=301, N=48, act=_lib.ACT_GELU, addend=True, pitch=3),
    "convt1_gelu_addend_cout6": dict(convt=1, taps=TAPS_CT1, I0=301, N=24, act=_lib.ACT_GELU, addend=True, pitch=3),
    "convt2_split_i0_8_n64": dict(convt=2, taps=TAPS_CT3, B=2, I1=12, I0=8, N=64, Cin=48, oc_split=4),
    "convt2_split_i0_32_n96": dict(convt=2, taps=TAPS_CT3, B=2, I1=5, I0=32, N=96, Cin=48, oc_split=4),
    "glu_gn_resid_freq": dict(I0=2 * 20 * 32, B=1, N=96, Cin=48, act=_lib.ACT_GLU, e_stats=True, resid=True,
                              stat=(20 * 32, 32, 32)),
    "glu_rowbias": dict(I0=3 * 32, B=4, N=96, Cin=48, act=_lib.ACT_GLU, rowbias=32, stat=(96, 1, 1)),
    "glu_rowbias_scalar": dict(I0=3 * 32, B=4, N=90, Cin=48, act=_lib.ACT_GLU, rowbias=32),
    "addend_stats_item": dict(B=3, I0=300, Cin=48, N=64, addend=True, stats=True),
    "addend_stats_freq_scalar": dict(B=1, I0=2 * 20 * 16, Cin=48, N=62, addend=True, stats=True, stat=(20 * 16, 16, 16)),
    "stats_only_item": dict(B=3, I0=500, N=96, Cin=48, store=False, stats=True),
    "stats_only_freq": dict(B=1, I0=2 * 40 * 16, N=96, Cin=48, store=False, stats=True, stat=(40 * 16, 16, 16)),
    "k8s4_j0_mult4": dict(B=2, I1=6, I0=64, m0=4, taps=TAPS8, Cin=48, N=96, act=_lib.ACT_GELU),
    "k8s4_j0_ragged": dict(B=2, I1=1, I0=250, m0=4, J0=998, taps=TAPS8, Cin=48, N=96, act=_lib.ACT_GELU),
    "3x3_glu": dict(B=2, I1=8, I0=64, taps=TAPS9, Cin=48, N=192, act=_lib.ACT_GLU),
    "item_affine_channel_major": dict(B=3, I0=250, m0=4, taps=TAPS8, Cin=2, N=48, a_mode=_lib.A_ITEM_AFFINE,
                                      channel_major=True, act=_lib.ACT_GELU),
    "gn_gelu_prologue_freq": dict(B=2, I0=30 * 16, Cin=24, N=48, a_mode=_lib.A_GN_GELU, stat=(30 * 16, 16, 16),
                                  stats=True),
    "ragged_m_n": dict(B=1, I0=1000, Cin=48, N=50),
    "ragged_n10_k16": dict(B=1, I0=777, Cin=16, N=10, act=_lib.ACT_GELU),
    "stats_item_resid": dict(B=4, I0=333, Cin=64, N=128, resid=True, stats=True),
}
BF16_TENSOR = {
    "x16_out32_gelu_stats": dict(B=2, I0=600, Cin=64, N=128, act=_lib.ACT_GELU, x16=True, stats=True),
    "x16_out16_gelu_stats": dict(B=2, I0=600, Cin=128, N=192, act=_lib.ACT_GELU, x16=True, out16=True, stats=True),
}


def _sweep():
    """One plain descriptor per kernel template the dispatcher can instantiate, and per CUDA-core column band."""
    out = {}
    for math_, tbks, widths in ((_lib.MATH_TF32, (16, 32), (16, 32, 64, 128)), (_lib.MATH_TF32, (16,), (256,)),
                                (_lib.MATH_TF32X3, (16,), (16, 32, 64, 128, 256)),
                                (_lib.MATH_BF16, (16, 32), (16, 32, 64, 128, 256)),
                                (_lib.MATH_BF16X3, (16, 32), (16, 32, 64, 96, 128, 192, 256))):
        for tbk in tbks:
            for n in widths:
                # Cin % 32 == 16 -> 16-deep k-blocks (and TF32X3 / 256-wide TF32 always); K >= 256 for the wide tiles
                cin = (272 if tbk == 16 else 256) if n == 256 else (48 if tbk == 16 else 64)
                out[f"{MATH_NAME[math_]}_k{tbk}_n{n}"] = (math_, dict(B=1, I0=WAVE, Cin=cin, N=n, bias=n != 128,
                                                                      act=_lib.ACT_GELU if n == 64 else _lib.ACT_NONE))
    for n in (16, 32, 64, 128, 256):
        out[f"bf16tensor_k64_n{n}"] = (_lib.MATH_BF16, dict(B=1, I0=WAVE, Cin=64 if n < 256 else 256, N=n, x16=True,
                                                              out16=n == 64))
    for n in (100, 48, 24, 12):
        out[f"simt_n{n}"] = (_lib.MATH_FP32, dict(B=2, I0=400, Cin=40, N=n))
    return out


SWEEP = _sweep()
ALL_MATHS = (_lib.MATH_FP32, _lib.MATH_TF32, _lib.MATH_TF32X3, _lib.MATH_BF16X3, _lib.MATH_BF16)
MATRIX = [(name, m, spec) for name, spec in FEATURES.items() for m in ALL_MATHS] + \
         [(name, _lib.MATH_BF16, spec) for name, spec in BF16_TENSOR.items()] + \
         [(name, m, spec) for name, (m, spec) in SWEEP.items()]
# kernel templates: (math, 1000 * k-block + tile width), gemm_tc.cu / gemm_tc_b16*.cu / launch_tc_width
TEMPLATES = {(_lib.MATH_TF32, 1000 * k + n) for k in (16, 32) for n in (16, 32, 64, 128)} | {(_lib.MATH_TF32, 16256)} | \
            {(_lib.MATH_TF32X3, 16000 + n) for n in (16, 32, 64, 128, 256)} | \
            {(_lib.MATH_BF16, 1000 * k + n) for k in (16, 32) for n in (16, 32, 64, 128, 256)} | \
            {(_lib.MATH_BF16X3, 1000 * k + n) for k in (16, 32) for n in (16, 32, 64, 96, 128, 192, 256)} | \
            {(_lib.MATH_BF16, 64000 + n) for n in (16, 32, 64, 128, 256)}


def _simt_band(d):
    return 128 if d.N > 64 else 64 if d.N > 32 else 32 if (d.N > 16 or d.act == _lib.ACT_GLU) else 16


# =====================================================================================================================
# CPU: the statement against the emulator and against torch's convolutions; the shadow checker rehearsed on the engines
@pytest.mark.parametrize("name", list(FEATURES))
def test_reference_matches_emulator(name):
    """Each feature descriptor through the numpy ABI emulator (fp32) against the float64 statement, with the shadow
    checker's extent, aliasing, unchanged-element and statistics checks."""
    c = Case("cpu", _lib.MATH_FP32, **FEATURES[name])
    keep = [v for v in vars(c).values() if torch.is_tensor(v)]
    sh = Shadow("cpu", host_blocks(keep))
    with E.emulated_abi():
        res = c.run(sh)
    assert not sh.failures, sh.failures
    assert res["err"][0] < 1e-6


def _conv_case(x, w, bias, **geo):
    """Descriptor over host tensors, evaluated by ref_conv_gemm alone."""
    d = GemmDesc()
    for k, v in geo.items():
        if k == "taps":
            d.taps = len(v)
            for i, (a, b) in enumerate(v):
                d.d1[i], d.d0[i] = a, b
        else:
            setattr(d, k, v)
    d.x, d.w, d.bias = x.data_ptr(), w.data_ptr(), (bias.data_ptr() if bias is not None else None)
    d.K, d.out = d.taps * d.Cin, 1 << 40              # never dereferenced: the statement returns values and indices
    ref = ref_conv_gemm(d, host_read)
    return ref, d


def _dense(ref, n):
    out = torch.full((n,), float("nan"), dtype=F64)
    out[ref.idx] = ref.vals
    return out


@pytest.mark.parametrize("kind", ["conv1d", "conv1d_channel_major_affine", "conv2d", "conv2d_affine", "rewrite3x3_glu",
                                  "convtr1d_2tap", "convtr1d_3tap", "convtr2d_2tap", "convtr2d_3tap_oc_split"])
def test_reference_matches_torch_conv(kind):
    """The statement on the engine's own weight packings (conv_w, convtr_w, convtr_w3, GLU interleave) reproduces
    F.conv1d / conv2d / conv_transpose1d / conv_transpose2d (+ the [2:2+L] crop) in float64."""
    g = torch.Generator().manual_seed(11)
    B, Cin, Co = 2, 8, 12
    if kind.startswith("conv1d"):
        L = 64
        Lo = L // 4
        w = torch.randn(Co, Cin, 8, generator=g)
        b = torch.randn(Co, generator=g)
        x = torch.randn(B, Cin, L, generator=g)
        norm = torch.zeros(B, 8)
        norm[:, 0], norm[:, 2] = torch.randn(B, generator=g), 1 + torch.rand(B, generator=g)
        geo = dict(M=B * Lo, N=Co, Cin=Cin, taps=TAPS8, I1=1, I0=Lo, m1=1, m0=4, J1=1, J0=L, os_b=Lo * Co, os_1=0,
                   os_0=Co)
        if kind.endswith("affine"):       # the mix [B, C, L] read channel-major, normalised per item on the fly
            xin = x
            geo.update(xs_b=Cin * L, xs_1=0, xs_0=1, xs_c=L, a_mode=_lib.A_ITEM_AFFINE, a_stats=norm.data_ptr(),
                       a_stats_stride=8)
            want = F.conv1d((x.double() - norm[:, :1, None].double()) * norm[:, 2:3, None].double(), w.double(),
                            b.double(), stride=4, padding=2)
        else:
            xin = x.transpose(1, 2).contiguous()
            geo.update(xs_b=L * Cin, xs_1=0, xs_0=Cin, xs_c=1)
            want = F.conv1d(x.double(), w.double(), b.double(), stride=4, padding=2)
        wp = conv_w(w).contiguous()
        ref, d = _conv_case(xin, wp, b, **geo)
        got = _dense(ref, B * Lo * Co).view(B, Lo, Co).transpose(1, 2)
    elif kind.startswith("conv2d"):
        Fin, T = 64, 5
        Fo = Fin // 4
        w = torch.randn(Co, Cin, 8, 1, generator=g)
        b = torch.randn(Co, generator=g)
        x = torch.randn(B, Cin, Fin, T, generator=g)
        norm = torch.zeros(B, 8)
        norm[:, 0], norm[:, 2] = torch.randn(B, generator=g), 1 + torch.rand(B, generator=g)
        xin = x.permute(0, 3, 2, 1).contiguous()          # [B, T, F, C]
        geo = dict(M=B * T * Fo, N=Co, Cin=Cin, taps=TAPS8, I1=T, I0=Fo, m1=1, m0=4, J1=T, J0=Fin,
                   xs_b=T * Fin * Cin, xs_1=Fin * Cin, xs_0=Cin, xs_c=1, os_b=T * Fo * Co, os_1=Fo * Co, os_0=Co)
        xn = x.double()
        if kind.endswith("affine"):
            geo.update(a_mode=_lib.A_ITEM_AFFINE, a_stats=norm.data_ptr(), a_stats_stride=8)
            xn = (xn - norm[:, 0].double().view(B, 1, 1, 1)) * norm[:, 2].double().view(B, 1, 1, 1)
        want = F.conv2d(xn, w.double(), b.double(), stride=(4, 1), padding=(2, 0))
        ref, d = _conv_case(xin, conv_w(w).contiguous(), b, **geo)
        got = _dense(ref, B * T * Fo * Co).view(B, T, Fo, Co).permute(0, 3, 2, 1)
    elif kind == "rewrite3x3_glu":
        Fr, T, Cc = 16, 6, 8
        w = torch.randn(2 * Cc, Cc, 3, 3, generator=g)
        b = torch.randn(2 * Cc, generator=g)
        x = torch.randn(B, Cc, Fr, T, generator=g)
        xin = x.permute(0, 3, 2, 1).contiguous()
        ref, d = _conv_case(xin, _interleave_glu(conv_w(w)), _interleave_glu(b), M=B * T * Fr, N=2 * Cc, Cin=Cc,
                            taps=TAPS9, I1=T, I0=Fr, m1=1, m0=1, J1=T, J0=Fr, xs_b=T * Fr * Cc, xs_1=Fr * Cc, xs_0=Cc,
                            xs_c=1, os_b=T * Fr * Cc, os_1=Fr * Cc, os_0=Cc, act=_lib.ACT_GLU)
        want = F.glu(F.conv2d(x.double(), w.double(), b.double(), padding=1), dim=1)
        got = _dense(ref, B * T * Fr * Cc).view(B, T, Fr, Cc).permute(0, 3, 2, 1)
    elif kind.startswith("convtr1d"):
        Tin, Cc, Cout = 40, 8, 6
        Tout, pitch = 4 * Tin - 3, 5                        # a crop short of the full length, padded item pitch
        three = kind.endswith("3tap")
        w = torch.randn(Cc, Cout, 8, generator=g)
        b = torch.randn(Cout, generator=g)
        x = torch.randn(B, Cc, Tin, generator=g)
        xin = x.transpose(1, 2).contiguous()
        I0 = Tin if three else Tin + 1
        ref, d = _conv_case(xin, (convtr_w3(w) if three else convtr_w(w)).contiguous(), b.repeat(4), M=B * I0,
                            N=4 * Cout, Cin=Cc, taps=TAPS_CT3 if three else TAPS_CT1, I1=1, I0=I0, m1=1, m0=1, J1=1,
                            J0=Tin, xs_b=Tin * Cc, xs_1=0, xs_0=Cc, xs_c=1, os_b=(Tout + pitch) * Cout, os_1=0,
                            os_0=Cout, convt=2 if three else 1, O0=Tout)
        want = F.conv_transpose1d(x.double(), w.double(), b.double(), stride=4)[..., 2:2 + Tout]
        full = _dense(ref, B * (Tout + pitch) * Cout).view(B, Tout + pitch, Cout)
        assert torch.isnan(full[:, Tout:]).all()            # the pitch rows are not written
        got = full[:, :Tout].transpose(1, 2)
    else:                                                   # convtr2d
        Fr, T, Cc, S = 8, 5, 8, 3
        three = "3tap" in kind
        Cout = 4 * S if three else 6
        w = torch.randn(Cc, Cout, 8, 1, generator=g)
        b = torch.randn(Cout, generator=g)
        x = torch.randn(B, Cc, Fr, T, generator=g)
        xin = x.permute(0, 3, 2, 1).contiguous()
        I0 = Fr if three else Fr + 1
        geo = dict(M=B * T * I0, N=4 * Cout, Cin=Cc, taps=TAPS_CT3 if three else TAPS_CT1, I1=T, I0=I0, m1=1, m0=1,
                   J1=T, J0=Fr, xs_b=T * Fr * Cc, xs_1=Fr * Cc, xs_0=Cc, xs_c=1, convt=2 if three else 1, O0=4 * Fr)
        if three:     # the last frequency decoder: source-major planes [B, T, S, 4F, 4]
            geo.update(os_b=T * 4 * Fr * Cout, os_1=4 * Fr * Cout, os_0=4, oc_split=4, oc_stride=4 * Fr * 4)
        else:
            geo.update(os_b=T * 4 * Fr * Cout, os_1=4 * Fr * Cout, os_0=Cout)
        ref, d = _conv_case(xin, (convtr_w3(w) if three else convtr_w(w)).contiguous(), b.repeat(4), **geo)
        want = F.conv_transpose2d(x.double(), w.double(), b.double(), stride=(4, 1))[:, :, 2:2 + 4 * Fr]
        dense = _dense(ref, B * T * 4 * Fr * Cout)
        if three:
            got = dense.view(B, T, S, 4 * Fr, 4).permute(0, 2, 4, 3, 1).reshape(B, Cout, 4 * Fr, T)
        else:
            got = dense.view(B, T, 4 * Fr, Cout).permute(0, 3, 2, 1)
    assert got.shape == want.shape
    assert not torch.isnan(got).any()
    assert float((got - want).norm() / want.norm()) < 1e-12


def _engine_forward(cfg, W, mix, mode, monkeypatch, tag, hdemucs=False, device="cpu"):
    from demucs_b200.hdemucs_engine import HDemucsEngine
    eng = (HDemucsEngine if hdemucs else Engine)(cfg, W, device, mode=mode)
    blocks = cuda_blocks if device != "cpu" else host_blocks(eng, mix)
    sh = Shadow(device, blocks, tag=tag)
    with shadowed(monkeypatch, sh):
        eng.forward(mix)
    return sh


@pytest.mark.parametrize("mode", MODES)
def test_shadow_rehearsal_htdemucs(mode, monkeypatch):
    """The shadow checker on every descriptor Engine(small_config) builds in each mode, under the numpy ABI."""
    cfg = small_config()
    W = init_weights(cfg, 1, layer_scale=0.5)
    mix = synth_mix(1, cfg.segment_length, 7)
    with E.emulated_abi():
        sh = _engine_forward(cfg, W, mix, mode, monkeypatch, f"small/{mode}")
    assert not sh.failures, "\n".join(sh.failures)
    n = sum(" arm=" in r for r in sh.records)
    assert n > 40
    if mode != "fp32":        # the three-tap transposed convs of the tensor-core forms
        assert any("convt2" in r for r in sh.records)
    if mode == "bf16":
        assert any("x16" in r for r in sh.records) and any("bd_attention_bf16" in r for r in sh.records)


@pytest.mark.parametrize("mode", ["fp32", "strict"])
def test_shadow_rehearsal_hdemucs(mode, monkeypatch):
    """The same on HDemucsEngine(hdemucs_small_config): 2-tap transposed convs, stats-only passes, BLSTM / LocalState
    projections."""
    from demucs_b200 import hdemucs as HD
    from oracle.make_golden import hdemucs_small_config
    cfg = hdemucs_small_config()
    W = HD.init_weights(cfg, 2, 0.5)
    mix = synth_mix(1, int(golden("hdemucs_small.npz")["length"]), 8)
    with E.emulated_abi():
        sh = _engine_forward(cfg, W, mix, mode, monkeypatch, f"hdemucs_small/{mode}", hdemucs=True)
    assert not sh.failures, "\n".join(sh.failures)
    assert any("stats_only" in r for r in sh.records)


# =====================================================================================================================
# GPU
DEV = "cuda:0"


def _print_worst(sh):
    print(f"worst rel-L2 per (arithmetic, feature), {sh.tag}:")
    for (tag, m, f), e in sorted(sh.worst.items()):
        print(f"    {m:<12} {f:<16} {e:.2e}")


def _htdemucs_inputs(six=False):
    from demucs_b200.config import htdemucs_6s_config
    if six:
        cfg = htdemucs_6s_config()
        return cfg, init_weights(cfg, 3, layer_scale=0.5), synth_mix(1, cfg.segment_length, 13)
    cfg = htdemucs_config()
    W, mix = forward_fixture_inputs(golden("htdemucs_ls05.npz"), cfg)
    return cfg, W, mix[:1].contiguous()


FORWARDS = [("htdemucs", m) for m in MODES] + [("htdemucs_6s", "strict"), ("htdemucs_6s", "bf16"),
                                              ("hdemucs_mmi", "fp32"), ("hdemucs_mmi", "strict")]


@pytest.mark.gpu
@pytest.mark.parametrize("model,mode", FORWARDS)
def test_gpu_forward_every_call(model, mode, monkeypatch):
    """Every bd_conv_gemm and attention launch of one real forward, on its own inputs, against float64."""
    if model == "hdemucs_mmi":
        from demucs_b200 import hdemucs as HD
        cfg = HD.hdemucs_mmi_config()
        g = golden("hdemucs_mmi.npz")
        ls = float(g["layer_scale"])
        W = HD.init_weights(cfg, int(g["seed"]), None if ls < 0 else ls)
        mix = synth_mix(1, int(g["length"]), 4321 + int(g["seed"]))
    else:
        cfg, W, mix = _htdemucs_inputs(model == "htdemucs_6s")
    sh = _engine_forward(cfg, W, mix.to(DEV), mode, monkeypatch, f"{model}/{mode}", hdemucs=model == "hdemucs_mmi",
                         device=DEV)
    _print_worst(sh)
    assert len(sh.records) > 50
    if model == "htdemucs_6s" and mode == "strict":     # the last freq decoder: exact 96-wide tile, convt=2, oc_split
        assert any("arm=bf16x3:16096" in r and "convt2" in r and "oc_split" in r for r in sh.records) or \
            any("arm=bf16x3:32096" in r and "convt2" in r and "oc_split" in r for r in sh.records)
    assert not sh.failures, "\n".join(sh.failures)


@pytest.mark.gpu
@pytest.mark.parametrize("name,math_,spec", MATRIX, ids=[f"{n}-{MATH_NAME[m]}" for n, m, _ in MATRIX])
def test_gpu_feature_matrix(name, math_, spec):
    """One fused feature (or kernel template) per descriptor: written elements finite and within the arm's bound,
    everything else bitwise unchanged (guards included), stats_out increments correct."""
    c = Case(DEV, math_, **spec, seed=len(name))
    arm = c.arm()
    if math_ == _lib.MATH_FP32 or spec.get("a_mode") or name == "k8s4_j0_ragged" or c.d.N < 16:
        assert arm == 0                                  # the CUDA-core arm
    elif name == "k8s4_j0_mult4" or name in SWEEP:
        assert arm != 0
    sh = Shadow(DEV, cuda_blocks, tag=name)
    res = c.run(sh)
    assert not sh.failures, "\n".join(sh.failures)
    if name in SWEEP and math_ != _lib.MATH_FP32:
        want = SWEEP[name]
        assert arm % 1000 == want[1]["N"], (name, arm)


@pytest.mark.gpu
def test_gpu_template_coverage():
    """The matrix reaches every kernel template gemm_tc.cu / gemm_tc_b16*.cu / launch_tc_width can instantiate, and all
    four CUDA-core column bands.  If the dispatcher changes, TEMPLATES changes with it."""
    reached, bands = set(), set()
    for name, math_, spec in MATRIX:
        c = Case(DEV, math_, **spec)
        arm = c.arm()
        if arm:
            reached.add((math_, arm))
        else:
            bands.add(_simt_band(c.d))
    missing = sorted((MATH_NAME[m], a) for m, a in TEMPLATES - reached)
    assert not missing, missing
    assert bands == {16, 32, 64, 128}
