"""Host-side orchestration of the HTDemucs forward on the sm_100a kernel library.

This is the Python mirror of ``HTDemucs.forward`` (reference demucs/htdemucs.py:527-660) and
of the modules it calls -- HEncLayer / HDecLayer (hdemucs.py:123-157,304-335), DConv
(demucs.py:86-154) and CrossTransformerEncoder (transformer.py:648-676) -- expressed as a
sequence of C-ABI kernel launches (include/demucs_b200.h).  PyTorch is used for device
memory and streams only; every arithmetic step runs in a hand-written kernel and there is no
fallback: a missing library or a failing launch raises.

Activations are kept "position-innermost channels-last": time branch [B, T, C], frequency
branch [B, T, F, C] (DESIGN.md section 3).  In that layout the token order of the transformer
``(t1 fr)`` (transformer.py:653) is the memory order, the strided k=8 convolutions and the
transposed convolutions read / write contiguous windows, and STFT frames are contiguous.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import math
import typing as tp

import numpy as np
import torch

from . import _lib
from ._lib import GemmDesc, call, ptr
from .config import HTDemucsConfig
from .weights import check_state_dict

# Precision modes (DESIGN.md section 7).  "strict" is the default of the drop-in: fp32 activations in HBM, every
# contraction on the tensor cores with error-compensated operands (bf16 hi/lo split, three products: 16 mantissa
# bits per operand) -- per-stem rel-L2 <= 1e-4 against the fp32 reference.  "bf16" is the reduced-precision mode
# (single bf16 product, <= 1e-2).  "tf32x3" / "tf32" are the kind::tf32 forms of the same two ideas, "fp32" runs the
# contractions on CUDA cores.
MODES = ("fp32", "tf32", "tf32x3", "strict", "bf16")
# arithmetic of every contraction of a mode: the implicit GEMM, the attention core and the register-level (mma.sync)
# thin-layer kernels (single pass, or hi/lo split operands with three products); "fp32" runs them on CUDA cores
_MATH = {"fp32": _lib.MATH_FP32, "tf32": _lib.MATH_TF32, "tf32x3": _lib.MATH_TF32X3, "strict": _lib.MATH_BF16X3,
         "bf16": _lib.MATH_BF16}


def _interleave_glu(w: torch.Tensor) -> torch.Tensor:
    """Reorder rows [a_0..a_{C-1}, g_0..g_{C-1}] -> [a_0, g_0, a_1, g_1, ...] so that a GLU pair
    (F.glu(z, dim=1): a * sigmoid(g), hdemucs.py:154,313; demucs.py:141) sits in adjacent columns."""
    half = w.shape[0] // 2
    return torch.stack([w[:half], w[half:]], dim=1).reshape(w.shape).contiguous()


def _sin_embedding_1d(length: int, dim: int, max_period: float) -> torch.Tensor:
    """create_sin_embedding, shift=0 (transformer.py:19-34) -> [length, dim] = [cos | sin]."""
    pos = torch.arange(length, dtype=torch.float32)[:, None]
    half = dim // 2
    k = torch.arange(half, dtype=torch.float32)[None, :]
    phase = pos / (max_period ** (k / (half - 1)))
    return torch.cat([torch.cos(phase), torch.sin(phase)], dim=-1)


def _sin_embedding_2d(dim: int, height: int, width: int, max_period: float) -> torch.Tensor:
    """create_2d_sin_embedding (transformer.py:37-70) as a token table [(t1 fr), dim]."""
    half = dim // 2
    div = torch.exp(torch.arange(0.0, half, 2) * -(math.log(max_period) / half))
    pw = torch.arange(0.0, width)[:, None] * div[None, :]     # [W, half/2]
    ph = torch.arange(0.0, height)[:, None] * div[None, :]    # [H, half/2]
    pe = torch.zeros(width, height, dim)
    pe[:, :, 0:half:2] = torch.sin(pw)[:, None, :]
    pe[:, :, 1:half:2] = torch.cos(pw)[:, None, :]
    pe[:, :, half::2] = torch.sin(ph)[None, :, :]
    pe[:, :, half + 1::2] = torch.cos(ph)[None, :, :]
    return pe.reshape(width * height, dim)


def conv_w(w):
    """[Cout, Cin, k(,1)] / [Cout, Cin, kf, kt] -> [Cout, taps*Cin], tap-major."""
    w = w.detach().float()
    co, ci = w.shape[:2]
    return w.reshape(co, ci, -1).permute(0, 2, 1).reshape(co, -1)


def convtr_w(w):
    """[Cin, Cout, 8(,1)] -> [4*Cout, 2*Cin]; row r*Cout+co, col tap*Cin+ci = w[ci,co,r+4tap]."""
    w = w.detach().float()
    ci, co = w.shape[:2]
    w = w.reshape(ci, co, 2, 4)                 # k = 4*tap + r
    return w.permute(3, 1, 2, 0).reshape(4 * co, 2 * ci)


def convtr_w3(w):
    """3-tap form of the same transposed conv: output row p = 4 outputs 4p+s, s<4, read x[p-1], x[p], x[p+1]:
    u = 4p+s+2 = 4*ti + k  =>  tap -1: k=s+6 (s<=1), tap 0: k=s+2, tap +1: k=s-2 (s>=2); other entries zero.
    Rows = input positions exactly, so tensor-core tiles carry no halo row (DESIGN.md section 4)."""
    w = w.detach().float()
    ci, co = w.shape[:2]
    w = w.reshape(ci, co, 8)
    out = torch.zeros(4, co, 3, ci)
    for s_ in range(4):
        out[s_, :, 1] = w[:, :, s_ + 2].t()
        if s_ <= 1:
            out[s_, :, 0] = w[:, :, s_ + 6].t()
        else:
            out[s_, :, 2] = w[:, :, s_ - 2].t()
    return out.reshape(4 * co, 3 * ci)


def pack_dconv(put, packed, state, prefix: str, depth: int, tc_forms: bool, idx=(0, 1, 3, 4, 6)) -> None:
    """DConv parameters of ``prefix`` into kernel layouts; ``idx`` = positions of (conv3, norm1, conv1x1, norm2,
    LayerScale) inside the reference's nn.Sequential (they shift when BLSTM / LocalState are inserted, demucs.py:146-149)."""
    i_c3, i_n1, i_c1, i_n2, i_ls = idx
    for d in range(depth):
        p = f"{prefix}.dconv.layers.{d}"
        put(f"{p}.w1", conv_w(state[f"{p}.{i_c3}.weight"]))
        put(f"{p}.b1", state[f"{p}.{i_c3}.bias"])
        put(f"{p}.g1", state[f"{p}.{i_n1}.weight"])
        put(f"{p}.be1", state[f"{p}.{i_n1}.bias"])
        put(f"{p}.w2", _interleave_glu(conv_w(state[f"{p}.{i_c1}.weight"])))
        put(f"{p}.b2", _interleave_glu(state[f"{p}.{i_c1}.bias"].detach().float()))
        put(f"{p}.g2", _interleave_glu(state[f"{p}.{i_n2}.weight"].detach().float()))
        put(f"{p}.be2", _interleave_glu(state[f"{p}.{i_n2}.bias"].detach().float()))
        put(f"{p}.scale", state[f"{p}.{i_ls}.scale"])
        put(f"{p}.w2t", packed[f"{p}.w2"].cpu().t())      # [hid, 2C] for the dedicated expansion kernels
        if tc_forms:
            # tensor-core forms: hidden width padded to a multiple of 16 with zero rows / columns
            hid = state[f"{p}.{i_c3}.weight"].shape[0]
            hp = (hid + 15) // 16 * 16

            def pad_rows(t):
                t = t.detach().float()
                return torch.cat([t, t.new_zeros((hp - hid,) + tuple(t.shape[1:]))], 0)
            put(f"{p}.w1p", pad_rows(packed[f"{p}.w1"].cpu()))
            put(f"{p}.b1p", pad_rows(state[f"{p}.{i_c3}.bias"]))
            put(f"{p}.g1p", pad_rows(state[f"{p}.{i_n1}.weight"]))
            put(f"{p}.be1p", pad_rows(state[f"{p}.{i_n1}.bias"]))
            put(f"{p}.w2p", pad_rows(packed[f"{p}.w2"].cpu().t()).t())


def pack_encoder(put, state, p: str) -> None:
    """HEncLayer ``p`` (hdemucs.py:123-157): the strided conv tap-major, the k=1 rewrite with its GLU pairs interleaved."""
    put(f"{p}.conv.w", conv_w(state[f"{p}.conv.weight"]))
    put(f"{p}.conv.b", state[f"{p}.conv.bias"])
    put(f"{p}.rewrite.w", _interleave_glu(conv_w(state[f"{p}.rewrite.weight"])))
    put(f"{p}.rewrite.b", _interleave_glu(state[f"{p}.rewrite.bias"].detach().float()))


def pack_decoder(put, state, p: str, tc_forms: bool) -> None:
    """HDecLayer ``p`` (hdemucs.py:304-335): the rewrite with its GLU pairs interleaved, the k=8 / s=4 transposed conv in
    its 2-tap form (and the 3-tap tensor-core form), its bias repeated for the 4 output phases of a row."""
    put(f"{p}.rewrite.w", _interleave_glu(conv_w(state[f"{p}.rewrite.weight"])))
    put(f"{p}.rewrite.b", _interleave_glu(state[f"{p}.rewrite.bias"].detach().float()))
    put(f"{p}.conv_tr.w", convtr_w(state[f"{p}.conv_tr.weight"]))
    if tc_forms:
        put(f"{p}.conv_tr.w3", convtr_w3(state[f"{p}.conv_tr.weight"]))
    put(f"{p}.conv_tr.b", state[f"{p}.conv_tr.bias"].detach().float().repeat(4))


def _pitch(n: int) -> int:
    """Item pitch of a time-branch skip tensor: rows padded to a multiple of 4 (zero rows).  That is the reference's own
    right-padding (hdemucs.py:132-135) and lets the next layer's stride-4 window be a (pos/4, pos%4) TMA box."""
    return (n + 3) // 4 * 4


def _tap(taps, name: str, t: torch.Tensor, fmt: str) -> None:
    """Record an intermediate in the reference's layout: [B,T,F,C] -> [B,C,F,T] ("f"), [B,T,C] -> [B,C,T] ("t")."""
    if taps is not None:
        taps[name] = (t.permute(0, 3, 2, 1) if fmt == "f" else t.permute(0, 2, 1)).clone()


def _conv3_geometry(T: int, Fr: int, C_: int, hp: int, dil: int) -> dict:
    """Implicit-GEMM geometry of the DConv's dilated k=3 conv over T, x [B, T, Fr, C] -> h [B, T, Fr, hp]: positions are
    the fast axis on the time branch (Fr = 1); on the frequency branch the conv runs along T, the slow axis."""
    if Fr == 1:
        return dict(taps=((0, -dil), (0, 0), (0, dil)), I1=1, I0=T, J1=1, J0=T, xs=(T * C_, 0, C_, 1), os_=(T * hp, 0, hp))
    return dict(taps=((-dil, 0), (0, 0), (dil, 0)), I1=T, I0=Fr, J1=T, J0=Fr,
                xs=(T * Fr * C_, Fr * C_, C_, 1), os_=(T * Fr * hp, Fr * hp, hp))


class PackedWeights:
    """Reference state_dict -> kernel layouts (one-time, on the device)."""

    def __init__(self, cfg: HTDemucsConfig, state: tp.Mapping[str, torch.Tensor], device, tc_forms: bool = False):
        check_state_dict(cfg, state)
        self.t: tp.Dict[str, torch.Tensor] = {}
        dev = device

        def put(name, tensor):
            self.t[name] = tensor.detach().to(device=dev, dtype=torch.float32).contiguous()

        for i in range(cfg.depth):
            for name in ("encoder", "tencoder"):
                pack_encoder(put, state, f"{name}.{i}")
                if cfg.dconv_mode & 1:
                    pack_dconv(put, self.t, state, f"{name}.{i}", cfg.dconv_depth, tc_forms)
            for name in ("decoder", "tdecoder"):
                pack_decoder(put, state, f"{name}.{i}", tc_forms)
                if cfg.dconv_mode & 2:
                    pack_dconv(put, self.t, state, f"{name}.{i}", cfg.dconv_depth, tc_forms)
        if cfg.freq_emb:
            # x + freq_emb_scale * (emb_scale * E[fr, c])  (htdemucs.py:577-582, hdemucs.py:60-66)
            put("freq_emb", cfg.freq_emb * cfg.emb_scale * state["freq_emb.embedding.weight"].detach().float())
        if cfg.bottom_channels:
            for n in ("channel_upsampler", "channel_downsampler", "channel_upsampler_t", "channel_downsampler_t"):
                put(f"{n}.w", state[f"{n}.weight"].detach().float().squeeze(-1))
                put(f"{n}.b", state[f"{n}.bias"])
        if cfg.t_layers > 0:
            for k, v in state.items():
                if k.startswith("crosstransformer."):
                    put(k, v)

    def __getitem__(self, k: str) -> torch.Tensor:
        return self.t[k]

    def nbytes(self) -> int:
        return sum(v.numel() * 4 for v in self.t.values())


class Engine:
    """One HTDemucs model resident on one GPU."""

    Weights = PackedWeights      # state_dict -> kernel layouts; HDemucsEngine packs the v3 state_dict instead

    def __init__(self, cfg: HTDemucsConfig, state: tp.Mapping[str, torch.Tensor], device="cuda", mode: str = "fp32"):
        cfg.validate()
        if mode not in MODES:
            raise ValueError(f"mode must be one of {MODES}")
        self.cfg = cfg
        self.mode = mode
        self.device = torch.device(device)
        if self.device.type != "cuda" and _lib.TEST_HOOK is None:
            raise _lib.KernelError("demucs_b200 runs on CUDA devices only (there is no CPU path)")
        _lib.lib()  # fail loudly now if the extension is missing
        self.W = self.Weights(cfg, state, self.device, tc_forms=(mode != "fp32"))
        # periodic Hann window and twiddles: computed in float64 and rounded once (torch.hann_window in float32 was
        # seen to come back ~3e-5 off on some runs of the same host, which is visible at the 1e-5 STFT tolerance)
        k = np.arange(cfg.nfft, dtype=np.float64)
        self.window = torch.from_numpy((0.5 - 0.5 * np.cos(2 * np.pi * k / cfg.nfft)).astype(np.float32)).to(self.device)
        tw = np.stack([np.cos(2 * np.pi * k / cfg.nfft), -np.sin(2 * np.pi * k / cfg.nfft)], axis=1)
        self.twiddle = torch.from_numpy(tw.astype(np.float32)).to(self.device).contiguous()
        self.single_pass = mode in ("tf32", "bf16")      # reduced-precision modes: single-pass mma.sync thin-layer kernels
        self.math = _MATH[mode]
        self._w16_cache: tp.Dict[tp.Tuple, tp.Tuple[torch.Tensor, torch.Tensor]] = {}
        self._bufs: tp.Dict[tp.Tuple, tp.Dict[str, torch.Tensor]] = {}
        self._pos: tp.Dict[tp.Tuple, torch.Tensor] = {}
        self.launches = 0
        self._prof: tp.Optional[list] = None

    # ------------------------------------------------------------------ plumbing
    def _stream(self) -> int:
        if self.device.type != "cuda":
            return 0
        return torch.cuda.current_stream(self.device).cuda_stream

    MAX_BUFFER_SETS = 6      # activation sets kept alive (one per (batch, length) met); older ones are released

    def _buf(self, key, name: str, numel: int, dtype=torch.float32, zero=False) -> torch.Tensor:
        pool = self._bufs.pop(key, None)
        if pool is None:
            # a new geometry (v3 models run every trailing chunk at its own length): drop the least recently used sets
            # so that a long session does not pin one multi-GB set per distinct length (the caching allocator hands the
            # memory on in stream order, so queued kernels still see their data)
            while len(self._bufs) >= self.MAX_BUFFER_SETS:
                self._bufs.pop(next(iter(self._bufs)))
            pool = {}
        self._bufs[key] = pool       # most recently used last
        t = pool.get(name)
        if t is None or t.numel() < numel or t.dtype != dtype:
            t = (torch.zeros if zero else torch.empty)(int(numel), dtype=dtype, device=self.device)
            pool[name] = t
        return t[:numel]

    def _k(self, name: str, *args, flops: float = 0.0, nbytes: float = 0.0, label: tp.Optional[str] = None,
           detail: str = "", kernels: int = 1) -> None:
        """Launch one kernel through the C ABI.  ``flops`` / ``nbytes`` are the ALGORITHMIC work of the
        launch (DESIGN.md section 5), recorded with CUDA events when a profile is being taken."""
        self.launches += kernels          # kernel launches behind this entry point (bench.py's gpu_launches)
        if self._prof is None:
            self._call(name, *args)
            return
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        self._call(name, *args)
        e1.record()
        self._prof.append((label or name, e0, e1, flops, nbytes, detail))

    def _call(self, name: str, *args) -> None:
        try:
            # an engine built on a non-CUDA device under the test emulator must not hand host pointers to the CUDA
            # library once the emulator is gone: on a machine with a GPU the kernels would fault on them
            if self.device.type != "cuda" and _lib.TEST_HOOK is None:
                raise _lib.KernelError("demucs_b200 runs on CUDA devices only (there is no CPU path)")
            _lib.call(name, *args)
        except Exception:
            # some workspaces are self-clearing (statistics accumulators, Gram matrices): a forward that dies half-way
            # would leave them dirty, so drop every cached buffer before the error propagates
            self._bufs.clear()
            raise

    def _w16(self, w: torch.Tensor) -> tp.Tuple[torch.Tensor, torch.Tensor]:
        """bf16 hi / lo planes of a packed weight matrix (or of a row slice of one): hi = bf16(w), lo = bf16(w - hi).
        Made once per weight, on the device; the tcgen05 bf16 arms read them by TMA."""
        key = (w.data_ptr(), tuple(w.shape))
        got = self._w16_cache.get(key)
        if got is None:
            w = w.contiguous()
            hi = w.to(torch.bfloat16)
            lo = (w - hi.float()).to(torch.bfloat16)
            got = (hi.contiguous(), lo.contiguous(), w)       # keep `w` alive: the key is its address
            self._w16_cache[key] = got
        return got[0], got[1]

    def _gemm(self, *, M, N, Cin, x, w, out, taps=((0, 0),), I1=1, I0=None, m1=1, m0=1, J1=1, J0=None,
              xs=(0, 0, None, 1), os_=(0, 0, None), bias=None, a_mode=_lib.A_NONE, a_stats=None,
              a_stats_stride=0, a_gamma=None, a_beta=None, act=_lib.ACT_NONE, rowbias=None, rowbias_period=0,
              resid=None, scale=None, addend=None, convt=0, O0=0, stats_out=None, stat=(0, 0, 0),
              e_stats=None, e_gamma=None, e_beta=None, oc_split=0, oc_stride=0, tc=True, xf=False, x16=False,
              out16=False) -> None:
        d = GemmDesc()
        I0 = M if I0 is None else I0
        d.M, d.N, d.K, d.Cin, d.taps = M, N, len(taps) * Cin, Cin, len(taps)
        d.I1, d.I0, d.m1, d.m0, d.J1, d.J0 = I1, I0, m1, m0, J1, (I0 if J0 is None else J0)
        for i, (a, b) in enumerate(taps):
            d.d1[i], d.d0[i] = a, b
        n_out = N // 2 if act == _lib.ACT_GLU else (N // 4 if convt else N)
        d.xs_b, d.xs_1, d.xs_0, d.xs_c = xs[0], xs[1], (Cin if xs[2] is None else xs[2]), xs[3]
        d.os_b, d.os_1, d.os_0 = os_[0], os_[1], (n_out if os_[2] is None else os_[2])
        d.x, d.w, d.bias = ptr(x), ptr(w), ptr(bias)
        d.a_mode, d.a_stats, d.a_stats_stride = a_mode, ptr(a_stats), a_stats_stride
        d.a_gamma, d.a_beta = ptr(a_gamma), ptr(a_beta)
        d.e_stats, d.e_gamma, d.e_beta = ptr(e_stats), ptr(e_gamma), ptr(e_beta)
        d.act, d.rowbias, d.rowbias_period = act, ptr(rowbias), rowbias_period
        d.resid, d.scale, d.addend = ptr(resid), ptr(scale), ptr(addend)
        d.out, d.convt, d.O0 = ptr(out), convt, O0
        d.oc_split, d.oc_stride = oc_split, oc_stride
        d.stats_out = ptr(stats_out)
        d.stat_div, d.stat_mul, d.stat_mod = stat
        # "bf16" mode: bf16 operands inside the transformer (two thirds of the flops, all of it in LayerScale'd residual
        # branches), single-pass tf32 for the convolutions of the U-Net, whose activations are the main signal path
        d.math = _lib.MATH_FP32 if not tc else (_lib.MATH_TF32 if (self.mode == "bf16" and not xf) else self.math)
        if d.math in (_lib.MATH_BF16X3, _lib.MATH_BF16) and Cin % 16 == 0 and _lib.TEST_HOOK is None:
            hi, lo = self._w16(w)
            d.w16_hi, d.w16_lo = ptr(hi), ptr(lo)
        d.x_bf16, d.out_bf16 = int(x16), int(out16)
        K = len(taps) * Cin
        rows_in = (M // (I1 * I0)) * d.J1 * d.J0          # input positions (each read once, algorithmically)
        nbytes = (2.0 if x16 else 4.0) * rows_in * Cin + (2.0 if d.w16_hi else 4.0) * N * K + \
            (2.0 if out16 else 4.0) * (M * (N if convt else n_out) if out is not None else 0)
        nbytes += 4.0 * M * n_out * ((resid is not None) + (addend is not None))
        arm = "simt"
        tile = 128 if N > 64 else 64 if N > 32 else 32 if (N > 16 or act == _lib.ACT_GLU) else 16
        if d.math != _lib.MATH_FP32 and _lib.TEST_HOOK is None:
            code = _lib.lib().bd_conv_gemm_arm(C.byref(d))         # 0: CUDA-core arm, else 1000*TBK + TBN
            if code:
                arm, tile = "tc", f"{code // 1000},{code % 1000}"
        self._k("bd_conv_gemm", C.byref(d), self._stream(), flops=2.0 * M * N * K, nbytes=nbytes,
                label=f"conv_gemm_{arm}<{tile}>",
                detail=f"M={M} N={N} K={K} taps={len(taps)} act={act} a={a_mode} stats={int(stats_out is not None)}")

    # ------------------------------------------------------------------ blocks
    def _dconv(self, key, prefix: str, x: torch.Tensor, B: int, T: int, Fr: int, C_: int, tag: str):
        """DConv residual branch in place on x (demucs.py:86-154); x is [B, T, Fr, C] (Fr = 1 for the
        time branch).  One GroupNorm(1) item = one (b, fr) row of the reference's [B*Fr, C, T] view
        (hdemucs.py:146-151); rows are walked in memory order, the slab map picks the item."""
        cfg, W = self.cfg, self.W
        hid = int(C_ / cfg.dconv_comp)
        M = B * T * Fr
        slabs = B * Fr
        stat = (T * Fr, Fr, Fr)                      # slab(m) = b*Fr + fr
        tc = self.mode != "fp32"
        narrow = tc and hid == 6 and C_ == 48     # dedicated mma.sync conv3, h stored 8 wide
        hp = 8 if narrow else ((hid + 15) // 16 * 16 if tc else hid)   # tensor-core arm: h is 16-column padded
        h = self._buf(key, f"dconv_h{tag}", M * hp)
        sums = self._buf(key, f"dconv_sums{tag}", 2 * slabs, torch.float64, zero=True)   # finalize clears it again
        mr1 = self._buf(key, f"dconv_mr1{tag}", 2 * slabs)
        mr2 = self._buf(key, f"dconv_mr2{tag}", 2 * slabs)
        sfx = "p" if tc else ""
        for dd in range(cfg.dconv_depth):
            p = f"{prefix}.dconv.layers.{dd}"
            dil = 2 ** dd
            # (1) h = conv3_dilated(x) and the GroupNorm statistics of h
            if narrow:
                self._k("bd_dconv_conv3", ptr(x), ptr(W[f"{p}.w1"]), ptr(W[f"{p}.b1"]), ptr(h), hp, ptr(sums), M, C_, hid,
                        T * Fr, Fr, dil, self.math, self._stream(), flops=2.0 * M * hid * 3 * C_, nbytes=4.0 * M * (C_ + hid),
                        label="dconv_conv3_mma", detail=f"M={M} C={C_} hid={hid} dil={dil}")
            else:
                self._gemm(M=M, N=hp, Cin=C_, x=x, w=W[f"{p}.w1{sfx}"], bias=W[f"{p}.b1{sfx}"], out=h,
                           stats_out=sums, stat=stat, tc=tc, **_conv3_geometry(T, Fr, C_, hp, dil))
            self._k("bd_finalize_group_stats", ptr(sums), ptr(mr1), slabs, float(T * hid), self._stream())
            # (2) statistics of u = conv1x1(gelu(gn(h))) WITHOUT storing u: the expanded [.., 2C] tensor never
            #     touches HBM, both passes recompute it from the 8x narrower h (csrc/dconv.cu)
            gram = self._buf(key, f"dconv_gram{tag}.{hid}", (slabs + 1) * (hid * hid + hid) + hid + 2, dtype=torch.float64,
                             zero=True)     # zero once: the kernels hand it back cleared
            self._k("bd_dconv_expand_stats", ptr(h), hp, hid, ptr(mr1), ptr(W[f"{p}.g1"]), ptr(W[f"{p}.be1"]),
                    ptr(W[f"{p}.w2t"]), ptr(W[f"{p}.b2"]), ptr(sums), ptr(gram), M, C_, T * Fr, Fr, self._stream(),
                    nbytes=4.0 * M * hid, flops=4.0 * M * hid * C_, label="dconv_expand_stats",
                    detail=f"M={M} C={C_} hid={hid}", kernels=2)
            self._k("bd_finalize_group_stats", ptr(sums), ptr(mr2), slabs, float(T * 2 * C_), self._stream())
            # (3) x += scale * GLU(gn(u)), in place: the dedicated kernels of csrc/dconv.cu (mma.sync fragments in
            #     "tf32" mode, exact FFMA otherwise).  The widest layers (hid 48; in "tf32x3" also hid 24) are a real
            #     GEMM and go through the tcgen05 kernel instead: activate h once, then GroupNorm / GLU /
            #     LayerScale / residual in the GEMM epilogue.
            if tc and hid >= (48 if self.single_pass else 24):
                self._k("bd_gn_gelu_apply", ptr(h), ptr(mr1), ptr(W[f"{p}.g1p"]), ptr(W[f"{p}.be1p"]), M, hp, T * Fr, Fr,
                        self._stream(), nbytes=8.0 * M * hp, label="bd_gn_gelu_apply")
                self._gemm(M=M, N=2 * C_, Cin=hp, x=h, w=W[f"{p}.w2p"], bias=W[f"{p}.b2"], e_stats=mr2,
                           e_gamma=W[f"{p}.g2"], e_beta=W[f"{p}.be2"], act=_lib.ACT_GLU, resid=x, scale=W[f"{p}.scale"],
                           out=x, stat=stat)
                continue
            self._k("bd_dconv_expand_update", ptr(h), hp, hid, ptr(mr1), ptr(W[f"{p}.g1"]), ptr(W[f"{p}.be1"]),
                    ptr(W[f"{p}.w2t"]), ptr(W[f"{p}.b2"]), ptr(mr2), ptr(W[f"{p}.g2"]), ptr(W[f"{p}.be2"]),
                    ptr(W[f"{p}.scale"]), ptr(x), M, C_, T * Fr, Fr,
                    self.math, self._stream(),
                    nbytes=4.0 * M * (hid + 2 * C_), flops=4.0 * M * hid * C_, label="dconv_expand_update",
                    detail=f"M={M} C={C_} hid={hid}")

    def _attention_block(self, key, x, kv_src, p: str, attn: str, B: int, Tq: int, Tk: int, tag: str):
        """x += gamma_1 * MHA(q=x_normed, k=v=kv_normed); both inputs are already layer-normed."""
        W, D, H = self.W, self.cfg.transformer_dim, self.cfg.t_heads
        Win, bin_ = W[f"{p}.{attn}.in_proj_weight"], W[f"{p}.{attn}.in_proj_bias"]
        if self.mode == "bf16":
            return self._attention_block_bf16(key, x, kv_src, Win, bin_, B, Tq, Tk, tag)
        att = self._buf(key, f"att{tag}", B * Tq * D)
        nws = _lib.call_value("bd_attention_workspace", B, H, Tq, Tk, self.math)
        ws = self._buf(key, f"att_ws{tag}", nws) if nws else None
        label = "attention_simt" if self.mode == "fp32" else "attention_tc"
        # kernels behind the entry point: + V transpose (+ Q / K splits) / the three bf16 conversions
        nk = {_lib.MATH_FP32: 1, _lib.MATH_TF32: 2, _lib.MATH_TF32X3: 4, _lib.MATH_BF16X3: 4, _lib.MATH_BF16: 4}[self.math]
        if kv_src is None:  # self attention: one packed projection
            qkv = self._buf(key, f"qkv{tag}", B * Tq * 3 * D)
            self._gemm(M=B * Tq, N=3 * D, Cin=D, x=x, w=Win, bias=bin_, out=qkv, xf=True)
            self._k("bd_attention", ptr(qkv), qkv.data_ptr() + 4 * D, qkv.data_ptr() + 8 * D, ptr(att),
                    B, H, Tq, Tq, 3 * D, 3 * D, 3 * D, D, self.math, ptr(ws), self._stream(),
                    flops=4.0 * B * Tq * Tq * D, nbytes=4.0 * B * Tq * D * 4, label=label, kernels=nk)
        else:
            q = self._buf(key, f"q{tag}", B * Tq * D)
            kv = self._buf(key, f"kv{tag}", B * Tk * 2 * D)
            self._gemm(M=B * Tq, N=D, Cin=D, x=x, w=Win[:D], bias=bin_[:D], out=q, xf=True)
            self._gemm(M=B * Tk, N=2 * D, Cin=D, x=kv_src, w=Win[D:], bias=bin_[D:], out=kv, xf=True)
            self._k("bd_attention", ptr(q), ptr(kv), kv.data_ptr() + 4 * D, ptr(att),
                    B, H, Tq, Tk, D, 2 * D, 2 * D, D, self.math, ptr(ws), self._stream(),
                    flops=4.0 * B * Tq * Tk * D, nbytes=4.0 * B * (2 * Tq + 2 * Tk) * D, label=label, kernels=nk)
        return att

    def _attention_block_bf16(self, key, x, kv_src, Win, bin_, B: int, Tq: int, Tk: int, tag: str):
        """The "bf16" mode's form of the block: the layer-normed inputs, the projections and the attention output
        are bf16 tensors that only ever travel from one tensor-core kernel to the next (TMA reads them in operand form,
        no conversion passes); the residual stream they are added to stays fp32."""
        D, H = self.cfg.transformer_dim, self.cfg.t_heads
        bf = torch.bfloat16
        att = self._buf(key, f"att16{tag}", B * Tq * D, bf)
        if kv_src is None:
            qkv = self._buf(key, f"qkv16{tag}", B * Tq * 3 * D, bf)
            self._gemm(M=B * Tq, N=3 * D, Cin=D, x=x, w=Win, bias=bin_, out=qkv, xf=True, x16=True, out16=True)
            self._k("bd_attention_bf16", ptr(qkv), qkv.data_ptr() + 2 * D, qkv.data_ptr() + 4 * D, ptr(att),
                    B, H, Tq, Tq, 3 * D, 3 * D, 3 * D, D, self._stream(),
                    flops=4.0 * B * Tq * Tq * D, nbytes=2.0 * B * Tq * D * 4, label="attention_tc")
        else:
            q = self._buf(key, f"q16{tag}", B * Tq * D, bf)
            kv = self._buf(key, f"kv16{tag}", B * Tk * 2 * D, bf)
            self._gemm(M=B * Tq, N=D, Cin=D, x=x, w=Win[:D], bias=bin_[:D], out=q, xf=True, x16=True, out16=True)
            self._gemm(M=B * Tk, N=2 * D, Cin=D, x=kv_src, w=Win[D:], bias=bin_[D:], out=kv, xf=True, x16=True, out16=True)
            self._k("bd_attention_bf16", ptr(q), ptr(kv), kv.data_ptr() + 2 * D, ptr(att),
                    B, H, Tq, Tk, D, 2 * D, 2 * D, D, self._stream(),
                    flops=4.0 * B * Tq * Tk * D, nbytes=2.0 * B * (2 * Tq + 2 * Tk) * D, label="attention_tc")
        return att

    def _ln(self, x, y, p: str, M: int, pos=None, period=0):
        D = self.cfg.transformer_dim
        y16 = y.dtype == torch.bfloat16
        self._k("bd_layer_norm", ptr(x), ptr(y), ptr(self.W[f"{p}.weight"]), ptr(self.W[f"{p}.bias"]),
                ptr(pos), period, M, D, int(y16), self._stream(), nbytes=(6.0 if y16 else 8.0) * M * D)

    def _transformer_layer(self, key, x, other_normed, p: str, cross: bool, B: int, T: int, Tk: int, tag: str):
        """One MyTransformerEncoderLayer / CrossTransformerEncoderLayer, norm_first, in place on x
        (transformer.py:363-372, 495-500)."""
        W, D, Hd = self.W, self.cfg.transformer_dim, self.cfg.ffn_dim
        M = B * T
        b16 = self.mode == "bf16"      # GEMM-to-GEMM tensors (layer-norm outputs, FFN hidden) are stored as bf16
        adt = torch.bfloat16 if b16 else torch.float32
        ln = self._buf(key, f"ln{tag}", M * D, adt)
        self._ln(x, ln, f"{p}.norm1", M)
        att = self._attention_block(key, ln, other_normed if cross else None, p,
                                    "cross_attn" if cross else "self_attn", B, T, Tk, tag)
        a = "cross_attn" if cross else "self_attn"
        self._gemm(M=M, N=D, Cin=D, x=att, w=W[f"{p}.{a}.out_proj.weight"], bias=W[f"{p}.{a}.out_proj.bias"],
                   out=x, resid=x, scale=W[f"{p}.gamma_1.scale"], xf=True, x16=b16)
        self._ln(x, ln, f"{p}.norm3" if cross else f"{p}.norm2", M)
        hbuf = self._buf(key, f"ffn{tag}", M * Hd, adt)
        self._gemm(M=M, N=Hd, Cin=D, x=ln, w=W[f"{p}.linear1.weight"], bias=W[f"{p}.linear1.bias"], out=hbuf,
                   act=_lib.ACT_GELU, xf=True, x16=b16, out16=b16)
        sums = self._buf(key, f"no_sums{tag}", 2 * B, torch.float64, zero=True)   # finalize clears it again
        mr = self._buf(key, f"no_mr{tag}", 2 * B)
        self._gemm(M=M, N=D, Cin=Hd, x=hbuf, w=W[f"{p}.linear2.weight"], bias=W[f"{p}.linear2.bias"], out=x,
                   resid=x, scale=W[f"{p}.gamma_2.scale"], I1=1, I0=T, J0=T, xs=(T * Hd, 0, Hd, 1),
                   os_=(T * D, 0, D), stats_out=sums, stat=(T, 1, 1), xf=True, x16=b16)
        self._k("bd_finalize_group_stats", ptr(sums), ptr(mr), B, float(T * D), self._stream())
        self._k("bd_group_norm_apply", ptr(x), ptr(mr), ptr(W[f"{p}.norm_out.weight"]),
                ptr(W[f"{p}.norm_out.bias"]), B, T, D, self._stream(), nbytes=8.0 * B * T * D)

    # ------------------------------------------------------------------ layer steps (shared with HDemucsEngine)
    def _stft(self, key, mix, taps, mag=None):
        """K1: STFT + CaC pack of mix [B, A, L] and the normalisation statistics -> (spec [B, T, 2048, 2A], norm).
        forward_core gives the spectrogram ``mag``: only its statistics (and the mix's) are computed then."""
        B, A, L = mix.shape
        T = self.cfg.frames(L)
        st = self._stream()
        spec = self._buf(key, "spec", B * T * 2048 * 4)
        stats = self._buf(key, "item_stats", 4 * B, torch.float64)
        norm = self._buf(key, "item_norm", 8 * B)
        stats.zero_()
        if mag is None:
            self._k("bd_stft_cac", ptr(mix), ptr(self.window), ptr(self.twiddle), ptr(spec), ptr(stats), B, A, L, st,
                    nbytes=4.0 * B * (A * L + T * 2048 * 4), flops=2.5 * 4096 * 12 * 2 * B * T)
        else:
            spec.view(B, T, 2048, 2 * A).copy_(mag.permute(0, 3, 2, 1))
            pair = self._buf(key, "core_stats", 4 * B, torch.float64)
            pair.zero_()
            self._k("bd_item_stats", ptr(spec), ptr(pair), B, 2 * A * 2048 * T, st, nbytes=4.0 * spec.numel())
            self._k("bd_item_stats", ptr(mix), pair.data_ptr() + 16 * B, B, A * L, st, nbytes=4.0 * mix.numel())
            stats.view(B, 4)[:, :2].copy_(pair[:2 * B].view(B, 2))
            stats.view(B, 4)[:, 2:].copy_(pair[2 * B:].view(B, 2))
        self._k("bd_finalize_item_norm", ptr(stats), ptr(norm), B, float(4 * 2048 * T), float(A * L), st)
        _tap(taps, "stft", spec.view(B, T, 2048, 4), "f")
        return spec, norm

    def _time_encoder(self, key, i, x, y_name, norm, taps, B, Tin, Tout, Cin, Cc, conv_only=False) -> torch.Tensor:
        """Time-branch HEncLayer i (hdemucs.py:123-157): Conv1d(k=8, s=4, p=2) + GELU of x (for i = 0 the mix, normalised
        on the fly) into buffer ``y_name``, DConv, k=1 rewrite + GLU into the returned skip tensor ``saved_t{i}``.
        ``conv_only`` (v3's empty time layer, hdemucs.py:137-143): the conv without activation alone; returns y."""
        W, p = self.W, f"tencoder.{i}"
        first = i == 0
        Tin_p = Tin if first else _pitch(Tin)
        y = self._buf(key, y_name, B * Tout * Cc)
        if first and self.mode != "fp32" and Cc == 48 and Cin == 2:     # dedicated mma.sync first-layer kernel
            self._k("bd_encoder_conv0", ptr(x), 1, norm.data_ptr() + 16, 8, ptr(W[f"{p}.conv.w"]), ptr(W[f"{p}.conv.b"]),
                    ptr(y), B, 1, Tout, Tin, Cin, Cc, self.math, self._stream(), flops=2.0 * B * Tout * Cc * 8 * Cin,
                    nbytes=4.0 * B * (Cin * Tin + Tout * Cc), label="encoder_conv0_mma", detail=f"M={B * Tout} cin={Cin}")
        else:
            self._gemm(M=B * Tout, N=Cc, Cin=Cin, x=x, w=W[f"{p}.conv.w"], bias=W[f"{p}.conv.b"], out=y,
                       taps=tuple((0, k - 2) for k in range(8)), I1=1, I0=Tout, m0=4, J1=1, J0=Tin_p,
                       xs=(Cin * Tin, 0, 1, Tin) if first else (Tin_p * Cin, 0, Cin, 1), os_=(Tout * Cc, 0, Cc),
                       a_mode=_lib.A_ITEM_AFFINE if first else _lib.A_NONE, a_stats=norm[4:] if first else None,
                       a_stats_stride=8, act=_lib.ACT_NONE if conv_only else _lib.ACT_GELU)
        if conv_only:
            _tap(taps, f"tenc{i}", y.view(B, Tout, Cc), "t")
            return y
        if self.cfg.dconv_mode & 1:
            self._dconv(key, p, y, B, Tout, 1, Cc, "_t")
        z = self._buf(key, f"saved_t{i}", B * _pitch(Tout) * Cc, zero=True)
        self._gemm(M=B * Tout, N=2 * Cc, Cin=Cc, x=y, w=W[f"{p}.rewrite.w"], bias=W[f"{p}.rewrite.b"], out=z,
                   act=_lib.ACT_GLU, I1=1, I0=Tout, J1=1, J0=Tout, xs=(Tout * Cc, 0, Cc, 1), os_=(_pitch(Tout) * Cc, 0, Cc))
        _tap(taps, f"tenc{i}", z.view(B, _pitch(Tout), Cc)[:, :Tout], "t")
        return z

    def _freq_encoder(self, key, i, x, y_name, norm, taps, B, T, Fin, Cin, Cc) -> torch.Tensor:
        """Frequency-branch HEncLayer i: Conv2d(k=(8,1), s=(4,1), p=(2,0)) + GELU of x [B, T, Fin, Cin] into buffer
        ``y_name``, DConv, k=1 rewrite + GLU (+ freq_emb after layer 0) into the returned skip tensor ``saved_f{i}``."""
        W, p = self.W, f"encoder.{i}"
        first = i == 0
        Fo = Fin // 4
        y = self._buf(key, y_name, B * T * Fo * Cc)
        if first and self.mode != "fp32" and Cc == 48 and Cin == 4:     # dedicated mma.sync first-layer kernel
            self._k("bd_encoder_conv0", ptr(x), 0, ptr(norm), 8, ptr(W[f"{p}.conv.w"]), ptr(W[f"{p}.conv.b"]), ptr(y),
                    B, T, Fo, Fin, Cin, Cc, self.math, self._stream(), flops=2.0 * B * T * Fo * Cc * 8 * Cin,
                    nbytes=4.0 * B * T * (Fin * Cin + Fo * Cc), label="encoder_conv0_mma", detail=f"M={B * T * Fo} cin={Cin}")
        else:
            self._gemm(M=B * T * Fo, N=Cc, Cin=Cin, x=x, w=W[f"{p}.conv.w"], bias=W[f"{p}.conv.b"], out=y,
                       taps=tuple((0, k - 2) for k in range(8)), I1=T, I0=Fo, m0=4, J1=T, J0=Fin,
                       xs=(T * Fin * Cin, Fin * Cin, Cin, 1), os_=(T * Fo * Cc, Fo * Cc, Cc),
                       a_mode=_lib.A_ITEM_AFFINE if first else _lib.A_NONE, a_stats=norm if first else None,
                       a_stats_stride=8, act=_lib.ACT_GELU)
        if self.cfg.dconv_mode & 1:
            self._dconv(key, p, y, B, T, Fo, Cc, "_f")
        z = self._buf(key, f"saved_f{i}", B * T * Fo * Cc)
        emb = W["freq_emb"] if (first and self.cfg.freq_emb) else None
        self._gemm(M=B * T * Fo, N=2 * Cc, Cin=Cc, x=y, w=W[f"{p}.rewrite.w"], bias=W[f"{p}.rewrite.b"], out=z,
                   act=_lib.ACT_GLU, rowbias=emb, rowbias_period=Fo if emb is not None else 0)
        _tap(taps, f"enc{i}", z.view(B, T, Fo, Cc), "f")
        return z

    def _freq_decoder(self, key, j, x, y_name, out, skip, taps, B, T, Fr, Cc, Cout) -> None:
        """Frequency-branch HDecLayer j: 3x3 rewrite + GLU of x [B, T, Fr, Cc] into buffer ``y_name`` (hdemucs.py:312-313),
        DConv, ConvTranspose2d(k=(8,1), s=(4,1)) + crop [2:-2] + GELU + skip into ``out`` (hdemucs.py:326-334).  The last
        layer (skip None) has no activation and writes source-major [B, T, S, F, 4]: an iSTFT frame is contiguous."""
        W, p = self.W, f"decoder.{j}"
        last = skip is None
        y = self._buf(key, y_name, B * T * Fr * Cc)
        taps9 = tuple((kt - 1, kf - 1) for kf in range(3) for kt in range(3))
        self._gemm(M=B * T * Fr, N=2 * Cc, Cin=Cc, x=x, w=W[f"{p}.rewrite.w"], bias=W[f"{p}.rewrite.b"], out=y,
                   taps=taps9, I1=T, I0=Fr, J1=T, J0=Fr, xs=(T * Fr * Cc, Fr * Cc, Cc, 1), os_=(T * Fr * Cc, Fr * Cc, Cc),
                   act=_lib.ACT_GLU)
        if self.cfg.dconv_mode & 2:
            self._dconv(key, p, y, B, T, Fr, Cc, "_f")
        three = self.mode != "fp32" and 4 * Cout >= 64   # tensor-core form: no halo row
        self._gemm(M=B * T * (Fr + (0 if three else 1)), N=4 * Cout, Cin=Cc, x=y,
                   w=W[f"{p}.conv_tr.w3" if three else f"{p}.conv_tr.w"], bias=W[f"{p}.conv_tr.b"], out=out,
                   taps=((0, -1), (0, 0), (0, 1)) if three else ((0, 0), (0, -1)), I1=T, I0=Fr + (0 if three else 1),
                   J1=T, J0=Fr, xs=(T * Fr * Cc, Fr * Cc, Cc, 1),
                   os_=(T * 4 * Fr * Cout, 4 * Fr * Cout, 4 if last else Cout),
                   oc_split=4 if last else 0, oc_stride=4 * Fr * 4 if last else 0, convt=2 if three else 1, O0=4 * Fr,
                   act=_lib.ACT_NONE if last else _lib.ACT_GELU, addend=skip)
        if taps is not None:
            if last:   # [B,T,S,F,4] -> [B,T,F,(s j)]
                S = self.cfg.n_sources
                _tap(taps, f"dec{j}", out.view(B, T, S, 4 * Fr, 4).permute(0, 1, 3, 2, 4).reshape(B, T, 4 * Fr, Cout), "f")
            else:
                _tap(taps, f"dec{j}", (out - skip).view(B, T, 4 * Fr, Cout), "f")

    def _time_decoder(self, key, j, x, y_name, out, skip, taps, B, Tin, Tout, Cc, Cout) -> None:
        """Time-branch HDecLayer j: k=3 rewrite + GLU of x into buffer ``y_name``, DConv, ConvTranspose1d(k=8, s=4) + crop
        [2:2+Tout] + GELU + skip into ``out``; the last layer (skip None) has no activation."""
        W, p = self.W, f"tdecoder.{j}"
        y = self._buf(key, y_name, B * Tin * Cc)
        self._gemm(M=B * Tin, N=2 * Cc, Cin=Cc, x=x, w=W[f"{p}.rewrite.w"], bias=W[f"{p}.rewrite.b"], out=y,
                   taps=((0, -1), (0, 0), (0, 1)), I1=1, I0=Tin, J1=1, J0=Tin, xs=(_pitch(Tin) * Cc, 0, Cc, 1),
                   os_=(Tin * Cc, 0, Cc), act=_lib.ACT_GLU)
        if self.cfg.dconv_mode & 2:
            self._dconv(key, p, y, B, Tin, 1, Cc, "_t")
        three = self.mode != "fp32" and 4 * Cout >= 64
        self._gemm(M=B * (Tin + (0 if three else 1)), N=4 * Cout, Cin=Cc, x=y,
                   w=W[f"{p}.conv_tr.w3" if three else f"{p}.conv_tr.w"], bias=W[f"{p}.conv_tr.b"], out=out,
                   taps=((0, -1), (0, 0), (0, 1)) if three else ((0, 0), (0, -1)), I1=1, I0=Tin + (0 if three else 1),
                   J1=1, J0=Tin, xs=(Tin * Cc, 0, Cc, 1), os_=(_pitch(Tout) * Cout, 0, Cout), convt=2 if three else 1,
                   O0=Tout, act=_lib.ACT_NONE if skip is None else _lib.ACT_GELU, addend=skip)
        if taps is not None:
            _tap(taps, f"tdec{j}", (out - skip if skip is not None else out).view(B, _pitch(Tout), Cout)[:, :Tout], "t")

    def _istft(self, xf, xt, norm, out_buf, B, T, L, L0) -> torch.Tensor:
        """K2: de-normalise the spectrogram branch xf, iSTFT, overlap-add in shared memory, crop to L0 samples, add the
        time branch xt -> [B, S, A, L0] (written into ``out_buf`` when given)."""
        S, A = self.cfg.n_sources, self.cfg.audio_channels
        if out_buf is not None:
            if out_buf.numel() != B * S * A * L0 or out_buf.dtype != torch.float32 or out_buf.device != self.device \
                    or not out_buf.is_contiguous():
                raise ValueError("out must be a contiguous float32 tensor of B*S*C*L elements on the engine's device")
            out = out_buf.view(B, S, A, L0)
        else:
            out = torch.empty(B, S, A, L0, dtype=torch.float32, device=self.device)
        self._k("bd_istft_ola", ptr(xf), ptr(norm), ptr(self.window), ptr(self.twiddle), ptr(xt), ptr(out),
                B, S, T, _pitch(L), L0, self._stream(), nbytes=4.0 * B * S * (T * 2048 * 4 + 2 * L + 2 * L0),
                flops=2.5 * 4096 * 12 * 2 * S * B * T)
        return out

    # ------------------------------------------------------------------ forward
    @torch.no_grad()
    def forward(self, mix: torch.Tensor, taps: tp.Optional[dict] = None, out: tp.Optional[torch.Tensor] = None) -> torch.Tensor:
        """mix [B, 2, L <= segment_length] (fp32, on self.device) -> [B, S, 2, L] (written into ``out`` when given)."""
        return self._run(mix, taps, out)

    @torch.no_grad()
    def forward_core(self, mag: torch.Tensor, mix: torch.Tensor) -> tp.Tuple[torch.Tensor, torch.Tensor]:
        """The network between the STFT and the iSTFT (reference ``HTDemucs.forward_core``, htdemucs.py:662-759, its
        ONNX-export surface): mag [B, 2*audio_channels, 2048, T] = ``_magnitude(_spec(mix))`` (any tensor of that
        shape is accepted, as in the reference), mix [B, audio_channels, L = training length] ->
        (spec_out [B, S, 2*audio_channels, 2048, T], time_out [B, S, audio_channels, L]), both de-normalised.
        The layout changes at this boundary (NCHW in and out) are plain copies; everything between runs in the
        same kernels as ``forward``."""
        return self._run(mix, None, None, mag)

    def _run(self, mix: torch.Tensor, *args):
        # kernels launch on the CURRENT device: make that the engine's device whatever the caller's is; and any
        # failure -- not only a kernel error -- may leave the self-clearing statistics workspaces dirty
        try:
            if mix.dim() != 3 or mix.shape[1] != self.cfg.audio_channels:
                raise ValueError(f"expected mix of shape [B, {self.cfg.audio_channels}, L], got {tuple(mix.shape)}")
            if mix.device != self.device or mix.dtype != torch.float32:
                raise ValueError("mix must be a float32 tensor on the engine's device")
            with torch.cuda.device(self.device) if self.device.type == "cuda" else contextlib.nullcontext():
                return self._forward(mix, *args)
        except BaseException:
            self._bufs.clear()
            raise

    def _forward(self, mix: torch.Tensor, taps: tp.Optional[dict], out_buf: tp.Optional[torch.Tensor], mag=None):
        cfg, W = self.cfg, self.W
        B, A, L0 = mix.shape
        L = cfg.segment_length
        if L0 > L:  # htdemucs.py:521-524
            raise ValueError(f"Given length {L0} is longer than training length {L}")
        key = (B, L)
        S = cfg.n_sources
        T = cfg.frames(L)
        chans = cfg.enc_channels
        if mag is not None and (L0 != L or tuple(mag.shape) != (B, 2 * A, 2048, T) or mag.device != self.device
                                or mag.dtype != torch.float32):
            raise ValueError(f"forward_core expects mag [B, {2 * A}, 2048, {T}] and mix [B, {A}, {L}] (float32, on "
                             f"the engine's device), got {tuple(mag.shape)} and {tuple(mix.shape)}")
        if L0 < L:  # htdemucs.py:534-537: zero-pad on the right up to the training length
            padded = self._buf(key, "mix_padded", B * A * L).view(B, A, L)
            padded.zero_()
            padded[..., :L0].copy_(mix)
            mix = padded
        mix = mix.contiguous()
        spec, norm = self._stft(key, mix, taps, mag)

        # ---- encoders ------------------------------------------------------------------------
        tl = cfg.time_lengths(L)
        saved, saved_t = [], []
        xf, Fin, Cin = spec, 2048, 2 * A
        xt, Cin_t = mix, A
        for i, Cc in enumerate(chans):
            xt = self._time_encoder(key, i, xt, "y_t", norm, taps, B, tl[i], tl[i + 1], Cin_t, Cc)
            xf = self._freq_encoder(key, i, xf, "y_f", norm, taps, B, T, Fin, Cin, Cc)
            saved_t.append(xt)
            saved.append(xf)
            Fin, Cin, Cin_t = Fin // 4, Cc, Cc

        Fb, Cb, T2 = Fin, chans[-1], tl[-1]
        Mf, Mt = B * T * Fb, B * T2
        # ping-pong buffers of the decoders, sized for their largest activation
        dec_f_numel = B * T * max(2048 * 4 * S, 512 * chans[0])
        dec_t_numel = B * max(_pitch(L) * 2 * S, _pitch(tl[1]) * chans[0])

        xd = self._buf(key, "dec_a", dec_f_numel)[: Mf * Cb]
        xtd = self._buf(key, "dec_ta", dec_t_numel)[: B * _pitch(T2) * Cb]

        # ---- cross-domain transformer ------------------------------------------------------------
        if cfg.t_layers > 0:
            D = cfg.transformer_dim
            x = self._buf(key, "tr_x", Mf * D)
            xt_ = self._buf(key, "tr_xt", Mt * D)
            if cfg.bottom_channels:
                self._gemm(M=Mf, N=D, Cin=Cb, x=xf, w=W["channel_upsampler.w"], bias=W["channel_upsampler.b"], out=x)
                self._gemm(M=Mt, N=D, Cin=Cb, x=xt, w=W["channel_upsampler_t.w"], bias=W["channel_upsampler_t.b"],
                           out=xt_, I1=1, I0=T2, J1=1, J0=T2, xs=(_pitch(T2) * Cb, 0, Cb, 1), os_=(T2 * D, 0, D))
            else:
                x.copy_(xf)
                xt_.view(B, T2, D).copy_(xt.view(B, _pitch(T2), Cb)[:, :T2])
            ct = "crosstransformer"
            pos2d = self._pos_table(("2d", Fb, T))
            pos1d = self._pos_table(("1d", T2))
            self._ln(x, x, f"{ct}.norm_in", Mf, pos2d, T * Fb)
            self._ln(xt_, xt_, f"{ct}.norm_in_t", Mt, pos1d, T2)
            for i in range(cfg.t_layers):
                if i % 2 == 0:
                    self._transformer_layer(key, x, None, f"{ct}.layers.{i}", False, B, T * Fb, T * Fb, "_f")
                    self._transformer_layer(key, xt_, None, f"{ct}.layers_t.{i}", False, B, T2, T2, "_t")
                else:
                    # both sides attend to the other's *pre-update* tokens (transformer.py:669-672)
                    kdt = torch.bfloat16 if self.mode == "bf16" else torch.float32
                    kf = self._buf(key, "kn_f", Mt * D, kdt)   # keys for the freq side = LN2(xt)
                    kt = self._buf(key, "kn_t", Mf * D, kdt)   # keys for the time side = LN2_t(old x)
                    self._ln(xt_, kf, f"{ct}.layers.{i}.norm2", Mt)
                    self._ln(x, kt, f"{ct}.layers_t.{i}.norm2", Mf)
                    self._transformer_layer(key, x, kf, f"{ct}.layers.{i}", True, B, T * Fb, T2, "_f")
                    self._transformer_layer(key, xt_, kt, f"{ct}.layers_t.{i}", True, B, T2, T * Fb, "_t")
                _tap(taps, f"xf.layer{i}", x.view(B, T, Fb, D), "f")
                _tap(taps, f"xt.layer{i}", xt_.view(B, T2, D), "t")
            # channel_downsampler (+ the decoder's skip add, hdemucs.py:310, fused as `addend`)
            if cfg.bottom_channels:
                self._gemm(M=Mf, N=Cb, Cin=D, x=x, w=W["channel_downsampler.w"], bias=W["channel_downsampler.b"],
                           out=xd, addend=saved[-1])
                self._gemm(M=Mt, N=Cb, Cin=D, x=xt_, w=W["channel_downsampler_t.w"],
                           bias=W["channel_downsampler_t.b"], out=xtd, addend=saved_t[-1], I1=1, I0=T2, J1=1, J0=T2,
                           xs=(T2 * D, 0, D, 1), os_=(_pitch(T2) * Cb, 0, Cb))
            else:
                torch.add(x, saved[-1], out=xd)
                xtd.view(B, _pitch(T2), Cb)[:, :T2].copy_(xt_.view(B, T2, Cb) + saved_t[-1].view(B, _pitch(T2), Cb)[:, :T2])
            if taps is not None:
                _tap(taps, "bottleneck", (xd - saved[-1]).view(B, T, Fb, Cb), "f")
                _tap(taps, "bottleneck_t", (xtd - saved_t[-1]).view(B, _pitch(T2), Cb)[:, :T2], "t")
        else:
            torch.add(xf, saved[-1], out=xd)
            torch.mul(saved_t[-1], 2.0, out=xtd)    # no transformer: x + skip with skip == x

        # ---- decoders ------------------------------------------------------------------------------
        Fcur = Fb
        for j in range(cfg.depth):
            Cc = chans[cfg.depth - 1 - j]
            last = j == cfg.depth - 1
            Cout = 4 * S if last else Cc // 2
            Cout_t = 2 * S if last else Cc // 2
            skip = None if last else saved[cfg.depth - 2 - j]
            skip_t = None if last else saved_t[cfg.depth - 2 - j]
            nxt = self._buf(key, ("dec_a", "dec_b")[(j + 1) % 2], dec_f_numel)[: B * T * 4 * Fcur * Cout]
            self._freq_decoder(key, j, xd, "y_f", nxt, skip, taps, B, T, Fcur, Cc, Cout)
            xd, Fcur = nxt, 4 * Fcur
            Tin, Tout = tl[cfg.depth - j], tl[cfg.depth - 1 - j]
            nxt = self._buf(key, ("dec_ta", "dec_tb")[(j + 1) % 2], dec_t_numel)[: B * _pitch(Tout) * Cout_t]
            self._time_decoder(key, j, xtd, "y_t", nxt, skip_t, taps, B, Tin, Tout, Cc, Cout_t)
            xtd = nxt

        if mag is not None:
            # forward_core: hand back both branches de-normalised (htdemucs.py:751-757), in the reference's layouts
            nm = norm.view(B, 8)
            spec_out = xd[: B * T * S * 2048 * 2 * A].view(B, T, S, 2048, 2 * A).permute(0, 2, 4, 3, 1)
            spec_out = spec_out * nm[:, 1].view(B, 1, 1, 1, 1) + nm[:, 0].view(B, 1, 1, 1, 1)
            time_out = xtd[: B * _pitch(L) * A * S].view(B, _pitch(L), S, A)[:, :L].permute(0, 2, 3, 1)
            time_out = time_out * nm[:, 5].view(B, 1, 1, 1) + nm[:, 4].view(B, 1, 1, 1)
            return spec_out.contiguous(), time_out.contiguous()
        out = self._istft(xd, xtd, norm, out_buf, B, T, L, L0)
        if taps is not None:
            only = torch.empty(B, S, A, L0, dtype=torch.float32, device=self.device)
            self._k("bd_istft_ola", ptr(xd), ptr(norm), ptr(self.window), ptr(self.twiddle), None, ptr(only),
                    B, S, T, _pitch(L), L0, self._stream())
            taps["istft"] = only
            taps["time_out"] = out - only
        return out

    def _pos_table(self, key) -> torch.Tensor:
        t = self._pos.get(key)
        if t is None:
            cfg = self.cfg
            D = cfg.transformer_dim
            if key[0] == "2d":
                t = _sin_embedding_2d(D, key[1], key[2], cfg.t_max_period)
            else:
                t = _sin_embedding_1d(key[1], D, cfg.t_max_period)
            t = (cfg.t_weight_pos_embed * t).to(self.device).contiguous()
            self._pos[key] = t
        return t
