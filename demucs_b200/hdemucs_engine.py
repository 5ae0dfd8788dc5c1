"""Host-side orchestration of the Hybrid Demucs v3 forward on the sm_100a kernel library.

Python mirror of ``HDemucs.forward`` (reference demucs/hdemucs.py:689-794) for the hdemucs_mmi family, as a sequence of
C-ABI launches.  It is an HTDemucs ``Engine`` with another weight packing: the STFT / iSTFT and the HTDemucs-style
encoder / decoder layers are the ``Engine``'s own steps; what is specific to v3:

* layers 0-3 are the HTDemucs encoder / decoder layers without a decoder DConv (``dconv_mode=1``) and with
  ``dconv_comp=4`` (hidden widths 12 / 24 / 48 / 96);
* layer 4 closes the frequency axis: its k=8 convolution over the 8 remaining bins is ONE GEMM over the contiguous
  8*384 floats of a frame (channels-last makes the (bin, channel) window a dense row), the time branch's conv-only
  layer is added as the GEMM's ``addend`` (``inject``, hdemucs.py:137-143), and the transposed convolution back to 8 bins
  is a GEMM with 8*384 output columns;
* layer 5 works on the merged branch along time (k=4, s=2): position pairs are viewed as 1536-channel rows so that it is a
  3-tap unit-stride implicit GEMM (zero blocks where a tap does not reach), its transposed form a 2-tap GEMM producing
  both output phases of a row;
* layers 4-5 normalise with GroupNorm(4) (``bd_gn_stats`` / ``bd_gn_act``, the decoder ones BEFORE the crop as the
  reference does) and their DConv branches carry a 2-layer BiLSTM over 200-step frames and LocalState attention
  (``bd_lstm_*``, ``bd_local_state``), with every projection around them a ``bd_conv_gemm``;
* the decoder starts from zeros (hdemucs.py:742-744), so its first layer reads the skip tensor directly.
"""
from __future__ import annotations

import math
import typing as tp

import torch

from . import _lib
from ._lib import ptr
from .engine import Engine, _conv3_geometry, _pitch, _tap, conv_w, convtr_w, pack_dconv, pack_decoder, pack_encoder
from .hdemucs import HDemucsConfig, param_specs


def _check_state(cfg: HDemucsConfig, state) -> None:
    specs = param_specs(cfg)
    missing = [k for k in specs if k not in state]
    extra = [k for k in state if k not in specs]
    if missing or extra:
        raise KeyError(f"state dict mismatch: missing={missing[:4]}... extra={extra[:4]}...")
    for k, (shape, _, _) in specs.items():
        if tuple(state[k].shape) != tuple(shape):
            raise ValueError(f"{k}: expected shape {shape}, got {tuple(state[k].shape)}")


class HDemucsWeights:
    """Reference ``HDemucs.state_dict()`` -> kernel layouts (one-time, on the device)."""

    def __init__(self, cfg: HDemucsConfig, state, device, tc_forms: bool):
        _check_state(cfg, state)
        self.t: tp.Dict[str, torch.Tensor] = {}

        def put(name, tensor):
            self.t[name] = tensor.detach().to(device=device, dtype=torch.float32).contiguous()

        f32 = lambda k: state[k].detach().float()   # noqa: E731
        L = cfg.layers()
        n_time = sum(1 for l in L if l["has_time"])
        for l in L:
            i, j = l["index"], cfg.depth - 1 - l["index"]
            e, d = f"encoder.{i}", f"decoder.{j}"
            big = l["lstm"] or l["attn"]
            # DConv: (conv3, norm1, [BLSTM], [LocalState], conv1x1, norm2, GLU, LayerScale) -- demucs.py:133-150
            k = 3 + int(l["lstm"]) + int(l["attn"])
            idx = (0, 1, k, k + 1, k + 3)
            put(f"{e}.rewrite.b_nat", f32(f"{e}.rewrite.bias"))
            if not l["norm"]:
                pack_encoder(put, state, e)
            else:
                # GroupNorm'd layers keep the reference's channel order: the GLU runs after the norm, in bd_gn_act
                put(f"{e}.conv.b", f32(f"{e}.conv.bias"))
                put(f"{e}.rewrite.w", conv_w(f32(f"{e}.rewrite.weight")))
                put(f"{e}.rewrite.b", f32(f"{e}.rewrite.bias"))
                for n in ("norm1", "norm2"):
                    put(f"{e}.{n}.g", f32(f"{e}.{n}.weight"))
                    put(f"{e}.{n}.b", f32(f"{e}.{n}.bias"))
                    put(f"{d}.{n}.g", f32(f"{d}.{n}.weight"))
                    put(f"{d}.{n}.b", f32(f"{d}.{n}.bias"))
                if l["last_freq"]:
                    put(f"{e}.conv.w", conv_w(f32(f"{e}.conv.weight")))                   # [Cout, 8*Cin]: one dense row per frame
                else:
                    # Conv1d(k=4, s=2, p=1) over position PAIRS: out[t] = w0 x[2t-1] + w1 x[2t] + w2 x[2t+1] + w3 x[2t+2];
                    # pair rows [x[2p] | x[2p+1]], taps (-1, 0, +1) with zero blocks where a tap does not reach
                    w = f32(f"{e}.conv.weight")                                           # [Cout, Cin, 4]
                    co, ci = w.shape[:2]
                    z = w.new_zeros(co, ci)
                    put(f"{e}.conv.wpair", torch.cat([z, w[:, :, 0], w[:, :, 1], w[:, :, 2], w[:, :, 3], z], dim=1))
            pack_dconv(put, self.t, state, e, cfg.dconv_depth, tc_forms, idx)
            if big:
                hid = state[f"{e}.dconv.layers.0.0.weight"].shape[0]
                for dd in range(cfg.dconv_depth):
                    p = f"{e}.dconv.layers.{dd}"
                    lp, ap = f"{p}.3", f"{p}.4"
                    for layer in range(2):
                        put(f"{p}.lstm.wih{layer}", torch.cat([f32(f"{lp}.lstm.weight_ih_l{layer}"),
                                                               f32(f"{lp}.lstm.weight_ih_l{layer}_reverse")], 0))
                        put(f"{p}.lstm.b{layer}", torch.cat([
                            f32(f"{lp}.lstm.bias_ih_l{layer}") + f32(f"{lp}.lstm.bias_hh_l{layer}"),
                            f32(f"{lp}.lstm.bias_ih_l{layer}_reverse") + f32(f"{lp}.lstm.bias_hh_l{layer}_reverse")], 0))
                        put(f"{p}.lstm.whhT{layer}", torch.stack([f32(f"{lp}.lstm.weight_hh_l{layer}").t(),
                                                                  f32(f"{lp}.lstm.weight_hh_l{layer}_reverse").t()], 0))
                    put(f"{p}.lstm.lin.w", f32(f"{lp}.linear.weight"))
                    put(f"{p}.lstm.lin.b", f32(f"{lp}.linear.bias"))
                    put(f"{p}.attn.qkc.w", torch.cat([f32(f"{ap}.{n}.weight").squeeze(-1) for n in ("query", "key", "content")], 0))
                    put(f"{p}.attn.qkc.b", torch.cat([f32(f"{ap}.{n}.bias") for n in ("query", "key", "content")], 0))
                    put(f"{p}.attn.dq.w", f32(f"{ap}.query_decay.weight").squeeze(-1))
                    put(f"{p}.attn.dq.b", f32(f"{ap}.query_decay.bias"))
                    put(f"{p}.attn.proj.w", f32(f"{ap}.proj.weight").squeeze(-1))
                    put(f"{p}.attn.proj.b", f32(f"{ap}.proj.bias"))
                    assert hid % 16 == 0
            # decoder of this index
            if l["norm"]:
                if l["freq"]:      # 3x3 on a single frequency row: only the middle kernel row meets data (padding 1)
                    put(f"{d}.rewrite.w", conv_w(f32(f"{d}.rewrite.weight")[:, :, 1, :]))
                else:
                    put(f"{d}.rewrite.w", conv_w(f32(f"{d}.rewrite.weight")))
                put(f"{d}.rewrite.b", f32(f"{d}.rewrite.bias"))
                w = f32(f"{d}.conv_tr.weight")
                if l["freq"]:      # ConvTranspose2d(k=(8,1), s=(4,1)) from one bin: bin f of the output = w[:, :, f]
                    ci, co = w.shape[:2]
                    put(f"{d}.conv_tr.w", w.reshape(ci, co, 8).permute(2, 1, 0).reshape(8 * co, ci))
                    put(f"{d}.conv_tr.b", f32(f"{d}.conv_tr.bias").repeat(8))
                else:              # ConvTranspose1d(k=4, s=2), full output: row p = (2p, 2p+1), taps p and p-1
                    ci, co = w.shape[:2]
                    put(f"{d}.conv_tr.w", w.reshape(ci, co, 2, 2).permute(3, 1, 2, 0).reshape(2 * co, 2 * ci))
                    put(f"{d}.conv_tr.b", f32(f"{d}.conv_tr.bias").repeat(2))
            else:
                pack_decoder(put, state, d, tc_forms)
            if not l["has_time"]:
                continue
            te, td = f"tencoder.{i}", f"tdecoder.{n_time - 1 - i}"
            if l["time_empty"]:    # conv-only layers (hdemucs.py:137-143); the decoder's GroupNorm runs before its crop
                put(f"{te}.conv.w", conv_w(f32(f"{te}.conv.weight")))
                put(f"{te}.conv.b", f32(f"{te}.conv.bias"))
                put(f"{td}.conv_tr.w", convtr_w(f32(f"{td}.conv_tr.weight")))
                put(f"{td}.conv_tr.b", f32(f"{td}.conv_tr.bias").repeat(4))
                put(f"{td}.norm2.g", f32(f"{td}.norm2.weight"))
                put(f"{td}.norm2.b", f32(f"{td}.norm2.bias"))
                continue
            pack_encoder(put, state, te)
            pack_dconv(put, self.t, state, te, cfg.dconv_depth, tc_forms)
            pack_decoder(put, state, td, tc_forms)
        if cfg.freq_emb:
            put("freq_emb", cfg.freq_emb * cfg.emb_scale * f32("freq_emb.embedding.weight"))

    def __getitem__(self, k: str) -> torch.Tensor:
        return self.t[k]


class HDemucsEngine(Engine):
    """One HDemucs (v3) model resident on one GPU."""

    Weights = HDemucsWeights

    def __init__(self, cfg: HDemucsConfig, state, device="cuda", mode: str = "strict"):
        super().__init__(cfg, state, device, mode)

    # ------------------------------------------------------------------ GroupNorm(4) helpers
    def _gn(self, key, x, y, p: str, B: int, rows_in: int, C_: int, act: int, row0: int = 0, rows_out: tp.Optional[int] = None,
            addend=None, y_item_stride: tp.Optional[int] = None, tag: str = ""):
        """y = act(GroupNorm(4)(x)) over x [B, rows_in, C] (statistics over all rows_in), rows [row0, row0+rows_out) kept."""
        G = self.cfg.norm_groups
        rows_out = rows_in if rows_out is None else rows_out
        Co = C_ // 2 if act == _lib.ACT_GLU else C_
        sums = self._buf(key, f"gn_sums{tag}", 2 * B * G, torch.float64, zero=True)     # finalize clears it again
        mr = self._buf(key, f"gn_mr{tag}", 2 * B * G)
        st = self._stream()
        self._k("bd_gn_stats", ptr(x), ptr(sums), B, rows_in, C_, G, st, nbytes=4.0 * B * rows_in * C_)
        self._k("bd_finalize_group_stats", ptr(sums), ptr(mr), B * G, float(rows_in * (C_ // G)), st)
        self._k("bd_gn_act", ptr(x), ptr(y), ptr(mr), ptr(self.W[f"{p}.g"]), ptr(self.W[f"{p}.b"]), ptr(addend), B, rows_in,
                row0, rows_out, C_, G, act, rows_out * Co if y_item_stride is None else y_item_stride, st,
                nbytes=4.0 * B * rows_out * (C_ + Co))

    # ------------------------------------------------------------------ DConv with BLSTM / LocalState / wide hidden
    def _dconv_big(self, key, prefix: str, x, B: int, T: int, Fr: int, C_: int, lstm: bool, attn: bool, tag: str):
        """DConv (demucs.py:86-154) where the hidden width exceeds the register kernels (> 48) or carries the BLSTM /
        LocalState modules: every contraction is a ``bd_conv_gemm``; x [B, T, Fr, C] is updated in place."""
        cfg, W = self.cfg, self.W
        hid = int(C_ / cfg.dconv_comp)
        tc = self.mode != "fp32"
        hp = (hid + 15) // 16 * 16 if tc else hid
        M, slabs = B * T * Fr, B * Fr
        stat = (T * Fr, Fr, Fr)
        h = self._buf(key, f"dconv_h{tag}", M * hp)
        sums = self._buf(key, f"dconv_sums{tag}", 2 * slabs, torch.float64, zero=True)
        mr1 = self._buf(key, f"dconv_mr1{tag}", 2 * slabs)
        mr2 = self._buf(key, f"dconv_mr2{tag}", 2 * slabs)
        sfx = "p" if tc else ""
        st = self._stream()
        for dd in range(cfg.dconv_depth):
            p = f"{prefix}.dconv.layers.{dd}"
            dil = 2 ** dd
            self._gemm(M=M, N=hp, Cin=C_, x=x, w=W[f"{p}.w1{sfx}"], bias=W[f"{p}.b1{sfx}"], out=h, stats_out=sums, stat=stat,
                       tc=tc, **_conv3_geometry(T, Fr, C_, hp, dil))
            self._k("bd_finalize_group_stats", ptr(sums), ptr(mr1), slabs, float(T * hid), st)
            self._k("bd_gn_gelu_apply", ptr(h), ptr(mr1), ptr(W[f"{p}.g1{sfx}"]), ptr(W[f"{p}.be1{sfx}"]), M, hp, T * Fr, Fr, st,
                    nbytes=8.0 * M * hp, label="bd_gn_gelu_apply")
            if lstm:
                assert Fr == 1 and hp == hid
                self._blstm(key, p, h, B, T, hid, tag)
            if attn:
                assert Fr == 1 and hp == hid
                self._local_state(key, p, h, B, T, hid, tag)
            # statistics of u = W2 h + b2 (no store), then x += scale * GLU(gn(u)) in the epilogue of the same product
            ugeo = dict(I1=1, I0=T, J1=1, J0=T, xs=(T * hp, 0, hp, 1), os_=(T * 2 * C_, 0, 2 * C_)) if Fr == 1 else {}
            self._gemm(M=M, N=2 * C_, Cin=hp, x=h, w=W[f"{p}.w2{sfx}" if tc else f"{p}.w2"], bias=W[f"{p}.b2"], out=None,
                       stats_out=sums, stat=stat, tc=tc, **ugeo)
            self._k("bd_finalize_group_stats", ptr(sums), ptr(mr2), slabs, float(T * 2 * C_), st)
            self._gemm(M=M, N=2 * C_, Cin=hp, x=h, w=W[f"{p}.w2{sfx}" if tc else f"{p}.w2"], bias=W[f"{p}.b2"], e_stats=mr2,
                       e_gamma=W[f"{p}.g2"], e_beta=W[f"{p}.be2"], act=_lib.ACT_GLU, resid=x, scale=W[f"{p}.scale"], out=x,
                       stat=stat, tc=tc)

    def _blstm(self, key, p: str, h, B: int, T: int, H: int, tag: str):
        """BLSTM(H, layers=2, max_steps=200, skip=True) in place on h [B, T, H] (demucs.py:37-67)."""
        W = self.W
        st = self._stream()
        width, stride = 200, 100
        framed = T > width
        if framed:
            nf = math.ceil(T / stride)
            N, Tt = B * nf, width
            seq = self._buf(key, f"lstm_frames{tag}", N * Tt * H)
            self._k("bd_lstm_frame", ptr(h), ptr(seq), B, T, H, nf, width, stride, st, nbytes=4.0 * (B * T + N * Tt) * H)
        else:
            nf, N, Tt, seq = 1, B, T, h
        pre = self._buf(key, f"lstm_pre{tag}", N * Tt * 8 * H)
        ws = self._buf(key, f"lstm_ws{tag}", 6 * N * H)
        cur, cin = seq, H
        for layer in range(2):
            self._gemm(M=N * Tt, N=8 * H, Cin=cin, x=cur, w=W[f"{p}.lstm.wih{layer}"], bias=W[f"{p}.lstm.b{layer}"], out=pre)
            out = self._buf(key, f"lstm_out{layer}{tag}", N * Tt * 2 * H)
            self._k("bd_lstm_bidir", ptr(pre), ptr(W[f"{p}.lstm.whhT{layer}"]), ptr(out), ptr(ws), N, Tt, H, st,
                    flops=16.0 * N * Tt * H * H, nbytes=4.0 * N * Tt * 10 * H, label="lstm_bidir")
            cur, cin = out, 2 * H
        if framed:
            lin = self._buf(key, f"lstm_lin{tag}", N * Tt * H)
            self._gemm(M=N * Tt, N=H, Cin=2 * H, x=cur, w=W[f"{p}.lstm.lin.w"], bias=W[f"{p}.lstm.lin.b"], out=lin)
            self._k("bd_lstm_unframe_add", ptr(lin), ptr(h), ptr(h), B, T, H, nf, width, stride, st, nbytes=12.0 * B * T * H)
        else:
            self._gemm(M=N * Tt, N=H, Cin=2 * H, x=cur, w=W[f"{p}.lstm.lin.w"], bias=W[f"{p}.lstm.lin.b"], out=h, resid=h)

    def _local_state(self, key, p: str, h, B: int, T: int, D: int, tag: str):
        """LocalState(D, heads=4, ndecay=4) in place on h [B, T, D] (demucs.py:186-216)."""
        W = self.W
        st = self._stream()
        qkc = self._buf(key, f"ls_qkc{tag}", B * T * 3 * D)
        dq = self._buf(key, f"ls_dq{tag}", B * T * 16)
        res = self._buf(key, f"ls_res{tag}", B * T * D)
        self._gemm(M=B * T, N=3 * D, Cin=D, x=h, w=W[f"{p}.attn.qkc.w"], bias=W[f"{p}.attn.qkc.b"], out=qkc)
        self._gemm(M=B * T, N=16, Cin=D, x=h, w=W[f"{p}.attn.dq.w"], bias=W[f"{p}.attn.dq.b"], out=dq)
        self._k("bd_local_state", ptr(qkc), ptr(dq), ptr(res), B, T, D, 4, st, flops=4.0 * B * T * T * D,
                nbytes=4.0 * B * T * 4 * D, label="local_state")
        self._gemm(M=B * T, N=D, Cin=D, x=res, w=W[f"{p}.attn.proj.w"], bias=W[f"{p}.attn.proj.b"], out=h, resid=h)

    def _dconv(self, key, prefix, x, B, T, Fr, C_, tag: str, lstm: bool = False, attn: bool = False):
        """DConv of a v3 layer: with BLSTM / LocalState or a hidden width beyond the register kernels (> 48) it is
        ``_dconv_big``, otherwise the HTDemucs form."""
        if lstm or attn or int(C_ / self.cfg.dconv_comp) > 48:
            self._dconv_big(key, prefix, x, B, T, Fr, C_, lstm, attn, tag)
        else:
            super()._dconv(key, prefix, x, B, T, Fr, C_, tag)

    # ------------------------------------------------------------------ forward
    def forward_core(self, mag, mix):
        raise NotImplementedError("forward_core is the HTDemucs ONNX surface (htdemucs.py:662-759)")

    def _forward(self, mix: torch.Tensor, taps: tp.Optional[dict], out_buf: tp.Optional[torch.Tensor]):
        cfg, W = self.cfg, self.W
        B, A, L = mix.shape
        if L < 2560:     # the reflect padding of _spec (1536 + up to 1023 samples) must stay inside the signal; the
            raise ValueError("input shorter than 2560 samples: the small-input guard of pad1d (hdemucs.py:29-36) is not built")
        mix = mix.contiguous()
        key = (B, L)
        T = cfg.frames(L)
        layers = cfg.layers()
        spec, norm = self._stft(key, mix, taps)        # hdemucs.py:693-709

        # ---- encoders --------------------------------------------------------------------------------------------
        tl = [L]
        for l in layers:
            if l["has_time"]:
                tl.append(int(math.ceil(tl[-1] / 4)))
        if tl[-1] != T:
            raise ValueError(f"time branch ends on {tl[-1]} steps but the spectrogram has {T} frames")
        saved, saved_t = [], []
        xf, Fin, Cin = spec, 2048, 2 * A
        xt, Cin_t = mix, A
        inject = None
        T5 = (T + 1) // 2        # Conv1d(k=4, s=2, p=1) after right-padding T to even
        for l in layers:
            i, Cc = l["index"], l["chout_z"]
            if l["time_empty"]:     # conv only; added to the frequency branch below (hdemucs.py:137-143)
                inject = self._time_encoder(key, i, xt, f"y_t{i}", norm, taps, B, tl[i], tl[i + 1], Cin_t, Cc, conv_only=True)
            elif l["has_time"]:
                xt = self._time_encoder(key, i, xt, f"y_t{i}", norm, taps, B, tl[i], tl[i + 1], Cin_t, Cc)
                saved_t.append(xt)
                Cin_t = Cc
            e = f"encoder.{i}"
            if l["freq"] and not l["last_freq"]:
                xf = self._freq_encoder(key, i, xf, f"y_f{i}", norm, taps, B, T, Fin, Cin, Cc)
                saved.append(xf)
                Fin, Cin = Fin // 4, Cc
                continue
            # GroupNorm'd layers on the merged branch: rows = time steps, one "frequency" left
            if l["last_freq"]:
                rows = T
                raw = self._buf(key, f"raw{i}", B * rows * Cc)
                self._gemm(M=B * rows, N=Cc, Cin=Fin * Cin, x=xf, w=W[f"{e}.conv.w"], bias=W[f"{e}.conv.b"], out=raw,
                           addend=inject)
            else:
                rows = T5
                raw = self._buf(key, f"raw{i}", B * rows * Cc)
                Tp = T + (T & 1)                  # HEncLayer right-pads the time axis to a multiple of its stride (hdemucs.py:131-135)
                src = xf
                if Tp != T:
                    src = self._buf(key, "z4_padded", B * Tp * Cin, zero=True)
                    src.view(B, Tp, Cin)[:, :T].copy_(xf.view(B, T, Cin))
                self._gemm(M=B * rows, N=Cc, Cin=2 * Cin, x=src, w=W[f"{e}.conv.wpair"], bias=W[f"{e}.conv.b"], out=raw,
                           taps=((0, -1), (0, 0), (0, 1)), I1=1, I0=rows, J1=1, J0=Tp // 2,
                           xs=(Tp * Cin, 0, 2 * Cin, 1), os_=(rows * Cc, 0, Cc))
            self._gn(key, raw, raw, f"{e}.norm1", B, rows, Cc, _lib.ACT_GELU, tag=f"_e{i}a")
            self._dconv(key, e, raw, B, rows, 1, Cc, f"_m{i}", l["lstm"], l["attn"])
            rw = self._buf(key, f"rw{i}", B * rows * 2 * Cc)
            self._gemm(M=B * rows, N=2 * Cc, Cin=Cc, x=raw, w=W[f"{e}.rewrite.w"], bias=W[f"{e}.rewrite.b"], out=rw)
            z = self._buf(key, f"saved_f{i}", B * rows * Cc)
            self._gn(key, rw, z, f"{e}.norm2", B, rows, 2 * Cc, _lib.ACT_GLU, tag=f"_e{i}b")
            saved.append(z)
            xf, Fin, Cin = z, 1, Cc
            _tap(taps, f"enc{i}", z.view(B, rows, 1, Cc), "f")

        # ---- decoders: x starts at zero, so layer 0 reads its skip tensor alone (hdemucs.py:742-749) ---------------
        n_time = len(tl) - 1
        xd = saved[-1]
        xtd = None
        for j in range(cfg.depth):
            l = layers[cfg.depth - 1 - j]
            Cc, Cout = l["chout_z"], l["dec_out_z"]
            d = f"decoder.{j}"
            last = j == cfg.depth - 1
            nxt_skip = None if last else saved[cfg.depth - 2 - j]
            if l["norm"] and not l["freq"]:
                # index 5: k=3 rewrite over time, GroupNorm + GLU; ConvTranspose1d(k=4, s=2) in full, GroupNorm, crop, GELU
                rows = T5
                rw = self._buf(key, f"drw{j}", B * rows * 2 * Cc)
                self._gemm(M=B * rows, N=2 * Cc, Cin=Cc, x=xd, w=W[f"{d}.rewrite.w"], bias=W[f"{d}.rewrite.b"], out=rw,
                           taps=((0, -1), (0, 0), (0, 1)), I1=1, I0=rows, J1=1, J0=rows, xs=(rows * Cc, 0, Cc, 1),
                           os_=(rows * 2 * Cc, 0, 2 * Cc))
                y = self._buf(key, f"dy{j}", B * rows * Cc)
                self._gn(key, rw, y, f"{d}.norm1", B, rows, 2 * Cc, _lib.ACT_GLU, tag=f"_d{j}a")
                full = self._buf(key, f"dfull{j}", B * (rows + 1) * 2 * Cout)
                self._gemm(M=B * (rows + 1), N=2 * Cout, Cin=Cc, x=y, w=W[f"{d}.conv_tr.w"], bias=W[f"{d}.conv_tr.b"], out=full,
                           taps=((0, 0), (0, -1)), I1=1, I0=rows + 1, J1=1, J0=rows, xs=(rows * Cc, 0, Cc, 1),
                           os_=((rows + 1) * 2 * Cout, 0, 2 * Cout))
                nxt = self._buf(key, f"dx{j}", B * T * Cout)
                self._gn(key, full, nxt, f"{d}.norm2", B, 2 * rows + 2, Cout, _lib.ACT_GELU, row0=1, rows_out=T,
                         addend=nxt_skip, tag=f"_d{j}b")
                _tap(taps, f"dec{j}", (nxt - nxt_skip).view(B, T, Cout), "t")
                xd = nxt
                continue
            if l["norm"]:
                # index 4: 3x3 rewrite on a single bin = k=3 over time; transposed conv to 8 bins = one GEMM; no crop
                rw = self._buf(key, f"drw{j}", B * T * 2 * Cc)
                self._gemm(M=B * T, N=2 * Cc, Cin=Cc, x=xd, w=W[f"{d}.rewrite.w"], bias=W[f"{d}.rewrite.b"], out=rw,
                           taps=((0, -1), (0, 0), (0, 1)), I1=1, I0=T, J1=1, J0=T, xs=(T * Cc, 0, Cc, 1),
                           os_=(T * 2 * Cc, 0, 2 * Cc))
                pre = self._buf(key, f"dy{j}", B * T * Cc)
                self._gn(key, rw, pre, f"{d}.norm1", B, T, 2 * Cc, _lib.ACT_GLU, tag=f"_d{j}a")
                full = self._buf(key, f"dfull{j}", B * T * 8 * Cout)
                self._gemm(M=B * T, N=8 * Cout, Cin=Cc, x=pre, w=W[f"{d}.conv_tr.w"], bias=W[f"{d}.conv_tr.b"], out=full)
                nxt = self._buf(key, f"dx{j}", B * T * 8 * Cout)
                self._gn(key, full, nxt, f"{d}.norm2", B, T * 8, Cout, _lib.ACT_GELU, addend=nxt_skip, tag=f"_d{j}b")
                _tap(taps, f"dec{j}", (nxt - nxt_skip).view(B, T, 8, Cout), "f")
                xd, Fcur = nxt, 8
                # time branch leaves the merged one here: conv_tr of `pre` only (empty layer), GroupNorm, crop, GELU
                td = f"tdecoder.{j - (cfg.depth - n_time)}"
                Ct, Tt = l["dec_out"], tl[n_time - 1]
                fullt = self._buf(key, "tfull", B * (T + 1) * 4 * Ct)
                self._gemm(M=B * (T + 1), N=4 * Ct, Cin=Cc, x=pre, w=W[f"{td}.conv_tr.w"], bias=W[f"{td}.conv_tr.b"], out=fullt,
                           taps=((0, 0), (0, -1)), I1=1, I0=T + 1, J1=1, J0=T, xs=(T * Cc, 0, Cc, 1),
                           os_=((T + 1) * 4 * Ct, 0, 4 * Ct))
                xtd = self._buf(key, "tdx0", B * _pitch(Tt) * Ct, zero=True)
                skip_t = saved_t[n_time - 2]
                self._gn(key, fullt, xtd, f"{td}.norm2", B, 4 * T + 4, Ct, _lib.ACT_GELU, row0=2, rows_out=Tt, addend=skip_t,
                         y_item_stride=_pitch(Tt) * Ct, tag="_td0")
                _tap(taps, "tdec0", (xtd - skip_t).view(B, _pitch(Tt), Ct)[:, :Tt], "t")
                continue
            # ---- index 3..0: the HTDemucs decoder layers without DConv ------------------------------------------------
            nxt = self._buf(key, f"dx{j}", B * T * 4 * Fcur * Cout)
            self._freq_decoder(key, j, xd, f"dy{j}", nxt, nxt_skip, taps, B, T, Fcur, Cc, Cout)
            xd, Fcur = nxt, 4 * Fcur
            jt = j - (cfg.depth - n_time)                      # 1..4
            Ct_in, Ct = l["chout"], l["dec_out"]
            Tin, Tout = tl[n_time - jt], tl[n_time - 1 - jt]
            skip_t = None if last else saved_t[n_time - 2 - jt]
            nxt_t = self._buf(key, f"tdx{jt}", B * _pitch(Tout) * Ct, zero=True)
            self._time_decoder(key, jt, xtd, f"dyt{jt}", nxt_t, skip_t, taps, B, Tin, Tout, Ct_in, Ct)
            xtd = nxt_t

        # ---- K2: de-normalise, iSTFT + overlap-add, crop, add the time branch (hdemucs.py:775-793) -----------------
        return self._istft(xd, xtd, norm, out_buf, B, T, L, L)
