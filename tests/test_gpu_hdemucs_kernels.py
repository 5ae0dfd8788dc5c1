"""The kernels only Hybrid Demucs v3 runs (csrc/hdemucs.cu) against a float64 statement of the same operations, arm by
arm, at the hdemucs_mmi shapes and at the edges of every dispatch decision.

The BLSTM and LocalState sit inside the DConv residual branch, behind LayerScale, so whole-model parity sees an error in
them scaled down by the LayerScale factor; the numpy emulator (tests/abi_emulator.py) restates the header in float32 and
shares any misreading of it.  Here every kernel is compared on its own output with float64:
- bd_lstm_bidir: the persistent kernel with 64 units per block (H <= 192) and with 32 (H <= 427), several batch chunks
  per call with a one-item last chunk, the step-per-launch kernel (H > 427, or BD_LSTM_STEPWISE set), per direction;
- bd_local_state: the tiled kernel (keys and content staged in shared memory) and the streaming one, up to the limits of
  both, with saturated decays, large scores and a masked diagonal that is the row maximum;
- bd_gn_stats (on the raw sums and on the finalised mean / rstd) and bd_gn_act, bd_lstm_frame / bd_lstm_unframe_add
  (bitwise);
- HDemucsEngine._blstm / _local_state / _dconv at the layer-4 and layer-5 geometries of hdemucs_mmi, on the increment
  of h or x.
The float64 statements are pinned on the CPU to nn.LSTM, F.group_norm, the oracle and the numpy emulator.  Which arm a
case reaches follows from the header's arithmetic (lstm_plan, local_state_arm); test_dispatch_matches_plan checks that
arithmetic against the kernels a profiler sees, test_case_coverage that the cases reach every arm.

Largest error per arm over the cases below, measured on one B200 (1000 W power limit); the bounds are about 3x these.
LSTM: largest per-direction rel-L2 and largest |error| of h (|h| < 1); the others: rel-L2 unless stated.
    lstm persistent<64>        1.1e-7, |dh| 2.2e-7 (one launch, or several with a last chunk of 1 or 4 items)
    lstm persistent<32>        1.2e-7, |dh| 3.3e-7 (H = 427 in three launches, the last of one item)
    lstm step-per-launch       1.3e-7, |dh| 2.9e-7 (H = 1024); BD_LSTM_STEPWISE at the persistent shapes 1.2e-7, 2.2e-7
    lstm gate regimes          6.3e-7, |dh| 1.2e-5 on each kernel: the forget-gate bias +6 lets the float32 cell state
                               build up over 200 steps; saturated gates alone stay at the plain level
    local_state                tiled 2.4e-7, streaming 2.5e-7; saturated decays 1.5e-7; scores x8 2.1e-6; masked
                               diagonal as the row maximum 1.8e-5 (scores near -100 carry float32 rounding of ~6e-6)
    gn_stats                   double sums 6.7e-16; (mean, rstd) 3.9e-8, with a common offset of 8x the spread 4.0e-7
                               (the float32 rounding of a mean 8 spreads from zero, measured in spreads)
    gn_act                     6.6e-8
    lstm_frame / unframe_add   bitwise
    Engine._blstm              fp32 6.0e-7, strict 4.4e-6
    Engine._local_state        fp32 5.4e-7, strict 6.1e-6
    Engine._dconv              fp32 1.6e-6, strict 1.2e-5 (two depth steps, BLSTM and LocalState on)
"""
import json
import math
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

from _fixtures import rel_l2
from demucs_b200 import _lib
from demucs_b200._lib import KernelError, ptr
from oracle import hdemucs_oracle as oracle
from test_gpu_dconv import ref_finalize, stat_err

DEV = "cuda:0"
F64 = torch.float64
GUARD, SENTINEL = 64, 1234.5                      # floats behind an output that no kernel may touch
B200_SMS = 148
LSTM_TOL = {"rel": 4e-7, "abs": 1e-6}             # per-direction rel-L2, largest |dh|
LSTM_REGIME_TOL = {"rel": 2e-6, "abs": 4e-5}
LS_TOL = {"plain": 8e-7, "decay_sat": 8e-7, "scores_x8": 6e-6, "diag_max": 5e-5}
GN_TOL = {"sums": 2e-15, "stats": 1.2e-6, "act": 2e-7}
ENGINE_TOL = {"fp32": {"blstm": 2e-6, "local_state": 2e-6, "dconv": 5e-6},
              "strict": {"blstm": 1.5e-5, "local_state": 2e-5, "dconv": 3.5e-5}}


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else B200_SMS


# ---------------------------------------------------------------------------------------------------------------------
# dispatch arithmetic of csrc/hdemucs.cu
def lstm_plan(H, N, sms):
    """(arm, items per launch) of bd_lstm_bidir: the persistent kernel when one block's slice of W_hh and its hidden
    vectors fit in 227 KB and the grid of one batch tile fits on the device, in chunks of per_chunk * NB items."""
    UB = 64 if H <= 192 else 32
    NB = 256 // UB
    smem = (H * 4 * UB + NB * H) * 4
    per_chunk = sms // (2 * -(-H // UB))
    if smem > 227 * 1024 or per_chunk < 1:
        return "step", [N]
    cap = per_chunk * NB
    return f"persistent{UB}", [min(cap, N - n0) for n0 in range(0, N, cap)]


def items_per_launch(H, sms):
    return lstm_plan(H, 1 << 20, sms)[1][0]


def local_state_arm(T, dh):
    if (2 * T * (dh + 1) + 8 * (T + dh)) * 4 <= 200 * 1024:
        return "tiled"
    return "stream" if 4 * (T + dh) * 4 <= 48 * 1024 else "error"


def tiled_max_T(dh):
    return (200 * 1024 // 4 - 8 * dh) // (2 * (dh + 1) + 8)


# ---------------------------------------------------------------------------------------------------------------------
# float64 statements of the header's operations (include/demucs_b200.h)
def ref_lstm_bidir(pre, whhT):
    """out [N, T, 2, H] of bd_lstm_bidir: pre [N, T, 2, 4H] = x W_ih^T + b_ih + b_hh, whhT [2, H, 4H], zero initial
    state, direction 1 runs from t = T - 1 down.  oracle.lstm_direction with an identity input projection."""
    N, T, _, H4 = pre.shape
    eye = torch.eye(H4, dtype=pre.dtype, device=pre.device)
    zero = pre.new_zeros(H4)
    outs = [oracle.lstm_direction(pre[:, :, d].transpose(0, 1), eye, whhT[d].t(), zero, zero, reverse=bool(d))
            for d in range(2)]
    return torch.stack(outs, 2).transpose(0, 1)                          # [N, T, 2, H]


def ref_local_state_core(qkc, dq, heads, dots_out=None):
    """out [N, T, D] of bd_local_state: per head, dots[t, s] = k_t . q_s / sqrt(dh) - |t - s| sum_f (f + 1) / 2 *
    sigmoid(dq[s, h*4 + f]) / 2, dots[s, s] = -100, softmax over keys t, content summed with those weights."""
    N, T, D3 = qkc.shape
    D = D3 // 3
    dh = D // heads
    v = qkc.to(F64).view(N, T, 3, heads, dh)
    q, k, c = v[:, :, 0], v[:, :, 1], v[:, :, 2]
    dots = torch.einsum("nthc,nshc->nhts", k, q) / math.sqrt(dh)
    dec = torch.sigmoid(dq.to(F64).view(N, T, heads, 4)) / 2                                 # [n, s, h, f]
    slope = (dec * torch.arange(1, 5, dtype=F64, device=qkc.device)).sum(-1) / math.sqrt(4)  # [n, s, h]
    idx = torch.arange(T, dtype=F64, device=qkc.device)
    dots = dots - (idx[:, None] - idx[None, :]).abs() * slope.permute(0, 2, 1)[:, :, None, :]
    dots = dots.masked_fill(torch.eye(T, dtype=torch.bool, device=qkc.device), -100.0)
    if dots_out is not None:
        dots_out.append(dots)
    w = torch.softmax(dots, dim=2)
    return torch.einsum("nhts,nthc->nshc", w, c).reshape(N, T, D)


def ref_gn_sums(x, G):
    """[B * G, 2] = (sum, sum of squares) of each (item, group) of x [B, rows, C]."""
    B, rows, C = x.shape
    v = x.to(F64).view(B, rows, G, C // G)
    return torch.stack([v.sum((1, 3)), (v * v).sum((1, 3))], -1).reshape(B * G, 2)


def ref_gn_act(x, mr, gamma, beta, G, act, row0=0, rows_out=None, addend=None):
    """act(GroupNorm_G(x))[:, row0:row0 + rows_out] (+ addend) with the statistics mr [B * G, 2] of all rows; GLU keeps
    value c and gate c + C / 2."""
    B, rows, C = x.shape
    rows_out = rows - row0 if rows_out is None else rows_out
    m = mr.to(F64).view(B, G, 1, 2).repeat_interleave(C // G, 1).view(B, 1, C, 2)
    v = (x.to(F64)[:, row0:row0 + rows_out] - m[..., 0]) * m[..., 1] * gamma.to(F64) + beta.to(F64)
    if act == _lib.ACT_GELU:
        v = F.gelu(v)
    elif act == _lib.ACT_GLU:
        v = v[..., :C // 2] * torch.sigmoid(v[..., C // 2:])
    return v if addend is None else v + addend.to(F64)


def ref_frame(x, nf, width, stride):
    """frames [B * nf, width, C]: frame k of item b holds x[b, k * stride + j], zero past the end (utils.unfold)."""
    B, T, C = x.shape
    xp = F.pad(x, (0, 0, 0, (nf - 1) * stride + width - T))
    return torch.stack([xp[:, k * stride:k * stride + width] for k in range(nf)], 1).reshape(B * nf, width, C)


def ref_unframe(frames, B, T, nf, width, stride):
    """[B, T, C]: frame 0 without its last `limit` steps, middle frames without `limit` at both ends, the last without
    its first `limit`, concatenated and cut to T (demucs.py:52-64, oracle.blstm)."""
    fr = frames.view(B, nf, width, -1)
    limit = stride // 2
    parts = [fr[:, k, (limit if k else 0):(width if k == nf - 1 else width - limit)] for k in range(nf)]
    return torch.cat(parts, 1)[:, :T]


# ---------------------------------------------------------------------------------------------------------------------
# 1. the float64 statements themselves (CPU)
@pytest.mark.parametrize("N,T,H", [(3, 7, 5), (2, 1, 8), (4, 12, 16)])
def test_lstm_statement_matches_nn_lstm(N, T, H):
    """ref_lstm_bidir on the header's operands (biases folded into pre, W_hh transposed) equals a bidirectional
    nn.LSTM in float64 loaded with the same weights."""
    torch.manual_seed(N * 100 + T)
    lstm = torch.nn.LSTM(6, H, bidirectional=True, batch_first=True, dtype=F64)
    x = torch.randn(N, T, 6, dtype=F64)
    with torch.no_grad():
        want, _ = lstm(x)
        pre = torch.stack([x @ getattr(lstm, f"weight_ih_l0{s}").t() + getattr(lstm, f"bias_ih_l0{s}") +
                           getattr(lstm, f"bias_hh_l0{s}") for s in ("", "_reverse")], 2)
        whhT = torch.stack([getattr(lstm, f"weight_hh_l0{s}").t() for s in ("", "_reverse")], 0)
        got = ref_lstm_bidir(pre, whhT).reshape(N, T, 2 * H)
    assert (got - want).abs().max() < 1e-13


def test_lstm_statement_matches_emulator():
    """The same statement against the numpy emulator's bd_lstm_bidir (float32): the operand layouts agree."""
    import abi_emulator as E
    g = torch.Generator().manual_seed(5)
    N, T, H = 3, 9, 12
    pre = torch.randn(N, T, 2, 4 * H, generator=g)
    whhT = (torch.rand(2, H, 4 * H, generator=g) * 2 - 1) / H ** 0.5
    out = torch.zeros(N, T, 2 * H)
    ws = torch.zeros(6 * N * H)
    E.bd_lstm_bidir(pre.data_ptr(), whhT.data_ptr(), out.data_ptr(), ws.data_ptr(), N, T, H, 0)
    want = ref_lstm_bidir(pre.double(), whhT.double()).reshape(N, T, 2 * H)
    assert rel_l2(out, want) < 1e-6


def _local_state_weights(D, g, heads=4):
    W = {}
    for n, co in (("query", D), ("key", D), ("content", D), ("query_decay", heads * 4), ("proj", D)):
        W[f"ls.{n}.weight"] = torch.randn(co, D, 1, generator=g, dtype=F64) / D ** 0.5
        W[f"ls.{n}.bias"] = 0.3 * torch.randn(co, generator=g, dtype=F64)
    return W


@pytest.mark.parametrize("heads,D,T", [(4, 16, 13), (4, 48, 40), (1, 8, 9), (8, 32, 21)])
def test_local_state_statement_matches_oracle(heads, D, T):
    """x + proj(core(qkc, dq)) with the projections in the kernel's channels-last layout (qkc = query | key | content,
    dq in h * 4 + f order) equals oracle.local_state(x)."""
    g = torch.Generator().manual_seed(heads * 100 + D)
    B = 2
    W = _local_state_weights(D, g, heads)
    x = torch.randn(B, D, T, generator=g, dtype=F64)
    xt = x.transpose(1, 2)                                                # [B, T, D]
    lin = lambda n: xt @ W[f"ls.{n}.weight"][:, :, 0].t() + W[f"ls.{n}.bias"]   # noqa: E731
    qkc = torch.cat([lin("query"), lin("key"), lin("content")], -1)
    core = ref_local_state_core(qkc, lin("query_decay"), heads)
    got = xt + core @ W["ls.proj.weight"][:, :, 0].t() + W["ls.proj.bias"]
    want = oracle.local_state(x, W, "ls", heads=heads).transpose(1, 2)
    assert (got - xt).abs().max() > 0.1
    assert (got - want).abs().max() < 1e-12


@pytest.mark.parametrize("act", [_lib.ACT_NONE, _lib.ACT_GELU, _lib.ACT_GLU])
def test_gn_statement_matches_group_norm(act):
    """ref_gn_sums + ref_finalize + ref_gn_act (crop, addend) equal F.group_norm followed by the activation."""
    g = torch.Generator().manual_seed(act)
    B, rows, C, G = 3, 29, 32, 4
    x = torch.randn(B, rows, C, generator=g, dtype=F64) * 2 + 5
    gam, bet = torch.randn(C, generator=g, dtype=F64), torch.randn(C, generator=g, dtype=F64)
    mr = ref_finalize(ref_gn_sums(x, G), rows * C // G)
    Co = C // 2 if act == _lib.ACT_GLU else C
    add = torch.randn(B, 20, Co, generator=g, dtype=F64)
    got = ref_gn_act(x, mr, gam, bet, G, act, row0=4, rows_out=20, addend=add)
    y = F.group_norm(x.transpose(1, 2), G, gam, bet, 1e-5)
    y = {_lib.ACT_NONE: y, _lib.ACT_GELU: F.gelu(y), _lib.ACT_GLU: F.glu(y, dim=1)}[act]
    want = y.transpose(1, 2)[:, 4:24] + add
    assert (got - want).abs().max() < 1e-12


@pytest.mark.parametrize("T", [150, 336, 401])
def test_frame_statement_matches_oracle_blstm(T):
    """ref_frame, the oracle's per-frame two-layer BLSTM and linear, then ref_unframe + the skip, equal oracle.blstm:
    nframes, the zero padding of the last frame and the kept ranges (limit = stride / 2) are the reference's."""
    g = torch.Generator().manual_seed(T)
    B, C = 2, 6
    W = {}
    for layer, cin in ((0, C), (1, 2 * C)):
        for s in ("", "_reverse"):
            W[f"b.lstm.weight_ih_l{layer}{s}"] = torch.randn(4 * C, cin, generator=g, dtype=F64) / cin ** 0.5
            W[f"b.lstm.weight_hh_l{layer}{s}"] = torch.randn(4 * C, C, generator=g, dtype=F64) / C ** 0.5
            W[f"b.lstm.bias_ih_l{layer}{s}"] = 0.1 * torch.randn(4 * C, generator=g, dtype=F64)
            W[f"b.lstm.bias_hh_l{layer}{s}"] = 0.1 * torch.randn(4 * C, generator=g, dtype=F64)
    W["b.linear.weight"] = torch.randn(C, 2 * C, generator=g, dtype=F64) / (2 * C) ** 0.5
    W["b.linear.bias"] = 0.1 * torch.randn(C, generator=g, dtype=F64)
    x = torch.randn(B, C, T, generator=g, dtype=F64)
    want = oracle.blstm(x, W, "b")
    width, stride = 200, 100
    framed = T > width
    nf = math.ceil(T / stride) if framed else 1
    seq = ref_frame(x.transpose(1, 2), nf, width, stride) if framed else x.transpose(1, 2)       # [N, Tt, C]
    s = seq.transpose(0, 1)
    names = ("weight_ih", "weight_hh", "bias_ih", "bias_hh")
    for layer in range(2):
        s = torch.cat([oracle.lstm_direction(s, *(W[f"b.lstm.{n}_l{layer}{sf}"] for n in names), reverse=bool(sf))
                       for sf in ("", "_reverse")], -1)
    y = (s @ W["b.linear.weight"].t() + W["b.linear.bias"]).transpose(0, 1)
    got = (ref_unframe(y, B, T, nf, width, stride) if framed else y) + x.transpose(1, 2)
    assert (got - want.transpose(1, 2)).abs().max() < 1e-12


# ---------------------------------------------------------------------------------------------------------------------
# cases, by the arm the header's arithmetic sends them to
def _lstm_cases():
    cases = {}
    for H in (16, 48, 100, 192):                      # 64 units per block, 4 items; 100: ragged last unit block
        for T in (1, 2, 200):
            cases[f"p64_H{H}_T{T}"] = (H, 7, T)
    for H in (200, 384, 427):                         # 32 units per block, 8 items; 427: the largest H that fits
        for T in (1, 2, 200):
            cases[f"p32_H{H}_T{T}"] = (H, 11, T)
    cases["mmi_l4_H192"] = (192, 64, 200)             # hdemucs_mmi, 16 items x 4 frames of 200 steps
    cases["mmi_l5_H384"] = (384, 16, 168)
    # several launches per call: only these reach the persistent kernel's `step > 0` guard, which keeps the hidden
    # state the previous chunk left in the ping-pong buffer out of the next chunk's first step
    cases["chunks_H384_N49"] = (384, 49, 168)         # 48 items per launch with 148 SMs
    cases["chunks_H192_N100"] = (192, 100, 200)       # 96 items per launch with 148 SMs
    cases["chunks_H192_last1"] = (192, ("chunks", 1, 1), 200)
    cases["chunks_H48_last1_T2"] = (48, ("chunks", 1, 1), 2)
    cases["chunks_H427_last1"] = (427, ("chunks", 2, 1), 200)
    for H in (428, 512, 1024):                        # one block's W_hh slice exceeds 227 KB: step per launch
        for T in (1, 2, 200):
            cases[f"step_H{H}_T{T}"] = (H, 5, T)
    return cases


LSTM_CASES = _lstm_cases()
STEPWISE_CASES = {k: LSTM_CASES[k] for k in ("p64_H16_T200", "p64_H100_T200", "p64_H192_T2", "p32_H200_T200",
                                              "p32_H427_T200", "p32_H427_T1", "mmi_l4_H192", "chunks_H192_last1")}


def resolve_n(H, N, sms):
    if isinstance(N, tuple):
        _, k, r = N
        return k * items_per_launch(H, sms) + r
    return N


# LocalState: (N, T, D, heads, regime)
LS_CASES = {}
for _dh in (16, 48, 96):
    for _T in (1, 2, 31, 33, 168, 336):
        LS_CASES[f"T{_T}_dh{_dh}"] = (2, _T, 4 * _dh, 4, "plain")
    _tm = tiled_max_T(_dh)
    LS_CASES[f"tiled_max_dh{_dh}"] = (1, _tm, 4 * _dh, 4, "plain")
    LS_CASES[f"stream_min_dh{_dh}"] = (1, _tm + 1, 4 * _dh, 4, "plain")
    LS_CASES[f"stream_max_dh{_dh}"] = (1, 3072 - _dh, 4 * _dh, 4, "plain")
for _T, _arm in ((336, "tiled"), (600, "stream")):
    for _reg in ("scores_x8", "decay_sat", "diag_max"):
        LS_CASES[f"{_reg}_{_arm}"] = (2, _T, 192, 4, _reg)
LS_CASES["heads1_tiled"] = (2, 168, 48, 1, "plain")
LS_CASES["heads8_tiled"] = (2, 168, 384, 8, "plain")
LS_CASES["heads1_stream"] = (1, 700, 48, 1, "plain")
LS_CASES["heads8_stream"] = (1, 600, 384, 8, "plain")


def test_case_coverage():
    """With this device's SM count (148 without one), the cases reach both persistent templates, the step-per-launch
    kernel, several-chunk launches whose last chunk holds one item (in both templates), and both LocalState arms up to
    their limits."""
    sms = sm_count()
    plans = {k: lstm_plan(H, resolve_n(H, N, sms), sms) for k, (H, N, T) in LSTM_CASES.items()}
    arms = {a for a, _ in plans.values()}
    assert arms == {"persistent64", "persistent32", "step"}
    assert all(plans[k][0] == "step" for k in LSTM_CASES if k.startswith("step_"))
    assert plans["p32_H427_T200"][0] == "persistent32" and lstm_plan(428, 11, sms)[0] == "step"
    last1 = {a for a, n in plans.values() if len(n) > 1 and n[-1] == 1}
    assert last1 == {"persistent64", "persistent32"}
    assert all(len(plans[k][1]) > 1 for k in LSTM_CASES if k.startswith("chunks_"))
    assert all(lstm_plan(H, resolve_n(H, N, sms), sms)[0].startswith("persistent")
               for H, N, T in STEPWISE_CASES.values())
    ls = {k: local_state_arm(T, D // h) for k, (n, T, D, h, r) in LS_CASES.items()}
    assert set(ls.values()) == {"tiled", "stream"}
    for dh in (16, 48, 96):
        assert ls[f"tiled_max_dh{dh}"] == "tiled" and ls[f"stream_min_dh{dh}"] == "stream"
        assert local_state_arm(3073 - dh, dh) == "error"
    assert (tiled_max_T(16), tiled_max_T(48), tiled_max_T(96)) == (1216, 479, 249)
    assert ls["T336_dh48"] == ls["T168_dh96"] == "tiled" and ls["T336_dh96"] == "stream"
    for reg in ("scores_x8", "decay_sat", "diag_max"):
        assert ls[f"{reg}_tiled"] == "tiled" and ls[f"{reg}_stream"] == "stream"


# ---------------------------------------------------------------------------------------------------------------------
# 2. bd_lstm_bidir
def lstm_operands(N, T, H, seed, regime="plain", device=DEV):
    g = torch.Generator().manual_seed(seed)
    pre = torch.randn(N, T, 2, 4 * H, generator=g)
    if regime == "saturate":                          # pre-activations up to |30|: expf saturates in every gate
        pre = (torch.rand(N, T, 2, 4 * H, generator=g) * 2 - 1) * 30
    elif regime == "forget":                          # forget gate ~ sigmoid(6): the cell state carries over 200 steps
        pre[..., H:2 * H] += 6.0
    whhT = (torch.rand(2, H, 4 * H, generator=g) * 2 - 1) / H ** 0.5   # nn.LSTM's initialisation range
    return pre.to(device), whhT.to(device)


def run_lstm(pre, whhT, N, T, H, ws=None):
    """bd_lstm_bidir into a guarded output; a fresh workspace is filled with garbage (the call must clear it)."""
    n_out = N * T * 2 * H
    out = torch.full((n_out + GUARD,), SENTINEL, device=pre.device)
    if ws is None:
        ws = torch.full((6 * N * H + GUARD,), SENTINEL, device=pre.device)
    _lib.call("bd_lstm_bidir", ptr(pre), ptr(whhT), ptr(out), ptr(ws), N, T, H, 0)
    torch.cuda.synchronize()
    assert torch.all(out[n_out:] == SENTINEL), "floats behind out were written"
    return out[:n_out].view(N, T, 2, H)


def lstm_errors(out, ref):
    """(largest per-direction rel-L2, largest |error|, description of the worst (item, step) row per direction)."""
    err = out.double() - ref
    rels, worst = [], []
    for d in range(2):
        rels.append(float(err[:, :, d].norm() / ref[:, :, d].norm().clamp_min(1e-30)))
        row = err[:, :, d].abs().amax(-1)                                 # [N, T]
        i = int(row.argmax())
        n, t = divmod(i, row.shape[1])
        first = 0 if d == 0 else row.shape[1] - 1                         # the step each direction starts on
        worst.append(f"dir{d} rel {rels[-1]:.2e} worst (n={n}, t={t}) {float(row[n, t]):.2e}, first step "
                     f"{float(row[:, first].max()):.2e}, last step {float(row[:, row.shape[1] - 1 - first].max()):.2e}")
    return max(rels), float(err.abs().max()), "; ".join(worst)


def check_lstm(label, H, N, T, regime="plain", seed=0):
    pre, whhT = lstm_operands(N, T, H, seed, regime)
    out = run_lstm(pre, whhT, N, T, H)
    rel, mx, desc = lstm_errors(out, ref_lstm_bidir(pre.double(), whhT.double()))
    arm, chunks = lstm_plan(H, N, sm_count())
    print(f"lstm {label} H={H} N={N} T={T} {arm} launches {chunks}: rel-L2 {rel:.2e}, max |dh| {mx:.2e} | {desc}")
    return rel, mx


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(LSTM_CASES))
def test_lstm_bidir(case):
    H, N, T = LSTM_CASES[case]
    N = resolve_n(H, N, sm_count())
    rel, mx = check_lstm(case, H, N, T, seed=len(case) * 31 + T)
    assert rel <= LSTM_TOL["rel"] and mx <= LSTM_TOL["abs"]


@pytest.mark.gpu
@pytest.mark.parametrize("regime", ["saturate", "forget"])
@pytest.mark.parametrize("H,N", [(192, 7), (384, 11), (512, 5)])
def test_lstm_bidir_gate_regimes(H, N, regime):
    """Saturated gates (|pre| up to 30) and a forget-gate bias of +6, so that the cell state builds up over 200 steps
    in float32, on each of the three kernels."""
    rel, mx = check_lstm(f"{regime}", H, N, 200, regime, seed=H + N)
    assert rel <= LSTM_REGIME_TOL["rel"] and mx <= LSTM_REGIME_TOL["abs"]


@pytest.mark.gpu
@pytest.mark.parametrize("H", [192, 384])
def test_lstm_bidir_workspace_reuse(H):
    """The engine keeps one workspace per layer: a second call on it gives the same bits, a call with fewer items after
    one with more (several chunks) is still right, and nothing behind the workspace or the output is written."""
    sms = sm_count()
    T = 200
    N1 = items_per_launch(H, sms) + 3
    N2 = 5
    ws = torch.full((6 * N1 * H + GUARD,), SENTINEL, device=DEV)
    pre, whhT = lstm_operands(N1, T, H, 40 + H)
    a = run_lstm(pre, whhT, N1, T, H, ws)
    b = run_lstm(pre, whhT, N1, T, H, ws)
    assert torch.equal(a, b), "a second call on the same workspace differs"
    pre2, whhT2 = lstm_operands(N2, T, H, 41 + H)
    c = run_lstm(pre2, whhT2, N2, T, H, ws)
    assert torch.all(ws[6 * N1 * H:] == SENTINEL), "floats behind the workspace were written"
    rel1, mx1, _ = lstm_errors(a, ref_lstm_bidir(pre.double(), whhT.double()))
    rel2, mx2, _ = lstm_errors(c, ref_lstm_bidir(pre2.double(), whhT2.double()))
    print(f"lstm workspace reuse H={H}: N={N1} rel {rel1:.2e} max {mx1:.2e}; then N={N2} rel {rel2:.2e} max {mx2:.2e}")
    assert max(rel1, rel2) <= LSTM_TOL["rel"] and max(mx1, mx2) <= LSTM_TOL["abs"]


def _kernel_counts(fn):
    """{kernel name: launches} of the device work of fn(), from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    counts = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            counts[e.name] = counts.get(e.name, 0) + 1
    return counts


def _launches(counts, kernel):
    return sum(v for k, v in counts.items() if kernel in k)


def _stepwise_child():
    """Run in a process with BD_LSTM_STEPWISE set: the persistent shapes through the step-per-launch kernel.  One JSON
    line per case on stdout."""
    sms = sm_count()
    for case, (H, N, T) in STEPWISE_CASES.items():
        N = resolve_n(H, N, sms)
        pre, whhT = lstm_operands(N, T, H, len(case) * 31 + T)
        box = {}
        counts = _kernel_counts(lambda: box.setdefault("out", run_lstm(pre, whhT, N, T, H)))
        rel, mx, desc = lstm_errors(box["out"], ref_lstm_bidir(pre.double(), whhT.double()))
        print(json.dumps(dict(case=case, H=H, N=N, T=T, rel=rel, max=mx, desc=desc,
                              step=_launches(counts, "lstm_step_kernel"),
                              persistent=_launches(counts, "lstm_persistent_kernel"))), flush=True)


@pytest.mark.gpu
def test_lstm_bidir_stepwise_env():
    """BD_LSTM_STEPWISE is read once per process, so the step-per-launch kernel at the shapes the persistent one takes
    runs in a child process; the parent waits for it and checks its results."""
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, BD_LSTM_STEPWISE="1",
               PYTHONPATH=os.pathsep.join([os.path.dirname(here), here] + [os.environ.get("PYTHONPATH", "")]))
    py = [sys.executable] + (["-s"] if sys.flags.no_user_site else [])
    res = subprocess.run(py + ["-c", "import test_gpu_hdemucs_kernels as m; m._stepwise_child()"], cwd=here, env=env,
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-4000:]
    rows = [json.loads(line) for line in res.stdout.splitlines() if line.startswith("{")]
    assert [r["case"] for r in rows] == list(STEPWISE_CASES)
    for r in rows:
        print(f"lstm stepwise-env {r['case']} H={r['H']} N={r['N']} T={r['T']}: {r['step']} step launches, rel-L2 "
              f"{r['rel']:.2e}, max |dh| {r['max']:.2e} | {r['desc']}")
        assert r["step"] == r["T"] and r["persistent"] == 0
        assert r["rel"] <= LSTM_TOL["rel"] and r["max"] <= LSTM_TOL["abs"]


# ---------------------------------------------------------------------------------------------------------------------
# 3. bd_local_state
def ls_operands(N, T, D, heads, regime, seed):
    g = torch.Generator().manual_seed(seed)
    dh = D // heads
    qkc = torch.randn(N, T, 3 * D, generator=g)
    dq = torch.randn(N, T, heads * 4, generator=g) - 2          # the reference initialises the decay bias at -2
    if regime == "scores_x8":                                   # scores in the tens: the max subtraction matters
        qkc[..., :2 * D] *= 8
    elif regime == "decay_sat":                                 # sigmoid(+-20): saturated decay weights
        dq = 20 * torch.sign(torch.randn(N, T, heads * 4, generator=g))
    elif regime == "diag_max":
        # k_t . q_s / sqrt(dh) = kappa_t ~ -98 and the strongest decay (2.5 per step): every off-diagonal score is below
        # -100 in most rows, so the masked diagonal is the row maximum while its neighbours still carry weight
        qkc[..., :D] = 1.0
        kappa = -98.0 + 0.3 * torch.randn(N, T, 1, generator=g)
        qkc[..., D:2 * D] = kappa / dh ** 0.5
        dq = torch.full((N, T, heads * 4), 20.0)
    return qkc.to(DEV), dq.to(DEV)


def run_local_state(qkc, dq, N, T, D, heads):
    n_out = N * T * D
    out = torch.full((n_out + GUARD,), SENTINEL, device=DEV)
    _lib.call("bd_local_state", ptr(qkc), ptr(dq), ptr(out), N, T, D, heads, 0)
    torch.cuda.synchronize()
    assert torch.all(out[n_out:] == SENTINEL), "floats behind out were written"
    return out[:n_out].view(N, T, D)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(LS_CASES))
def test_local_state(case):
    N, T, D, heads, regime = LS_CASES[case]
    qkc, dq = ls_operands(N, T, D, heads, regime, seed=len(case) + T)
    out = run_local_state(qkc, dq, N, T, D, heads)
    dots = []
    ref = ref_local_state_core(qkc, dq, heads, dots)
    e = rel_l2(out.cpu(), ref.cpu())
    arm = local_state_arm(T, D // heads)
    extra = ""
    if regime == "diag_max":
        diag_is_max = dots[0].argmax(2) == torch.arange(T, device=DEV)          # [n, h, s]
        share = float(diag_is_max.double().mean())
        extra = f", masked diagonal is the row maximum in {share:.0%} of rows"
        assert share > 0.8
        del diag_is_max
    del dots
    print(f"local_state {case} N={N} T={T} D={D} heads={heads} {arm}: rel-L2 {e:.2e}{extra}")
    assert e <= LS_TOL[regime]


@pytest.mark.gpu
@pytest.mark.parametrize("dh", [16, 48, 96])
def test_local_state_too_long(dh):
    """One step beyond the streaming kernel's 48 KB of score rows the call is refused before any launch."""
    T = 3073 - dh
    qkc = torch.zeros(1, T, 12 * dh, device=DEV)
    dq = torch.zeros(1, T, 16, device=DEV)
    out = torch.full((T * 4 * dh,), SENTINEL, device=DEV)
    with pytest.raises(KernelError, match="too long"):
        _lib.call("bd_local_state", ptr(qkc), ptr(dq), ptr(out), 1, T, 4 * dh, 4, 0)
    torch.cuda.synchronize()
    assert torch.all(out == SENTINEL)


@pytest.mark.gpu
def test_dispatch_matches_plan():
    """The kernels a profiler sees at the arm boundaries are the ones lstm_plan and local_state_arm predict, launch
    counts included (one persistent launch per chunk, one step launch per time step)."""
    sms = sm_count()
    checks = []
    for H, N, T in ((192, resolve_n(192, ("chunks", 1, 1), sms), 3), (193, 9, 3), (427, 9, 2), (428, 9, 4), (16, 3, 1)):
        pre, whhT = lstm_operands(N, T, H, H)
        counts = _kernel_counts(lambda: run_lstm(pre, whhT, N, T, H))
        arm, chunks = lstm_plan(H, N, sms)
        seen = {"persistent64": _launches(counts, "lstm_persistent_kernel<64>"),
                "persistent32": _launches(counts, "lstm_persistent_kernel<32>"),
                "step": _launches(counts, "lstm_step_kernel")}
        want = {a: 0 for a in seen}
        want[arm] = T if arm == "step" else len(chunks)
        checks.append((f"lstm H={H} N={N} T={T}", seen, want))
    for dh in (16, 48, 96):
        for T in (tiled_max_T(dh), tiled_max_T(dh) + 1):
            qkc, dq = ls_operands(1, T, 4 * dh, 4, "plain", T)
            counts = _kernel_counts(lambda: run_local_state(qkc, dq, 1, T, 4 * dh, 4))
            seen = {"tiled": _launches(counts, "local_state_tiled_kernel"),
                    "stream": _launches(counts, "local_state_kernel")}
            want = {"tiled": 0, "stream": 0}
            want[local_state_arm(T, dh)] = 1
            checks.append((f"local_state T={T} dh={dh}", seen, want))
    for label, seen, want in checks:
        print(f"dispatch {label}: {seen}")
    assert all(seen == want for _, seen, want in checks), [(lbl, s, w) for lbl, s, w in checks if s != w]


# ---------------------------------------------------------------------------------------------------------------------
# 4. GroupNorm(G), frame / unframe
@pytest.mark.gpu
@pytest.mark.parametrize("B,rows,C,offset", [(2, 4000, 768, 8.0), (3, 338, 384, 8.0), (2, 2688, 1536, 0.0),
                                             (1, 7, 16, 8.0)])
def test_gn_stats(B, rows, C, offset):
    """rows * C / G above 64 * 2048 (the capped grid loops) and a common offset of 8x the spread per group, so that
    E[x^2] - E[x]^2 cancels ~65-fold in the finalize step.  Checked on the double sums and on (mean, rstd)."""
    G = 4
    g = torch.Generator().manual_seed(rows + C)
    spread = 0.5 + torch.rand(B, 1, G, 1, generator=g)
    sign = torch.sign(torch.randn(B, 1, G, 1, generator=g))
    x = (torch.randn(B, rows, G, C // G, generator=g) + offset * sign) * spread
    x = x.reshape(B, rows, C).to(DEV)
    sums = torch.zeros(B * G, 2, dtype=F64, device=DEV)
    _lib.call("bd_gn_stats", ptr(x), ptr(sums), B, rows, C, G, 0)
    want = ref_gn_sums(x, G)
    es = float(((sums - want).abs() / want.abs()).max())
    mr = torch.full((B * G, 2), float("nan"), device=DEV)
    _lib.call("bd_finalize_group_stats", ptr(sums), ptr(mr), B * G, float(rows * (C // G)), 0)
    torch.cuda.synchronize()
    ref = ref_finalize(want, rows * (C // G))
    em = stat_err(mr, ref)
    cancel = float((want[:, 1] / (rows * C // G) / (1 / ref[:, 1] ** 2)).max())
    print(f"gn_stats B={B} rows={rows} C={C} offset {offset}: sums {es:.2e}, (mean, rstd) {em:.2e}, "
          f"E[x^2] / var {cancel:.0f}")
    assert es <= GN_TOL["sums"] and em <= GN_TOL["stats"]


GN_ACT_GEO = {   # B, rows_in, row0, rows_out, C, y item pitch in rows (> rows_out: a gap between items)
    "crop_gap": (3, 338, 1, 336, 384, 340),           # decoder.0 of hdemucs_mmi: full transposed conv, crop, GELU
    "crop_td0": (2, 1348, 2, 1343, 96, 1344),         # the time branch's conv_tr of layer 4, cropped, padded pitch
    "whole": (2, 168, 0, 168, 3072, 168),             # an encoder's norm2 + GLU over 2C channels
}


@pytest.mark.gpu
@pytest.mark.parametrize("addend", [False, True])
@pytest.mark.parametrize("act", [_lib.ACT_NONE, _lib.ACT_GELU, _lib.ACT_GLU])
@pytest.mark.parametrize("geo", list(GN_ACT_GEO))
def test_gn_act(geo, act, addend):
    B, rows_in, row0, rows_out, C, pitch = GN_ACT_GEO[geo]
    G = 4
    Co = C // 2 if act == _lib.ACT_GLU else C
    g = torch.Generator().manual_seed(rows_in + act)
    x = (torch.randn(B, rows_in, C, generator=g) * 1.5 + 0.7).to(DEV)
    mr = ref_finalize(ref_gn_sums(x, G), rows_in * (C // G)).float()
    gam, bet = (1 + 0.3 * torch.randn(C, generator=g)).to(DEV), (0.2 * torch.randn(C, generator=g)).to(DEV)
    stride = pitch * Co
    add = torch.randn(B * stride, generator=g).to(DEV) if addend else None
    y = torch.full((B * stride + GUARD,), SENTINEL, device=DEV)
    _lib.call("bd_gn_act", ptr(x), ptr(y), ptr(mr), ptr(gam), ptr(bet), ptr(add), B, rows_in, row0, rows_out, C, G, act,
              stride, 0)
    torch.cuda.synchronize()
    yi = y[:B * stride].view(B, stride)
    assert torch.all(yi[:, rows_out * Co:] == SENTINEL) and torch.all(y[B * stride:] == SENTINEL), "gap written"
    a = add.view(B, stride)[:, :rows_out * Co].view(B, rows_out, Co) if addend else None
    want = ref_gn_act(x, mr, gam, bet, G, act, row0, rows_out, a)
    e = rel_l2(yi[:, :rows_out * Co].cpu(), want.cpu())
    print(f"gn_act {geo} act={act} addend={addend}: rel-L2 {e:.2e}")
    assert e <= GN_TOL["act"]


@pytest.mark.gpu
@pytest.mark.parametrize("T", [201, 250, 300, 336, 399, 400, 401])
def test_lstm_frame_unframe(T):
    """Bitwise: framing is a copy, un-framing one float addition.  The frames handed to unframe are random (frames of
    the input would agree wherever they overlap and hide a shifted limit), and it runs in place (skip = out) as
    HDemucsEngine._blstm calls it."""
    B, C, width, stride = 3, 192, 200, 100
    nf = math.ceil(T / stride)
    g = torch.Generator().manual_seed(T)
    x = torch.randn(B, T, C, generator=g).to(DEV)
    n_fr = B * nf * width * C
    fr = torch.full((n_fr + GUARD,), SENTINEL, device=DEV)
    _lib.call("bd_lstm_frame", ptr(x), ptr(fr), B, T, C, nf, width, stride, 0)
    torch.cuda.synchronize()
    assert torch.all(fr[n_fr:] == SENTINEL)
    assert torch.equal(fr[:n_fr].view(B * nf, width, C), ref_frame(x, nf, width, stride))
    frames = torch.randn(B * nf, width, C, generator=g).to(DEV)
    h = torch.full((B * T * C + GUARD,), SENTINEL, device=DEV)
    h[:B * T * C] = x.reshape(-1)
    _lib.call("bd_lstm_unframe_add", ptr(frames), ptr(h), ptr(h), B, T, C, nf, width, stride, 0)
    torch.cuda.synchronize()
    assert torch.all(h[B * T * C:] == SENTINEL)
    assert torch.equal(h[:B * T * C].view(B, T, C), ref_unframe(frames, B, T, nf, width, stride) + x)


# ---------------------------------------------------------------------------------------------------------------------
# 5. HDemucsEngine at the layer-4 and layer-5 geometries of hdemucs_mmi, against the oracle in float64
ENGINE_LAYERS = [("encoder.4", 768, 336), ("encoder.5", 1536, 168)]     # prefix, C, T (7.8 s segment)
ENGINE_B = [1, 4]


@pytest.fixture(scope="module")
def mmi():
    """(cfg, state, {mode: engine}, float64 weights of the two layers on the CPU, oracle cache)."""
    from demucs_b200 import hdemucs as HD
    from demucs_b200.hdemucs_engine import HDemucsEngine
    cfg = HD.hdemucs_mmi_config()
    state = HD.init_weights(cfg, 7, layer_scale=1.0)
    engines = {m: HDemucsEngine(cfg, state, DEV, mode=m) for m in ENGINE_TOL}
    W = {k: v.double() for k, v in state.items() if k.startswith(("encoder.4.dconv", "encoder.5.dconv"))}
    return cfg, engines, W, {}


def _oracle_increment(mmi, op, prefix, C, T, B):
    cfg, _, W, cache = mmi
    key = (op, prefix, B)
    if key not in cache:
        hid = C // cfg.dconv_comp
        g = torch.Generator().manual_seed(C + T + B)
        x = torch.randn(B, T, C if op == "dconv" else hid, generator=g)
        y = x.double().transpose(1, 2)
        p = f"{prefix}.dconv.layers.0"
        with torch.no_grad():
            if op == "blstm":
                out = oracle.blstm(y, W, f"{p}.3")
            elif op == "local_state":
                out = oracle.local_state(y, W, f"{p}.4")
            else:
                out = oracle.dconv(y, W, f"{prefix}.dconv", cfg.dconv_depth, True, True)
        cache[key] = (x, (out - y).transpose(1, 2).contiguous())
    return cache[key]


@pytest.mark.gpu
@pytest.mark.parametrize("op", ["blstm", "local_state", "dconv"])
@pytest.mark.parametrize("mode", list(ENGINE_TOL))
@pytest.mark.parametrize("B", ENGINE_B)
def test_engine_layers(B, mode, op, mmi):
    """_blstm / _local_state on h, _dconv (BLSTM and LocalState both on) on x, each called twice on one buffer key so
    that the cached buffers and the LSTM workspace are reused; compared on the increment, which LayerScale and the skip
    would otherwise hide.  LayerScale 1."""
    cfg, engines, _, _ = mmi
    eng = engines[mode]
    for prefix, C, T in ENGINE_LAYERS:
        hid = C // cfg.dconv_comp
        x, inc_ref = _oracle_increment(mmi, op, prefix, C, T, B)
        x = x.to(DEV)
        for rep in range(2):
            xo = x.clone()
            key = ("hdemucs-kernel-test", B, op)
            p = f"{prefix}.dconv.layers.0"
            if op == "blstm":
                eng._blstm(key, p, xo, B, T, hid, "_t")
            elif op == "local_state":
                eng._local_state(key, p, xo, B, T, hid, "_t")
            else:
                eng._dconv(key, prefix, xo, B, T, 1, C, "_t", lstm=True, attn=True)
            torch.cuda.synchronize()
            e = rel_l2((xo - x).cpu(), inc_ref)
            print(f"Engine.{op} mode={mode} {prefix} C={C} T={T} B={B} call {rep}: increment rel-L2 {e:.2e}")
            assert e <= ENGINE_TOL[mode][op]
