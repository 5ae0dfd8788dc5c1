"""The fused attention kernels (K6) against a float64 statement of the same operation, arm by arm, at the tile edges
and in the softmax regimes of trained models.

Arms (keys per step TK, K / V stages NS):
- fp32          bd_attention, BD_MATH_FP32: attention_simt_kernel, 64 query rows x 64 keys, exact online softmax;
- tf32          bd_attention, BD_MATH_TF32: attention_tc_kernel<false> + V transpose, TK 128, NS 3;
- tf32x3        bd_attention, BD_MATH_TF32X3: attention_tc_kernel<true> + split / transpose pre-pass, TK 64, NS 2;
- bf16x3        bd_attention, BD_MATH_BF16X3 (strict mode): attention_b16_kernel<true,false> + split, TK 128, NS 2;
- bf16          bd_attention, BD_MATH_BF16: attention_b16_kernel<false,false> + bf16 conversion, TK 128, NS 4;
- bf16_tensors  bd_attention_bf16 (bf16 mode): attention_b16_kernel<false,true>, bf16 in and out, TK 128, NS 4.
The tensor-core arms deal key tiles alternately to two softmax groups (group g owns tiles j = g, g + 2, ...).  A
group keeps its running maximum until a tile's maximum exceeds it by more than 8 (log2 units); only then, after its
first tile, does it rescale its O accumulator in tensor memory, and the two groups are merged at the end.
Random-normal q / k never reach that rescale (test_case_coverage counts it on the inputs of test_attention: zero times;
the largest rise is 5.8), so the regimes below are built from q and k directly: coordinate 0 of every head carries a
per-row scale in q and a per-key pattern in k, on top of noise that moves a logit by about 0.25 (natural units):
    plain       random normal q, k, v
    rising      every tile of a group has a maximum more than 12 above the group's previous one: O is rescaled at every
                tile after the first
    mixed       the rising pattern on rows 0-15 of every 32-row quarter, flat logits on rows 16-31: within one warp some
                lanes raise and the others keep corr = 1
    needle_*    one key 100 above the rest (144 in log2 units), in the partial last tile, in a tile of group 0 only
                or of group 1 only: the other group's merge weight underflows to 0
    just_below  every later tile's maximum about 7.4 above the maximum of its group's first tile: P reaches ~2^7.4
                under a stale maximum and nothing is rescaled
    negative    every logit near -30: a zero key past Tk or a zero query row that escaped its mask would have logit 0
                and dominate the row
    uniform     q = 0: the output is the mean of V over exactly Tk keys
    large       logits of standard deviation ~20
The shapes give, for TK = 64 and 128, 1 to 7 key tiles each with a full and with a partial last tile, a group 1
without tiles, a group that owns only the partial tile, and more tiles than twice each arm's stage ring;
test_case_coverage checks all of it from the inputs.

Every call runs on a workspace filled with NaN (a read of workspace the pre-pass did not write turns into NaN even where
P = 0) with a NaN guard behind it, into an output with sentinel guard rows behind the last item; padded variants put NaN
into the gaps of strided q / k / v and write o with ldo > D.  Nothing outside o[b, r < Tq, c < D] may change.

Errors: whole-tensor rel-L2 and the largest per-row rel-L2 over every (item, head, query row) of 64 outputs (a wrong
128-row tail tile is diluted ~18-fold in the whole-tensor figure of a 2 x 8 x 2688 output).  The bf16 arms are also
compared against the statement on q / k / v rounded to bf16 (RN, as split_rows_b16_kernel rounds and as the bf16
tensors arrive), which isolates the softmax and accumulation error; in the large regime the single-pass tf32 arm is
judged against the statement on q / k / v truncated to tf32 (the tensor core reads the top 19 bits of an fp32 operand).

Largest error per arm and regime (whole-tensor rel-L2 / largest per-row rel-L2) over the cases, the padded cases
counted as negative, measured on one B200 (1000 W power limit); the bounds in TOL and BIG_ROW_TOL are about 3x these
(2.5x to 5x, at least 1e-7).  "vs tf32" / "vs bf16": against the operand-rounded statement; test_attn*: the
transformer shapes of test_attention and test_attention_bf16_tensors.  The single-pass arms' large-regime figures
against the unrounded statement (tf32 1.8e-3 / 2.0e-2, bf16 1.3e-2 / 1.5e-1) are the operand rounding of logits with a
spread of 20 and are reported, not judged.
                fp32           tf32           tf32 vs tf32   tf32x3
    plain       6.8e-7/1.5e-6  1.7e-3/3.7e-3  -              4.4e-6/7.2e-6
    rising      7.6e-6/1.3e-5  8.2e-4/1.0e-3  -              7.4e-6/1.3e-5
    mixed       7.8e-6/1.5e-5  8.3e-4/1.1e-3  -              7.4e-6/1.3e-5
    needle      0/0            7.1e-4/9.7e-4  -              8.0e-8/1.2e-7
    just_below  1.2e-6/1.8e-6  8.1e-4/9.8e-4  -              3.1e-6/3.8e-6
    negative    4.7e-6/8.1e-6  8.5e-4/1.1e-3  -              5.5e-6/7.6e-6
    uniform     4.9e-7/5.6e-7  4.3e-4/4.6e-4  -              1.1e-6/1.2e-6
    large       2.0e-6/3.0e-5  1.8e-3/2.0e-2  3.6e-4/9.6e-4  2.2e-6/2.7e-5
    test_attn*  9.8e-7/2.1e-6  1.7e-3/4.3e-3  -              9.7e-6/1.7e-5
                bf16x3         bf16           bf16 vs bf16   bf16_tensors (vs bf16)
    plain       8.1e-6/1.9e-5  3.6e-3/8.9e-3  2.0e-3/3.3e-3  2.7e-3/3.8e-3
    rising      7.2e-6/1.3e-5  2.4e-3/3.4e-3  1.6e-3/2.3e-3  2.3e-3/3.4e-3
    mixed       7.3e-6/1.2e-5  2.4e-3/3.5e-3  1.6e-3/2.5e-3  2.3e-3/3.3e-3
    needle      2.7e-6/3.4e-6  1.8e-3/2.1e-3  3.1e-6/5.3e-6  0/0
    just_below  4.9e-6/7.8e-6  2.5e-3/3.6e-3  1.8e-3/2.7e-3  2.4e-3/3.4e-3
    negative    5.9e-6/8.6e-6  2.4e-3/3.6e-3  1.6e-3/2.6e-3  2.4e-3/3.2e-3
    uniform     2.7e-6/3.3e-6  2.0e-3/2.2e-3  4.5e-8/5.4e-8  1.8e-3/2.1e-3
    large       2.6e-5/3.8e-4  1.3e-2/1.5e-1  6.7e-4/3.9e-3  1.5e-3/4.8e-3
    test_attn*  8.0e-6/2.0e-5  3.5e-3/9.0e-3  -              2.3e-3/3.9e-3
The needle outputs are v of the needle key: exact on the fp32 arm and on bf16 tensors, P = 1 and every other P = 0.

bd_attention on the fp32 arm used to accept q / k / v / o pointers that are not 16-byte aligned and then read and write
them as float4; it now refuses them on the host like the tensor-core arms (test_loud_errors).
"""
import functools
import math

import pytest
import torch
import torch.nn.functional as F

from demucs_b200 import _lib
from demucs_b200._lib import KernelError

DEV = "cuda:0"
F64 = torch.float64
HD = 64
SL2 = 0.125 * math.log2(math.e)             # logit scale of the kernels' exp2 domain
LAZY = 8.0                                  # the running maximum is raised when a tile's exceeds it by more than this
UNDERFLOW = 126.0                           # ex2.approx.ftz of anything below -126 is 0
GUARD_ROWS, WS_GUARD, SENTINEL = 3, 64, 1234.5

ARMS = {   # math mode (None: bd_attention_bf16), keys per step, K / V stages (None: no ring)
    "fp32": (_lib.MATH_FP32, 64, None),
    "tf32": (_lib.MATH_TF32, 128, 3),
    "tf32x3": (_lib.MATH_TF32X3, 64, 2),
    "bf16x3": (_lib.MATH_BF16X3, 128, 2),
    "bf16": (_lib.MATH_BF16, 128, 4),
    "bf16_tensors": (None, 128, 4),
}
ARM_OF_MATH = {m: a for a, (m, _, _) in ARMS.items() if m is not None}

# (whole-tensor rel-L2, largest per-row rel-L2) per arm, reference and regime (the three needle placements share one
# entry).  "f64": the statement on the operands as passed; "bf16" / "tf32": on the operands rounded as the arm reads
# them.  None: reported, not judged.
TOL = {
    "fp32": {
        "f64": {"plain": (2e-6, 5e-6), "rising": (2e-5, 4e-5), "mixed": (2e-5, 5e-5), "needle": (1e-7, 1e-7),
                "just_below": (4e-6, 5e-6), "negative": (2e-5, 3e-5), "uniform": (2e-6, 2e-6), "large": (6e-6, 9e-5)},
    },
    "tf32": {
        "f64": {"plain": (5e-3, 1e-2), "rising": (3e-3, 3e-3), "mixed": (3e-3, 3e-3), "needle": (2e-3, 3e-3),
                "just_below": (3e-3, 3e-3), "negative": (3e-3, 3e-3), "uniform": (2e-3, 2e-3), "large": None},
        "tf32": {"large": (1e-3, 3e-3)},
    },
    "tf32x3": {
        "f64": {"plain": (2e-5, 2e-5), "rising": (2e-5, 4e-5), "mixed": (2e-5, 4e-5), "needle": (2e-7, 4e-7),
                "just_below": (9e-6, 1e-5), "negative": (2e-5, 2e-5), "uniform": (3e-6, 4e-6), "large": (6e-6, 8e-5)},
    },
    "bf16x3": {
        "f64": {"plain": (3e-5, 6e-5), "rising": (2e-5, 4e-5), "mixed": (2e-5, 4e-5), "needle": (8e-6, 1e-5),
                "just_below": (2e-5, 2e-5), "negative": (2e-5, 3e-5), "uniform": (8e-6, 1e-5), "large": (8e-5, 1e-3)},
    },
    "bf16": {
        "f64": {"plain": (1e-2, 3e-2), "rising": (7e-3, 1e-2), "mixed": (7e-3, 1e-2), "needle": (5e-3, 6e-3),
                "just_below": (7e-3, 1e-2), "negative": (7e-3, 1e-2), "uniform": (6e-3, 7e-3), "large": None},
        "bf16": {"plain": (6e-3, 1e-2), "rising": (5e-3, 7e-3), "mixed": (5e-3, 7e-3), "needle": (9e-6, 2e-5),
                 "just_below": (5e-3, 8e-3), "negative": (5e-3, 8e-3), "uniform": (2e-7, 2e-7), "large": (2e-3, 1e-2)},
    },
    "bf16_tensors": {
        "bf16": {"plain": (8e-3, 1e-2), "rising": (7e-3, 1e-2), "mixed": (7e-3, 1e-2), "needle": (1e-7, 1e-7),
                 "just_below": (7e-3, 1e-2), "negative": (7e-3, 1e-2), "uniform": (6e-3, 6e-3), "large": (5e-3, 2e-2)},
    },
}
# per-row bound of the transformer shapes, whose whole-tensor bounds test_attention takes as parameters
BIG_ROW_TOL = {"fp32": 6e-6, "tf32": 2e-2, "tf32x3": 5e-5, "bf16x3": 6e-5, "bf16": 3e-2, "bf16_tensors": 1e-2}


# ---------------------------------------------------------------------------------------------------------------------
# the float64 statement
def ref_attention(q, k, v, device=DEV):
    """softmax(Q_h K_h^T / 8) V_h with head h on columns [64h, 64h + 64), in float64, one (item, head) at a time."""
    B, Tq, D = q.shape
    q, k, v = (t.to(device, F64) for t in (q, k, v))
    out = torch.empty(B, Tq, D, dtype=F64, device=device)
    for b in range(B):
        for h in range(D // HD):
            c = slice(h * HD, (h + 1) * HD)
            out[b, :, c] = torch.softmax(q[b, :, c] @ k[b, :, c].t() / 8.0, dim=-1) @ v[b, :, c]
    return out


def bf16_rounded(x):
    return x.to(torch.bfloat16).float()


def tf32_truncated(x):
    return (x.float().contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


@pytest.mark.parametrize("B,H,Tq,Tk", [(2, 3, 17, 29), (1, 8, 5, 1), (3, 1, 40, 40)])
def test_statement_matches_mha(B, H, Tq, Tk):
    """ref_attention equals nn.MultiheadAttention's forward in float64 with identity in / out projections: the 1/8 scale
    and the head column layout are the reference's."""
    g = torch.Generator().manual_seed(B * 100 + Tq)
    D = HD * H
    q, k, v = (3 * torch.randn(B, T, D, generator=g, dtype=F64) for T in (Tq, Tk, Tk))
    eye, zero = torch.eye(D, dtype=F64), torch.zeros(D, dtype=F64)
    want, _ = F.multi_head_attention_forward(q.transpose(0, 1), k.transpose(0, 1), v.transpose(0, 1), D, H,
                                             torch.cat([eye, eye, eye]), torch.cat([zero, zero, zero]), None, None,
                                             False, 0.0, eye, zero, training=False, need_weights=False)
    got = ref_attention(q, k, v, device="cpu")
    assert (got - want.transpose(0, 1)).abs().max() < 1e-12


# ---------------------------------------------------------------------------------------------------------------------
# inputs
def old_inputs(B, H, Tq, Tk, seed=0):
    """The random-normal (q, k, v) of test_attention: one packed [B, T, 3D] draw when Tq == Tk, else q and packed kv."""
    g = torch.Generator().manual_seed(seed)
    D = HD * H
    if Tq == Tk:
        qkv = torch.randn(B, Tq, 3 * D, generator=g)
        return qkv[..., :D], qkv[..., D:2 * D], qkv[..., 2 * D:]
    q = torch.randn(B, Tq, D, generator=g)
    kv = torch.randn(B, Tk, 2 * D, generator=g)
    return q, kv[..., :D], kv[..., D:]


def ntiles(Tk, TK):
    return -(-Tk // TK)


def needle_key(regime, Tk, TK):
    nt = ntiles(Tk, TK)
    if regime == "needle_last":
        return Tk - 1
    j = (2 if nt >= 3 else 0) if regime == "needle_g0" else (3 if nt >= 4 else 1)
    return min(j * TK + 17, Tk - 1)


@functools.lru_cache(maxsize=8)
def regime_inputs(B, H, Tq, Tk, regime, TK, seed):
    """(q [B, Tq, D], k, v [B, Tk, D]) float32 on the CPU.  The structured regimes set coordinate 0 of every head:
    q = A (per row), k = c (per key), so that logit = A c / 8 + noise; A and c are exact in bf16 and tf32."""
    g = torch.Generator().manual_seed(seed)
    D = HD * H
    v = torch.randn(B, Tk, D, generator=g)
    if regime == "plain":
        return torch.randn(B, Tq, D, generator=g), torch.randn(B, Tk, D, generator=g), v
    if regime == "large":
        return 4.5 * torch.randn(B, Tq, D, generator=g), 4.5 * torch.randn(B, Tk, D, generator=g), v
    if regime == "uniform":
        return torch.zeros(B, Tq, D), torch.randn(B, Tk, D, generator=g), v
    q = torch.randn(B, Tq, D, generator=g)
    k = (0.05 if regime == "just_below" else 0.25) * torch.randn(B, Tk, D, generator=g)
    r, t = torch.arange(Tq), torch.arange(Tk)
    i = (t // TK) // 2                                          # index of the key's tile within its group
    u = torch.where(t % TK == 0, 0.0, -0.5 * ((t * 7 + 3) % 5).float())   # 0 on every tile's first key
    A = torch.full((Tq,), 8.0)
    if regime in ("rising", "mixed"):
        A = 8.0 + (r % 4).float()
        if regime == "mixed":
            A = torch.where(r % 32 < 16, A, torch.zeros(()))
        c = 10.0 * i + u
    elif regime == "just_below":
        c = torch.where(i > 0, 5.125, 0.0) + u
    elif regime == "negative":
        c = -30.0 - 0.25 * ((t * 7 + 3) % 9).float()
    elif regime.startswith("needle"):
        c = torch.zeros(Tk)
        c[needle_key(regime, Tk, TK)] = 100.0
    else:
        raise ValueError(regime)
    q[..., ::HD] = A[None, :, None]
    k[..., ::HD] = c[None, :, None]
    return q, k, v


def _cases():
    cases = {}
    tks = (1, 63, 64, 65, 127, 128, 129, 191, 192, 193, 255, 256, 257, 320, 330, 384, 385, 448, 449, 512, 513, 640,
           700, 768, 800, 896, 897, 1153)
    tqs = (1, 31, 33, 63, 64, 65, 127, 128, 129, 257, 300)
    for n, Tk in enumerate(tks):
        for j in range(2):
            Tq = tqs[(3 * n + 5 * j) % len(tqs)]
            B, H = (1, 3)[(n + j) % 2], (1, 3, 8)[(n + 2 * j) % 3]
            cases[f"plain_B{B}H{H}_{Tq}x{Tk}"] = (B, H, Tq, Tk, "cross", "plain")
    for B, H, T in ((1, 1, 1), (3, 1, 64), (1, 3, 129), (3, 8, 300), (2, 3, 513), (1, 8, 897)):
        cases[f"plain_self_B{B}H{H}_{T}"] = (B, H, T, T, "self", "plain")
    for regime in ("negative", "uniform"):
        for B, H, Tq, Tk in ((1, 1, 1, 1), (3, 3, 33, 65), (2, 1, 129, 129), (3, 3, 65, 193), (1, 8, 300, 257),
                             (2, 3, 128, 897), (2, 1, 129, 449)):
            cases[f"{regime}_B{B}H{H}_{Tq}x{Tk}"] = (B, H, Tq, Tk, "cross", regime)
        cases[f"{regime}_self_B3H3_385"] = (3, 3, 385, 385, "self", regime)
    for regime in ("rising", "mixed", "just_below", "large"):
        cases[f"{regime}_B2H3_129x449"] = (2, 3, 129, 449, "cross", regime)
        cases[f"{regime}_B1H8_300x897"] = (1, 8, 300, 897, "cross", regime)
        cases[f"{regime}_self_B3H1_385"] = (3, 1, 385, 385, "self", regime)
    for regime in ("needle_last", "needle_g0", "needle_g1"):
        cases[f"{regime}_B2H3_129x449"] = (2, 3, 129, 449, "cross", regime)
        cases[f"{regime}_B1H8_300x897"] = (1, 8, 300, 897, "cross", regime)
        cases[f"{regime}_self_B2H1_385"] = (2, 1, 385, 385, "self", regime)
    cases["large_self_B1H8_2688"] = (1, 8, 2688, 2688, "self", "large")
    return cases


CASES = _cases()


# ---------------------------------------------------------------------------------------------------------------------
# the census: what the tensor-core softmax does with each case's inputs, restated on float64 logits
def lazy_census(q, k, TK):
    """Walk the lazy rescale of one call at key tile TK in float64 (log2 units) and count what it does:
    tiles (per group), raised (row, later tile) pairs and the smallest rise among them, the largest rise that stays
    at or below the threshold, 32-row quarters where some valid lanes raise and others do not, the largest gap between
    the two groups' final maxima (the merge weight of the lower group is 2^-gap) and the largest logit."""
    B, Tq, D = q.shape
    Tk = k.shape[1]
    nt = ntiles(Tk, TK)
    res = dict(tiles=(len(range(0, nt, 2)), len(range(1, nt, 2))), raised=0, later=0, rise_min=math.inf,
               below=-math.inf, mixed=0, gap=0.0, smax=-math.inf)
    q64, k64 = q.double(), k.double()
    for b in range(B):
        for h in range(D // HD):
            c = slice(h * HD, (h + 1) * HD)
            s = (q64[b, :, c] @ k64[b, :, c].t()) * SL2                                  # [Tq, Tk]
            res["smax"] = max(res["smax"], float(s.max()))
            tmax = F.pad(s, (0, nt * TK - Tk), value=-math.inf).view(Tq, nt, TK).amax(-1)
            final = []
            for g in (0, 1):
                js = list(range(g, nt, 2))
                if not js:
                    continue
                m = tmax[:, js[0]].clone()
                for j in js[1:]:
                    rise = tmax[:, j] - m
                    up = rise > LAZY
                    res["later"] += Tq
                    res["raised"] += int(up.sum())
                    if up.any():
                        res["rise_min"] = min(res["rise_min"], float(rise[up].min()))
                    if (~up).any():
                        res["below"] = max(res["below"], float(rise[~up].max()))
                    for r0 in range(0, Tq, 32):
                        blk = up[r0:r0 + 32]
                        res["mixed"] += int(bool(blk.any()) and not bool(blk.all()))
                    m = torch.where(up, tmax[:, j], m)
                final.append(m)
            if len(final) == 2:
                res["gap"] = max(res["gap"], float((final[0] - final[1]).abs().max()))
    return res


@functools.lru_cache(maxsize=None)
def case_census(case, TK):
    B, H, Tq, Tk, layout, regime = CASES[case]
    q, k, _ = regime_inputs(B, H, Tq, Tk, regime, TK, seed_of(case))
    return lazy_census(q, k, TK)


def seed_of(case):
    return sum(map(ord, case))


def test_case_coverage():
    """The cases reach every tile edge and every softmax path they exist for, at both tensor-core tile widths, and the
    random-normal inputs of test_attention never reach the rescale."""
    report = []
    for TK in (64, 128):
        shapes = {(ntiles(Tk, TK), Tk % TK != 0) for B, H, Tq, Tk, lay, reg in CASES.values()}
        assert {(n, p) for n in range(1, 8) for p in (False, True)} <= shapes, TK
        assert (2, True) in shapes                                  # group 1 owns only the partial last tile
        for arm, (_, tk, ns) in ARMS.items():
            if tk == TK and ns:
                assert max(ntiles(Tk, TK) for _, _, _, Tk, _, _ in CASES.values()) > 2 * ns, arm
        for case, (B, H, Tq, Tk, layout, regime) in CASES.items():
            if regime in ("plain", "uniform", "large"):
                continue
            c = case_census(case, TK)
            report.append(f"TK={TK} {case}: tiles/group {c['tiles']}, raised {c['raised']}/{c['later']} later "
                          f"(row, tile) pairs, smallest raising rise {c['rise_min']:.1f}, largest rise below "
                          f"{c['below']:.2f}, mixed quarters {c['mixed']}, merge gap {c['gap']:.0f}, "
                          f"largest logit {c['smax']:.1f}")
            nt = ntiles(Tk, TK)
            if regime == "rising":
                assert min(c["tiles"]) >= 2 and c["raised"] == c["later"] and c["rise_min"] > 12.0, case
            elif regime == "mixed":
                assert min(c["tiles"]) >= 2 and c["mixed"] > 0 and c["rise_min"] > 12.0, case
                assert 0.4 < c["raised"] / c["later"] < 0.6, case
            elif regime == "just_below":
                assert min(c["tiles"]) >= 2 and c["raised"] == 0 and 7.0 < c["below"] < 7.8, case
            elif regime == "negative":
                assert c["smax"] < -40.0, case
            elif regime.startswith("needle"):
                j = needle_key(regime, Tk, TK) // TK
                want = {"needle_last": (nt - 1, Tk % TK != 0), "needle_g0": (j, j % 2 == 0),
                        "needle_g1": (j, j % 2 == 1)}[regime]
                assert j == want[0] and want[1] and c["gap"] > UNDERFLOW, case
    for B, H, Tq, Tk in SHAPES:
        q, k, _ = old_inputs(B, H, Tq, Tk)
        for TK in (64, 128):
            c = lazy_census(q, k, TK)
            report.append(f"TK={TK} random normal B{B} H{H} {Tq}x{Tk}: raised {c['raised']}, largest rise "
                          f"{c['below']:.2f}")
            assert c["raised"] == 0 and c["below"] < LAZY
    print("\n".join(report))


# ---------------------------------------------------------------------------------------------------------------------
# calls
def pack(q, k, v, layout, pad, dtype):
    """Device buffers as the engine lays them out (self: one [B, T, 3D] projection, cross: q [B, Tq, D] and packed kv
    [B, Tk, 2D]), each row `pad` elements longer than needed with NaN in the gap.  (buffers, pointers, leading dims)"""
    B, Tq, D = q.shape
    Tk = k.shape[1]
    es = 2 if dtype == torch.bfloat16 else 4
    if layout == "self":
        assert Tq == Tk
        buf = torch.full((B, Tq, 3 * D + pad), float("nan"), dtype=dtype, device=DEV)
        buf[..., :3 * D] = torch.cat([q, k, v], -1).to(DEV, dtype)
        p = buf.data_ptr()
        return [buf], (p, p + es * D, p + es * 2 * D), (3 * D + pad,) * 3
    qb = torch.full((B, Tq, D + pad), float("nan"), dtype=dtype, device=DEV)
    qb[..., :D] = q.to(DEV, dtype)
    kv = torch.full((B, Tk, 2 * D + pad), float("nan"), dtype=dtype, device=DEV)
    kv[..., :2 * D] = torch.cat([k, v], -1).to(DEV, dtype)
    return [qb, kv], (qb.data_ptr(), kv.data_ptr(), kv.data_ptr() + es * D), (D + pad, 2 * D + pad, 2 * D + pad)


def launch(arm, ptrs, lds, o_ptr, ldo, B, H, Tq, Tk, ws_ptr):
    math_ = ARMS[arm][0]
    if math_ is None:
        _lib.call("bd_attention_bf16", *ptrs, o_ptr, B, H, Tq, Tk, *lds, ldo, 0)
    else:
        _lib.call("bd_attention", *ptrs, o_ptr, B, H, Tq, Tk, *lds, ldo, math_, ws_ptr, 0)


def poisoned_workspace(arm, B, H, Tq, Tk):
    """(NaN-filled workspace of bd_attention_workspace floats plus a NaN guard, its size)."""
    math_ = ARMS[arm][0]
    n = 0 if math_ is None else _lib.call_value("bd_attention_workspace", B, H, Tq, Tk, math_)
    return torch.full((n + WS_GUARD,), float("nan"), device=DEV), n


def bits(t):
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32)


def run(arm, q, k, v, layout="cross", pad=0, opad=0):
    """One call of `arm` on device copies of q / k / v; returns o [B, Tq, D] as float32.  The workspace is NaN with a
    NaN guard, o lies in a sentinel-filled [B * Tq + GUARD_ROWS, D + opad] buffer: the guard, the rows behind the last
    item and the columns past D must come back bitwise unchanged, o free of NaN."""
    dtype = torch.bfloat16 if ARMS[arm][0] is None else torch.float32
    B, Tq, D = q.shape
    Tk = k.shape[1]
    keep, ptrs, lds = pack(q, k, v, layout, pad, dtype)
    ldo = D + opad
    ob = torch.full((B * Tq + GUARD_ROWS, ldo), SENTINEL, dtype=dtype, device=DEV)
    before = ob.clone()
    ws, n = poisoned_workspace(arm, B, D // HD, Tq, Tk)
    launch(arm, ptrs, lds, ob.data_ptr(), ldo, B, D // HD, Tq, Tk, ws.data_ptr())
    torch.cuda.synchronize()
    assert torch.equal(bits(ws[n:]), bits(torch.full_like(ws[n:], float("nan")))), "workspace guard written"
    assert torch.equal(bits(ob[B * Tq:]), bits(before[B * Tq:])), "rows behind the last item written"
    assert torch.equal(bits(ob[:, D:]), bits(before[:, D:])), "columns past D written"
    out = ob[:B * Tq, :D].float().view(B, Tq, D)
    assert not torch.isnan(out).any(), "NaN in the output (a read of unwritten workspace or of a padding gap)"
    return out


def errors(out, ref):
    """(whole-tensor rel-L2, largest per-row rel-L2 over (item, head, query row), where that row is)."""
    B, Tq, D = ref.shape
    d = (out.to(ref.device, F64) - ref).view(B, Tq, D // HD, HD)
    r = ref.view(B, Tq, D // HD, HD)
    whole = float(d.norm() / r.norm().clamp_min(1e-300))
    rows = d.norm(dim=-1) / r.norm(dim=-1).clamp_min(1e-300)                             # [B, Tq, H]
    i = int(rows.argmax())
    b, rest = divmod(i, Tq * (D // HD))
    t, h = divmod(rest, D // HD)
    return whole, float(rows.max()), f"(b={b}, h={h}, row={t})"


def references(arm, q, k, v, regime):
    """{name: float64 reference} the arm is compared with."""
    refs = {}
    if arm != "bf16_tensors":
        refs["f64"] = ref_attention(q, k, v)
    if arm in ("bf16", "bf16_tensors"):
        refs["bf16"] = ref_attention(bf16_rounded(q), bf16_rounded(k), bf16_rounded(v))
    if arm == "tf32" and regime == "large":
        refs["tf32"] = ref_attention(tf32_truncated(q), tf32_truncated(k), tf32_truncated(v))
    return refs


def check(arm, label, regime, out, refs, tol=None):
    """Print every comparison, then assert the judged ones; tol overrides TOL[arm][ref][regime]."""
    failed = []
    key = "needle" if regime.startswith("needle") else regime
    for name, ref in refs.items():
        whole, row, where = errors(out, ref)
        bound = tol if tol is not None else TOL[arm][name][key]
        print(f"attention {arm} {label} vs {name}: rel-L2 {whole:.2e}, worst row {row:.2e} {where}"
              + ("" if bound else " (not judged)"))
        if bound and not (whole <= bound[0] and row <= bound[1]):
            failed.append(f"{name}: rel-L2 {whole:.2e} (bound {bound[0]:.0e}), worst row {row:.2e} {where} "
                          f"(bound {bound[1]:.0e})")
    assert not failed, f"{arm} {label}: " + "; ".join(failed)


# ---------------------------------------------------------------------------------------------------------------------
# kernel against the statement
@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("arm", list(ARMS))
def test_attention_case(arm, case):
    B, H, Tq, Tk, layout, regime = CASES[case]
    q, k, v = regime_inputs(B, H, Tq, Tk, regime, ARMS[arm][1], seed_of(case))
    out = run(arm, q, k, v, layout)
    check(arm, case, regime, out, references(arm, q, k, v, regime))


@pytest.mark.gpu
@pytest.mark.parametrize("layout,B,H,Tq,Tk", [("self", 2, 3, 193, 193), ("cross", 3, 3, 129, 449),
                                              ("cross", 1, 8, 1, 65)])
@pytest.mark.parametrize("arm", list(ARMS))
def test_padded_poisoned_io(arm, layout, B, H, Tq, Tk):
    """q / k / v rows longer than D with NaN in the gaps, o written with ldo > D (a multiple of 4, of 8 for bf16) in
    front of guard rows, the negative regime (a zero read anywhere would dominate its row)."""
    bf = ARMS[arm][0] is None
    q, k, v = regime_inputs(B, H, Tq, Tk, "negative", ARMS[arm][1], B + Tq + Tk)
    out = run(arm, q, k, v, layout, pad=8 if bf else 12, opad=8 if bf else 4)
    check(arm, f"padded {layout} B{B} H{H} {Tq}x{Tk}", "negative", out, references(arm, q, k, v, "negative"))


@pytest.mark.gpu
@pytest.mark.parametrize("arm", list(ARMS))
def test_invariances(arm):
    """Bitwise: item b of a batch equals a B = 1 call at the offset pointers, head h of an H-head call equals an H = 1
    call at pointer + 64h with the same leading dims, two identical calls agree.  The CTAs are independent and the
    pre-passes elementwise, so nothing may depend on the batch, the head count or the run."""
    B, H, Tq, Tk = 3, 3, 129, 449
    dtype = torch.bfloat16 if ARMS[arm][0] is None else torch.float32
    es = 2 if dtype == torch.bfloat16 else 4
    D = HD * H
    q, k, v = regime_inputs(B, H, Tq, Tk, "rising", ARMS[arm][1], 77)
    keep, ptrs, lds = pack(q, k, v, "cross", 0, dtype)

    def call(ptrs_, o, o_off, B_, H_):
        ws, _ = poisoned_workspace(arm, B_, H_, Tq, Tk)
        launch(arm, ptrs_, lds, o.data_ptr() + es * o_off, D, B_, H_, Tq, Tk, ws.data_ptr())
        torch.cuda.synchronize()

    full = torch.zeros(B, Tq, D, dtype=dtype, device=DEV)
    call(ptrs, full, 0, B, H)
    again = torch.zeros_like(full)
    call(ptrs, again, 0, B, H)
    assert torch.equal(bits(full), bits(again)), "two identical calls differ"
    for b in range(B):
        o = torch.zeros_like(full)
        offs = (b * Tq * lds[0], b * Tk * lds[1], b * Tk * lds[2])
        call(tuple(p + es * off for p, off in zip(ptrs, offs)), o, b * Tq * D, 1, H)
        assert torch.equal(bits(o[b]), bits(full[b])), f"item {b} differs from a one-item call"
    for h in range(H):
        o = torch.zeros_like(full)
        call(tuple(p + es * HD * h for p in ptrs), o, HD * h, B, 1)
        c = slice(HD * h, HD * (h + 1))
        assert torch.equal(bits(o[..., c]), bits(full[..., c])), f"head {h} differs from a one-head call"


@pytest.mark.gpu
@pytest.mark.parametrize("arm", list(ARMS))
def test_loud_errors(arm):
    """A leading dim the vector loads cannot take, a pointer that is not 16-byte aligned and (tensor-core arms) a NULL
    workspace are refused on the host with the entry point's message, before any launch."""
    math_ = ARMS[arm][0]
    bf = math_ is None
    dtype, es, mult = (torch.bfloat16, 2, 8) if bf else (torch.float32, 4, 4)
    B, H, Tq, Tk = 1, 2, 70, 90
    D = HD * H
    buf = torch.zeros(4 * (B * max(Tq, Tk) * 3 * D + 64), dtype=dtype, device=DEV)
    o = torch.full((B * Tq * D + 64,), SENTINEL, dtype=dtype, device=DEV)
    p = buf.data_ptr()
    ws, _ = poisoned_workspace(arm, B, H, Tq, Tk)
    good = dict(ptrs=(p, p + es * D, p + es * 2 * D), lds=(3 * D,) * 3, o=o.data_ptr(), ldo=D, ws=ws.data_ptr())
    name = "bd_attention_bf16" if bf else "bd_attention"
    bad = [(dict(lds=(3 * D + mult // 2, 3 * D, 3 * D)), f"leading dims must be multiples of {mult}"),
           (dict(lds=(3 * D, 3 * D, 3 * D + mult // 2)), f"leading dims must be multiples of {mult}"),
           (dict(ldo=D + mult // 2), f"leading dims must be multiples of {mult}"),
           (dict(ptrs=(p + 8, p + es * D, p + es * 2 * D)), "unaligned tensor"),
           (dict(ptrs=(p, p + es * D + 8, p + es * 2 * D)), "unaligned tensor"),
           (dict(o=o.data_ptr() + 8), "unaligned tensor")]
    if math_ not in (None, _lib.MATH_FP32):
        bad.append((dict(ws=None), "needs a workspace"))
    for change, msg in bad:
        a = dict(good, **change)
        with pytest.raises(KernelError, match=f"{name} failed .*{msg}"):
            launch(arm, a["ptrs"], a["lds"], a["o"], a["ldo"], B, H, Tq, Tk, a["ws"])
    torch.cuda.synchronize()
    assert torch.all(o == SENTINEL)


# ---------------------------------------------------------------------------------------------------------------------
# the transformer shapes (2688 / 1344 tokens), random normal
SHAPES = [(2, 8, 2688, 2688), (2, 8, 1344, 1344), (1, 8, 2688, 1344), (1, 8, 1344, 2688), (3, 2, 100, 300),
          (2, 2, 352, 173), (1, 1, 128, 128), (1, 1, 129, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,Tq,Tk", SHAPES)
@pytest.mark.parametrize("math_mode,tol", [(_lib.MATH_FP32, 3e-6), (_lib.MATH_TF32, 2e-3),
                                           (_lib.MATH_TF32X3, 3e-5), (_lib.MATH_BF16X3, 3e-5),
                                           (_lib.MATH_BF16, 8e-3)])
def test_attention(B, H, Tq, Tk, math_mode, tol):
    arm = ARM_OF_MATH[math_mode]
    q, k, v = old_inputs(B, H, Tq, Tk)
    out = run(arm, q, k, v, "self" if Tq == Tk else "cross")
    check(arm, f"B{B} H{H} {Tq}x{Tk}", "plain", out, {"f64": ref_attention(q, k, v)}, (tol, BIG_ROW_TOL[arm]))


@pytest.mark.parametrize("B,H,Tq,Tk", [(2, 8, 2688, 2688), (1, 8, 1344, 2688), (2, 2, 352, 173), (1, 1, 129, 1)])
@pytest.mark.gpu
def test_attention_bf16_tensors(B, H, Tq, Tk):
    """bf16 q / k / v read by TMA without a conversion pass, bf16 output: against fp64 on the same bf16 inputs."""
    g = torch.Generator().manual_seed(4)
    D = HD * H
    if Tq == Tk:
        qkv = bf16_rounded(torch.randn(B, Tq, 3 * D, generator=g))
        q, k, v = qkv[..., :D], qkv[..., D:2 * D], qkv[..., 2 * D:]
    else:
        q = bf16_rounded(torch.randn(B, Tq, D, generator=g))
        kv = bf16_rounded(torch.randn(B, Tk, 2 * D, generator=g))
        q, k, v = q, kv[..., :D], kv[..., D:]
    out = run("bf16_tensors", q, k, v, "self" if Tq == Tk else "cross")
    check("bf16_tensors", f"B{B} H{H} {Tq}x{Tk}", "plain", out, {"bf16": ref_attention(q, k, v)},
          (6e-3, BIG_ROW_TOL["bf16_tensors"]))
