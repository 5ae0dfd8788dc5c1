"""The DConv expansion stage (csrc/dconv.cu) and the small normalisation kernels (csrc/norm.cu) against a float64
statement of the same operations, arm by arm.

The DConv branch reaches the stems through LayerScale (1e-3 at initialisation), so whole-model parity sees an error in
its statistics or its update about 1000x smaller than it is.  Here every arm is compared on its own output:
- bd_dconv_expand_stats: the Gram-matrix arm and the register arm, on the (mean, rstd) their sums finalise to;
- bd_dconv_expand_update: the mma.sync arms (single pass, hi/lo split) and the exact FFMA arm, on the increment of x;
- the wide-layer update as the engine issues it: bd_gn_gelu_apply + bd_conv_gemm with the GroupNorm / GLU / LayerScale
  epilogue, in place on x;
- Engine._dconv at the htdemucs encoder geometries, in every mode, against oracle.dconv;
- bd_finalize_group_stats, bd_gn_gelu_apply, bd_item_stats, bd_group_norm_apply and bd_layer_norm (fp32 output).
The float64 statement itself is checked against the oracle on the CPU (test_reference_chain_matches_oracle).

Largest error per arm over the cases below, measured on one B200 (1000 W power limit): rel-L2 of the increment of x,
or for statistics the max over slabs of |dmean| / std and |drstd| / rstd.
    expand_stats             Gram arm 3.7e-8, register arm 6.1e-8; common offset of 8x the spread 3.6e-7
    expand_update            mma single pass 4.0e-4, mma hi/lo split 1.6e-7, FFMA 1.8e-7; bd_dconv_tail 9.1e-8
    wide-layer GEMM update   TF32X3 3.8e-7, BF16X3 4.5e-6, TF32 7.9e-4, BF16 2.3e-3
    Engine._dconv            fp32 7.8e-7, tf32x3 4.7e-6, strict 7.6e-6, tf32 / bf16 9.8e-4 (two depth steps)
    norm.cu kernels          6.2e-8 or less
"""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from _fixtures import rel_l2
from demucs_b200 import _lib
from demucs_b200._lib import GemmDesc, ptr
from demucs_b200.config import htdemucs_config
from demucs_b200.engine import MODES, Engine, pack_dconv
from demucs_b200.weights import _dconv_specs, init_from_specs, init_weights
from oracle import htdemucs_oracle as oracle

DEV = "cuda:0"
F64 = torch.float64
STAT_TOL = 1e-6                                  # (mean, rstd) of a GroupNorm slab
TOL = {"mma": 1.5e-3, "mma_x3": 1e-6, "ffma": 1e-6}  # increment of x, per arm of bd_dconv_expand_update
GUARD, SENTINEL = 32, 1234.5                     # rows behind x that no kernel may touch


# ---------------------------------------------------------------------------------------------------------------------
# float64 statement of the expansion stage (include/demucs_b200.h), rows in memory order, slab map
#     slab(m) = (m / rows_per_item) * slabs_per_item + m % slabs_per_item
def slab_index(M, rpi, spi, device=None):
    m = torch.arange(M, device=device)
    return (m // rpi) * spi + m % spi


def ref_conv3(x, w1, b1, rpi, spi, dil):
    """h = b1 + sum_tap w1[:, tap] . x[row (tap - 1) * dil positions away]; the position of row m is
    (m % rpi) // spi, neighbours outside the item read zero.  x [M, C], w1 [hid, 3C] tap-major."""
    M, Cc = x.shape
    m = torch.arange(M, device=x.device)
    t, T = (m % rpi) // spi, rpi // spi
    h = b1.expand(M, -1).clone()
    for tap in range(3):
        tt = t + (tap - 1) * dil
        ok = (tt >= 0) & (tt < T)
        src = torch.where(ok, m + (tap - 1) * dil * spi, m)
        h += torch.where(ok[:, None], x[src], 0.0) @ w1[:, tap * Cc:(tap + 1) * Cc].t()
    return h


def ref_sums(v, rpi, spi, slabs):
    """[slabs, 2] = (sum, sum of squares) of the rows v [M, n] of each slab."""
    sl = slab_index(v.shape[0], rpi, spi, v.device)
    s = torch.zeros(slabs, dtype=F64, device=v.device).index_add_(0, sl, v.sum(1))
    q = torch.zeros(slabs, dtype=F64, device=v.device).index_add_(0, sl, (v * v).sum(1))
    return torch.stack([s, q], 1)


def ref_finalize(sums, count):
    """(mean, rstd) of nn.GroupNorm: biased variance, clamped at zero, eps 1e-5."""
    mean = sums[:, 0] / count
    var = (sums[:, 1] / count - mean * mean).clamp_min(0.0)
    return torch.stack([mean, 1.0 / torch.sqrt(var + 1e-5)], 1)


def ref_gn(v, mr, gamma, beta, rpi, spi):
    sl = slab_index(v.shape[0], rpi, spi, v.device)
    return (v - mr[sl, :1]) * mr[sl, 1:] * gamma + beta


def ref_expand(h, hid, mr1, g1, be1, w2t, b2, rpi, spi):
    """u = W2 gelu(GN1(h)) + b2 with interleaved (value, gate) columns: [M, 2C]."""
    return F.gelu(ref_gn(h[:, :hid], mr1, g1, be1, rpi, spi)) @ w2t + b2


def ref_increment(u, mr2, g2, be2, scale, rpi, spi):
    """scale * GN2(u)[2c] * sigmoid(GN2(u)[2c + 1]): what the update adds to x [M, C]."""
    v = ref_gn(u, mr2, g2, be2, rpi, spi)
    return scale * v[:, 0::2] * torch.sigmoid(v[:, 1::2])


@pytest.mark.parametrize("Fr", [1, 8])
def test_reference_chain_matches_oracle(Fr):
    """The functions above, chained in the engine's order (conv3, statistics, finalize, GELU + expand, statistics,
    finalize, update) on weights packed by the engine's own pack_dconv, reproduce oracle.dconv / _dconv_rows: this fixes
    the slab map and the (value, gate) interleaving that every GPU test below compares against."""
    cfg = htdemucs_config()
    Cc, B, T = 96, 2, 45
    hid = int(Cc / cfg.dconv_comp)
    specs = {}
    _dconv_specs("encoder.1", Cc, cfg, specs)
    state = init_from_specs(specs, seed=3, layer_scale=1.0)            # float32 values: exact in float64 too
    packed = {}
    pack_dconv(lambda n, t: packed.__setitem__(n, t.detach().to(F64).contiguous()), packed, state, "encoder.1",
               cfg.dconv_depth, False)
    g = torch.Generator().manual_seed(4)
    x = torch.randn(B, T, Fr, Cc, generator=g, dtype=F64)
    rows, rpi, slabs = x.reshape(-1, Cc), T * Fr, B * Fr
    for d in range(cfg.dconv_depth):
        p = f"encoder.1.dconv.layers.{d}"
        h = ref_conv3(rows, packed[f"{p}.w1"], packed[f"{p}.b1"], rpi, Fr, 2 ** d)
        mr1 = ref_finalize(ref_sums(h, rpi, Fr, slabs), T * hid)
        u = ref_expand(h, hid, mr1, packed[f"{p}.g1"], packed[f"{p}.be1"], packed[f"{p}.w2t"], packed[f"{p}.b2"], rpi, Fr)
        mr2 = ref_finalize(ref_sums(u, rpi, Fr, slabs), T * 2 * Cc)
        rows = rows + ref_increment(u, mr2, packed[f"{p}.g2"], packed[f"{p}.be2"], packed[f"{p}.scale"], rpi, Fr)
    W = {k: v.to(F64) for k, v in state.items()}
    if Fr == 1:
        want = oracle.dconv(x[:, :, 0].transpose(1, 2), W, "encoder.1.dconv", cfg.dconv_depth).transpose(1, 2)
    else:
        want = oracle._dconv_rows(x.permute(0, 3, 2, 1), W, "encoder.1.dconv", cfg.dconv_depth).permute(0, 3, 2, 1)
    got = rows.view(B, T, Fr, Cc).reshape(want.shape)
    assert (got - x.reshape(want.shape)).abs().max() > 0.1               # the branch is not negligible here
    assert (got - want).abs().max() < 1e-12 * want.abs().max()


# ---------------------------------------------------------------------------------------------------------------------
# GPU operands
class Stage:
    """Random operands of one expansion stage in the kernels' layouts (float32 on the device), the float64 reference
    quantities derived from exactly those float32 values, and the slab map.  Every slab of h gets its own level and
    spread, so that a row read with another slab's statistics shows.  Columns hid..ldh of h hold `pad`."""

    def __init__(self, hid, C, B, T, spi, ldh=None, short=0, seed=0, pad=float("nan"), offset=0.0):
        g = torch.Generator().manual_seed(seed)
        self.hid, self.C, self.T, self.spi = hid, C, T, spi
        self.rpi, self.ldh, self.slabs = T * spi, ldh or hid, B * spi
        self.M = B * self.rpi - short                       # short > 0: the last item is a few rows short
        N = 2 * C
        sl = slab_index(self.M, self.rpi, spi)
        lvl, spread = torch.randn(self.slabs, generator=g), 0.5 + torch.rand(self.slabs, generator=g)
        h = torch.full((self.M, self.ldh), pad)
        h[:, :hid] = torch.randn(self.M, hid, generator=g) * spread[sl, None] + lvl[sl, None]
        self.g1, self.be1 = 1 + 0.2 * torch.randn(hid, generator=g), 0.1 * torch.randn(hid, generator=g)
        self.w2t = torch.randn(hid, N, generator=g) / hid ** 0.5
        self.b2 = 0.3 * torch.randn(N, generator=g)
        self.g2, self.be2 = 1 + 0.2 * torch.randn(N, generator=g), 0.1 * torch.randn(N, generator=g)
        self.scale = 0.5 + torch.rand(C, generator=g)
        self.x = torch.randn(self.M, C, generator=g)
        # GroupNorm statistics of h as the conv3 pass hands them over (per-slab row counts: the last item may be short)
        h64 = h[:, :hid].double()
        cnt = torch.bincount(sl, minlength=self.slabs).double() * hid
        mean = torch.zeros(self.slabs, dtype=F64).index_add_(0, sl, h64.sum(1)) / cnt
        sq = torch.zeros(self.slabs, dtype=F64).index_add_(0, sl, (h64 * h64).sum(1)) / cnt
        self.mr1 = torch.stack([mean, 1 / torch.sqrt(sq - mean * mean + 1e-5)], 1).float()
        for k in ("g1", "be1", "w2t", "b2", "g2", "be2", "scale", "x", "mr1"):
            setattr(self, k, getattr(self, k).to(DEV))
        self.h = h.to(DEV)
        if offset:                                          # common offset of u, `offset` times its spread
            self.b2 += offset * float(self.expand().std())
        self.u = self.expand()
        self.count2 = float(T * N)
        self.mr2_ref = ref_finalize(ref_sums(self.u, self.rpi, spi, self.slabs), self.count2)
        self.mr2 = self.mr2_ref.float()
        self.inc_ref = ref_increment(self.u, self.mr2.double(), self.g2.double(), self.be2.double(), self.scale.double(),
                                     self.rpi, spi)

    def expand(self):
        d = lambda t: t.double()   # noqa: E731
        return ref_expand(d(self.h), self.hid, d(self.mr1), d(self.g1), d(self.be1), d(self.w2t), d(self.b2),
                          self.rpi, self.spi)

    def gram_ws(self):
        return torch.zeros((self.slabs + 1) * (self.hid ** 2 + self.hid) + self.hid + 2, dtype=F64, device=DEV)

    def stats(self, ws):
        """(mean, rstd) [slabs, 2] from bd_dconv_expand_stats (ws = Gram workspace or None) + bd_finalize_group_stats."""
        sums = torch.zeros(self.slabs, 2, dtype=F64, device=DEV)
        _lib.call("bd_dconv_expand_stats", ptr(self.h), self.ldh, self.hid, ptr(self.mr1), ptr(self.g1), ptr(self.be1),
                  ptr(self.w2t), ptr(self.b2), ptr(sums), ptr(ws), self.M, self.C, self.rpi, self.spi, 0)
        mr = torch.full((self.slabs, 2), float("nan"), device=DEV)
        _lib.call("bd_finalize_group_stats", ptr(sums), ptr(mr), self.slabs, self.count2, 0)
        torch.cuda.synchronize()
        assert not sums.any(), "finalize hands the sums back cleared"
        return mr

    def x_guarded(self):
        xg = torch.full((self.M + GUARD, self.C), SENTINEL, device=DEV)
        xg[:self.M] = self.x
        return xg

    def increment(self, xg):
        """x_out - x_in of the first M rows; the guard rows behind them must be untouched."""
        torch.cuda.synchronize()
        assert torch.all(xg[self.M:] == SENTINEL), "rows behind x were written"
        return xg[:self.M] - self.x

    def update(self, math_mode):
        xg = self.x_guarded()
        _lib.call("bd_dconv_expand_update", ptr(self.h), self.ldh, self.hid, ptr(self.mr1), ptr(self.g1), ptr(self.be1),
                  ptr(self.w2t), ptr(self.b2), ptr(self.mr2), ptr(self.g2), ptr(self.be2), ptr(self.scale), ptr(xg),
                  self.M, self.C, self.rpi, self.spi, math_mode, 0)
        return self.increment(xg)


def stat_err(mr, want):
    """max over slabs of |dmean| / std and |drstd| / rstd (std = 1 / rstd, eps included)."""
    mr = mr.double()
    return max(float(((mr[:, 0] - want[:, 0]).abs() * want[:, 1]).max()),
               float(((mr[:, 1] - want[:, 1]).abs() / want[:, 1]).max()))


# ---------------------------------------------------------------------------------------------------------------------
# 1. bd_dconv_expand_stats
GRAM_SPI = [1, 2, 8, 16, 32, 64, 128, 512]
T_OF_SPI = {1: 1001, 2: 533, 8: 133, 16: 67, 32: 37, 64: 19, 128: 13, 512: 5}   # none a multiple of 32
PADDED = {6: 8, 12: 16, 24: 32, 48: 64}           # the engine's h width (8 for the narrow layer, else multiples of 16)


@pytest.mark.gpu
@pytest.mark.parametrize("padded", [False, True])
@pytest.mark.parametrize("spi", GRAM_SPI)
@pytest.mark.parametrize("hid", [6, 12, 24, 48])
def test_expand_stats_gram_and_register(hid, spi, padded):
    """Both arms on every slab geometry the Gram arm accepts.  The Gram workspace must come back zero in its first
    slabs * (hid^2 + hid) entries, and a second call on it (not cleared in between) must give the same statistics: the
    engine zeroes it once.  spi 1 (1001 rows per item) and 512 (2560) are items shorter than 32 * max(32, spi) rows."""
    st = Stage(hid, 8 * hid, B=3 if padded else 1, T=T_OF_SPI[spi], spi=spi, ldh=PADDED[hid] if padded else hid,
               seed=hid * 1000 + spi)
    ws = st.gram_ws()
    gram = st.stats(ws)
    assert not ws[:st.slabs * (hid * hid + hid)].any(), "Gram workspace not handed back zero"
    gram2 = st.stats(ws)
    reg = st.stats(None)
    errs = [stat_err(gram, st.mr2_ref), stat_err(gram2, st.mr2_ref), stat_err(reg, st.mr2_ref),
            stat_err(gram, reg.double())]
    print(f"expand_stats hid={hid} spi={spi} ldh={st.ldh} M={st.M}: gram {errs[0]:.2e} again {errs[1]:.2e} "
          f"register {errs[2]:.2e} gram-vs-register {errs[3]:.2e}")
    assert max(errs) <= STAT_TOL


# shapes gram_supported() refuses, and the launch configurations of the register arm
REGISTER_CASES = {
    "hid5_C40": dict(hid=5, C=40, B=3, T=211, spi=1),            # W2 1.6 KB: 128 threads, 8 CTAs per SM
    "hid10_C400": dict(hid=10, C=400, B=2, T=37, spi=8),         # W2 31 KB: 128 threads, 2 CTAs per SM
    "hid40_C320": dict(hid=40, C=320, B=2, T=37, spi=4),         # W2 100 KB: 512 threads
    "spi3": dict(hid=12, C=96, B=3, T=101, spi=3),
    "spi48": dict(hid=24, C=192, B=2, T=29, spi=48),
    "odd_ldh": dict(hid=6, C=48, B=3, T=333, spi=1, ldh=7),
    "short_item": dict(hid=12, C=96, B=3, T=41, spi=8, short=3),  # M three rows short of a whole item
    "chunks16": dict(hid=48, C=384, B=3, T=37, spi=1),            # M = 111: every row split into 16 column chunks
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(REGISTER_CASES))
def test_expand_stats_register_only(case):
    """The register arm without a workspace; for the shapes the Gram arm refuses also with one, which must stay unused."""
    st = Stage(**REGISTER_CASES[case], seed=len(case))
    errs = [stat_err(st.stats(None), st.mr2_ref)]
    if case != "chunks16":                       # hid 48, spi 1, whole items: the Gram arm would take it
        ws = st.gram_ws()
        errs.append(stat_err(st.stats(ws), st.mr2_ref))
        assert not ws.any()
    print(f"expand_stats {case} M={st.M}: register arm " + ", ".join(f"{e:.2e}" for e in errs))
    assert max(errs) <= STAT_TOL


@pytest.mark.gpu
@pytest.mark.parametrize("gram", [True, False])
def test_expand_stats_offset(gram):
    """u with a common offset of 8x its spread: E[u^2] - E[u]^2 cancels about 65-fold in the finalize step, so the fp32
    partial sums of each arm show.  The Gram arm accumulates g g^T and sum(g) per lane in fp32 and meets the offset
    (through b2) only in fp64; the register arm sums u and u^2 per row in fp32.  Measured on a B200: Gram 3.5e-7,
    register 3.6e-7, against 6e-8 or less without the offset; the bound is that of every other case, 1e-6."""
    st = Stage(24, 192, B=2, T=67, spi=16, ldh=32, offset=8.0, seed=77)
    mean, std = st.mr2_ref[:, 0], 1 / st.mr2_ref[:, 1]
    assert float((mean.abs() / std).min()) > 4
    e = stat_err(st.stats(st.gram_ws() if gram else None), st.mr2_ref)
    print(f"expand_stats offset regime, {'gram' if gram else 'register'} arm: {e:.2e}")
    assert e <= STAT_TOL


# ---------------------------------------------------------------------------------------------------------------------
# 2. bd_dconv_expand_update, compared on the increment of x with mr2 taken from the float64 reference
def update_arm(hid, C, math_mode):
    """The arm bd_dconv_expand_update dispatches to (csrc/dconv.cu)."""
    mma = hid in (6, 12, 24, 48) and C % 48 == 0
    if mma and math_mode in (_lib.MATH_TF32, _lib.MATH_BF16):
        return "mma"
    if mma and hid == 6 and math_mode in (_lib.MATH_TF32X3, _lib.MATH_BF16X3):
        return "mma_x3"
    return "ffma"


def check_update(st, math_mode, label):
    arm = update_arm(st.hid, st.C, math_mode)
    inc = st.update(math_mode)
    e = rel_l2(inc.cpu(), st.inc_ref.cpu())
    ref32 = st.update(_lib.MATH_FP32)
    d = rel_l2(inc.cpu(), ref32.cpu())
    print(f"expand_update {label} math={math_mode} arm={arm} M={st.M}: rel-L2 {e:.2e} (vs FP32 arm {d:.2e})")
    assert e <= TOL[arm]
    # the arm really ran: the dispatcher must not fall through to another arm
    if arm == "mma":
        assert d > 1e-5
    elif arm == "mma_x3":
        assert not torch.equal(inc, ref32)
    else:
        assert torch.equal(inc, ref32)


MATHS = [_lib.MATH_FP32, _lib.MATH_TF32, _lib.MATH_BF16, _lib.MATH_TF32X3, _lib.MATH_BF16X3]


@pytest.mark.gpu
@pytest.mark.parametrize("math_mode", MATHS)
@pytest.mark.parametrize("hid", [6, 12, 24, 48])
def test_expand_update_arms(hid, math_mode):
    """C = 8 * hid, 8 slabs per item (neighbouring rows in different slabs), M = 888 (not a multiple of 32), padded h."""
    st = Stage(hid, 8 * hid, B=3, T=37, spi=8, ldh=PADDED[hid], seed=hid)
    check_update(st, math_mode, f"hid={hid}")


UPDATE_EDGES = {
    "hid5_C40": (REGISTER_CASES["hid5_C40"], _lib.MATH_FP32),
    "hid10_C400": (REGISTER_CASES["hid10_C400"], _lib.MATH_TF32X3),
    "hid40_C320": (REGISTER_CASES["hid40_C320"], _lib.MATH_BF16X3),
    "hid8_C64_tf32": (dict(hid=8, C=64, B=2, T=45, spi=2), _lib.MATH_TF32),     # C % 48 != 0: the FFMA arm
    "M20_mma": (dict(hid=6, C=48, B=1, T=5, spi=4, ldh=8), _lib.MATH_TF32),
    "M20_x3": (dict(hid=6, C=48, B=1, T=5, spi=4, ldh=8), _lib.MATH_BF16X3),
    "M20_ffma": (dict(hid=12, C=96, B=1, T=5, spi=4), _lib.MATH_FP32),
    "odd_ldh_mma": (REGISTER_CASES["odd_ldh"], _lib.MATH_TF32),
    "odd_ldh_ffma": (REGISTER_CASES["odd_ldh"], _lib.MATH_FP32),
    "spi3_mma": (REGISTER_CASES["spi3"], _lib.MATH_BF16),
    "spi48_ffma": (REGISTER_CASES["spi48"], _lib.MATH_TF32X3),
    "short_item_mma": (REGISTER_CASES["short_item"], _lib.MATH_TF32),
    "short_item_ffma": (REGISTER_CASES["short_item"], _lib.MATH_FP32),
    "chunks16_ffma": (REGISTER_CASES["chunks16"], _lib.MATH_FP32),
    "chunks16_mma": (REGISTER_CASES["chunks16"], _lib.MATH_TF32),
    "chunks4_ffma": (dict(hid=24, C=192, B=1, T=13, spi=8, ldh=32), _lib.MATH_BF16X3),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(UPDATE_EDGES))
def test_expand_update_edges(case):
    kw, math_mode = UPDATE_EDGES[case]
    check_update(Stage(**kw, seed=len(case) + 100), math_mode, case)


@pytest.mark.gpu
@pytest.mark.parametrize("spi", [1, 8])
def test_dconv_tail_matches_update(spi):
    """bd_dconv_tail, the header's statement of the update, given u: equal to the FP32 arm up to fp32 rounding."""
    st = Stage(12, 96, B=3, T=37, spi=spi, seed=spi)
    u = st.u.float().contiguous()
    xg = st.x_guarded()
    _lib.call("bd_dconv_tail", ptr(xg), ptr(u), ptr(st.mr2), ptr(st.g2), ptr(st.be2), ptr(st.scale), st.M, st.C,
              st.rpi, st.spi, 0)
    tail = st.increment(xg)
    ffma = st.update(_lib.MATH_FP32)
    e, d = rel_l2(tail.cpu(), st.inc_ref.cpu()), rel_l2(tail.cpu(), ffma.cpu())
    print(f"dconv_tail spi={spi}: rel-L2 {e:.2e}, vs the FP32 update arm {d:.2e}")
    assert e <= 1e-6 and d <= 1e-6


# ---------------------------------------------------------------------------------------------------------------------
# 3. the wide-layer update as Engine._dconv issues it: activate h once, then one GEMM whose epilogue does GroupNorm 2,
#    GLU, LayerScale and the residual, in place on x (resid = out = x)
@pytest.mark.gpu
@pytest.mark.parametrize("math_mode,tol", [(_lib.MATH_BF16X3, 1e-5), (_lib.MATH_TF32X3, 1e-6), (_lib.MATH_TF32, 3e-3),
                                           (_lib.MATH_BF16, 6e-3)])
@pytest.mark.parametrize("Cc,Fr,T", [(192, 1, 1001), (192, 8, 101), (192, 32, 37), (384, 1, 1001), (384, 8, 101),
                                     (384, 32, 37)])
def test_wide_update_gemm(Cc, Fr, T, math_mode, tol):
    """N = 2C of 384 / 768, A = the activated h with its padded width, slab map (T * Fr, Fr, Fr).  BF16X3 carries 16
    mantissa bits per operand (hi + lo), hence its ~4e-6 against TF32X3's 4e-7."""
    hid = Cc // 8
    hp = (hid + 15) // 16 * 16
    st = Stage(hid, Cc, B=2, T=T, spi=Fr, ldh=hp, pad=0.0, seed=Cc + Fr)
    a = st.h.clone()
    g1p = torch.cat([st.g1, torch.zeros(hp - hid, device=DEV)])
    be1p = torch.cat([st.be1, torch.zeros(hp - hid, device=DEV)])
    _lib.call("bd_gn_gelu_apply", ptr(a), ptr(st.mr1), ptr(g1p), ptr(be1p), st.M, hp, st.rpi, st.spi, 0)
    w2p = torch.zeros(2 * Cc, hp, device=DEV)
    w2p[:, :hid] = st.w2t.t()
    xg = st.x_guarded()
    d = GemmDesc()
    d.M, d.N, d.K, d.Cin, d.taps = st.M, 2 * Cc, hp, hp, 1
    d.I1, d.I0, d.m1, d.m0, d.J1, d.J0 = 1, st.M, 1, 1, 1, st.M
    d.xs_b, d.xs_1, d.xs_0, d.xs_c = 0, 0, hp, 1
    d.os_b, d.os_1, d.os_0 = 0, 0, Cc
    d.x, d.w, d.bias, d.out = ptr(a), ptr(w2p), ptr(st.b2), ptr(xg)
    d.e_stats, d.e_gamma, d.e_beta = ptr(st.mr2), ptr(st.g2), ptr(st.be2)
    d.act, d.resid, d.scale = _lib.ACT_GLU, ptr(xg), ptr(st.scale)
    d.stat_div, d.stat_mul, d.stat_mod = st.rpi, st.spi, st.spi
    d.math = math_mode
    if math_mode in (_lib.MATH_BF16X3, _lib.MATH_BF16):
        w_hi = w2p.to(torch.bfloat16)
        w_lo = (w2p - w_hi.float()).to(torch.bfloat16)
        d.w16_hi, d.w16_lo = ptr(w_hi), ptr(w_lo)
    assert _lib.lib().bd_conv_gemm_arm(C.byref(d)) != 0          # a tensor-core arm
    _lib.call("bd_conv_gemm", C.byref(d), 0)
    inc = st.increment(xg)
    act_ref = F.gelu(ref_gn(st.h[:, :hid].double(), st.mr1.double(), st.g1.double(), st.be1.double(), st.rpi, st.spi))
    ea = rel_l2(a[:, :hid].cpu(), act_ref.cpu())
    assert torch.all(a[:, hid:] == 0)
    e = rel_l2(inc.cpu(), st.inc_ref.cpu())
    print(f"wide update C={Cc} Fr={Fr} math={math_mode}: gn_gelu {ea:.2e}, increment rel-L2 {e:.2e}")
    assert ea <= 1e-6 and e <= tol


# ---------------------------------------------------------------------------------------------------------------------
# 4. Engine._dconv at the htdemucs encoder geometries, against oracle.dconv over both depth steps
ENGINE_LAYERS = [("encoder.0", 48, 512, 7), ("encoder.1", 96, 128, 13), ("encoder.2", 192, 32, 37),
                 ("encoder.3", 384, 8, 101), ("tencoder.0", 48, 1, 1001), ("tencoder.3", 384, 1, 1001)]


@pytest.fixture(scope="module")
def htdemucs_state():
    cfg = htdemucs_config()
    return cfg, init_weights(cfg, 11, layer_scale=1.0)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_engine_dconv(mode, htdemucs_state):
    """Every layer is run twice on one buffer key, so that the cached Gram workspaces and statistics accumulators are
    reused as in a forward.  LayerScale 1: the branch is as large as x.  In tf32x3 and strict the error grows with C
    (0.6e-6 at C = 48 to 4.7e-6 at C = 384 in tf32x3): it comes from the tensor-core conv3 GEMM over K = 3C, and strict
    adds the 16-bit operands of BF16X3; hence 2e-5, the bound of those GEMM arithmetics in test_gpu_gemm.py."""
    cfg, state = htdemucs_state
    eng = Engine(cfg, state, DEV, mode)
    W = {k: v.to(DEV, F64) for k, v in state.items() if ".dconv." in k}
    tol = {"fp32": 1e-5, "tf32": 3e-3, "bf16": 3e-3, "tf32x3": 2e-5, "strict": 2e-5}[mode]
    B = 2
    g = torch.Generator().manual_seed(12)
    cases = []
    for prefix, Cc, Fr, T in ENGINE_LAYERS:
        x = torch.randn(B, T, Fr, Cc, generator=g).to(DEV)
        y = x.double().permute(0, 3, 2, 1)                                  # [B, C, Fr, T]
        if Fr == 1:
            want = oracle.dconv(y[:, :, 0], W, f"{prefix}.dconv", cfg.dconv_depth)[:, :, None]
        else:
            want = oracle._dconv_rows(y, W, f"{prefix}.dconv", cfg.dconv_depth)
        cases.append((prefix, Cc, Fr, T, x, (want - y).permute(0, 3, 2, 1)))
    for rep in range(2):
        for prefix, Cc, Fr, T, x, inc_ref in cases:
            xo = x.clone()
            eng._dconv(("dconv-test", B), prefix, xo, B, T, Fr, Cc, "_f" if Fr > 1 else "_t")
            torch.cuda.synchronize()
            e = rel_l2((xo - x).cpu(), inc_ref.cpu())
            print(f"Engine._dconv mode={mode} {prefix} C={Cc} Fr={Fr} T={T} call {rep}: rel-L2 {e:.2e}")
            assert e <= tol


# ---------------------------------------------------------------------------------------------------------------------
# 5. the small normalisation kernels of norm.cu
@pytest.mark.gpu
def test_finalize_group_stats():
    """Biased variance, eps 1e-5, a negative variance (rounding, or worse) clamped to zero, sums handed back cleared.
    count = 37: the unbiased variance would differ by 1 / 36."""
    g = torch.Generator().manual_seed(21)
    slabs, count = 300, 37.0
    mean = 2 * torch.randn(slabs, generator=g, dtype=F64)
    var = 3 * torch.rand(slabs, generator=g, dtype=F64) + 0.01
    var[::7] = -1e-9 * mean[::7] ** 2
    var[3::7] = -0.5
    sums = torch.stack([mean * count, (var + mean * mean) * count], 1).to(DEV)
    want = ref_finalize(sums.clone(), count)
    mr = torch.full((slabs, 2), float("nan"), device=DEV)
    _lib.call("bd_finalize_group_stats", ptr(sums), ptr(mr), slabs, count, 0)
    torch.cuda.synchronize()
    assert not sums.any()
    assert torch.all(mr[::7, 1] == mr[3::7, 1]) and abs(float(mr[0, 1]) - 1e-5 ** -0.5) < 1e-4
    e = float(((mr.double() - want).abs() / want.abs()).max())
    print(f"finalize_group_stats: max relative error {e:.2e}")
    assert e <= 1e-7


@pytest.mark.gpu
@pytest.mark.parametrize("Cc,T,spi", [(8, 333, 1), (32, 37, 8), (48, 101, 3), (64, 7, 512)])
def test_gn_gelu_apply(Cc, T, spi):
    st = Stage(Cc, 8, B=3, T=T, spi=spi, seed=Cc)
    h = st.h.clone()
    _lib.call("bd_gn_gelu_apply", ptr(h), ptr(st.mr1), ptr(st.g1), ptr(st.be1), st.M, Cc, st.rpi, st.spi, 0)
    torch.cuda.synchronize()
    want = F.gelu(ref_gn(st.h.double(), st.mr1.double(), st.g1.double(), st.be1.double(), st.rpi, st.spi))
    e = rel_l2(h.cpu(), want.cpu())
    print(f"gn_gelu_apply C={Cc} spi={spi}: rel-L2 {e:.2e}")
    assert e <= 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("n", [4 * 20011, 4 * 400003])     # the second one exceeds the capped grid: several strides
def test_item_stats(n):
    g = torch.Generator().manual_seed(n % 97)
    B = 3
    x = (torch.randn(B, n, generator=g) + torch.arange(B)[:, None] - 1.0).to(DEV)
    sums = torch.zeros(B, 2, dtype=F64, device=DEV)
    _lib.call("bd_item_stats", ptr(x), ptr(sums), B, n, 0)
    torch.cuda.synchronize()
    xd = x.double()
    es = float(((sums[:, 0] - xd.sum(1)).abs() / xd.abs().sum(1)).max())
    eq = float(((sums[:, 1] - (xd * xd).sum(1)).abs() / (xd * xd).sum(1)).max())
    print(f"item_stats n={n}: sum {es:.2e}, sum of squares {eq:.2e}")
    assert es <= 1e-7 and eq <= 1e-7


@pytest.mark.gpu
def test_group_norm_apply():
    g = torch.Generator().manual_seed(22)
    B, rows, Cc = 3, 1001, 512
    x = (torch.randn(B, rows, Cc, generator=g) * 2 + 1).to(DEV)
    mr = torch.stack([torch.randn(B, generator=g), 0.3 + torch.rand(B, generator=g)], 1).to(DEV)
    gam, bet = (1 + 0.2 * torch.randn(Cc, generator=g)).to(DEV), (0.1 * torch.randn(Cc, generator=g)).to(DEV)
    y = x.clone()
    _lib.call("bd_group_norm_apply", ptr(y), ptr(mr), ptr(gam), ptr(bet), B, rows, Cc, 0)
    torch.cuda.synchronize()
    md = mr.double()
    want = (x.double() - md[:, None, :1]) * md[:, None, 1:] * gam.double() + bet.double()
    e = rel_l2(y.cpu(), want.cpu())
    print(f"group_norm_apply: rel-L2 {e:.2e}")
    assert e <= 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("Cc,pos,alias", [(512, True, False), (768, False, False), (1024, True, True)])
def test_layer_norm_fp32_output(Cc, pos, alias):
    """fp32 output, both register-tile instantiations (C <= 512 and C <= 1024), optional positional table, y = x."""
    g = torch.Generator().manual_seed(Cc)
    M = 3001
    x = (torch.randn(M, Cc, generator=g) * 3 + 0.5).to(DEV)
    gam, bet = torch.randn(Cc, generator=g).to(DEV), torch.randn(Cc, generator=g).to(DEV)
    table = torch.randn(7, Cc, generator=g).to(DEV) if pos else None
    want = F.layer_norm(x.double(), (Cc,), gam.double(), bet.double(), 1e-5)
    if pos:
        want = want + table.double()[torch.arange(M, device=DEV) % 7]
    y = x if alias else torch.full_like(x, float("nan"))
    _lib.call("bd_layer_norm", ptr(x), ptr(y), ptr(gam), ptr(bet), ptr(table), 7 if pos else 0, M, Cc, 0, 0)
    torch.cuda.synchronize()
    e = rel_l2(y.cpu(), want.cpu())
    print(f"layer_norm fp32 C={Cc} pos={pos} in-place={alias}: rel-L2 {e:.2e}")
    assert e <= 1e-6
