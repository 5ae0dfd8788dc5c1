"""GPU: the strict-mode (bf16 hi/lo) tcgen05 GEMM with its split A operand in tensor memory and the exact 96 / 192-column
tiles, against float64 torch, and bit for bit against the in-place shared-memory split (BD_TC_SMEM_A=1) and the
power-of-two tiles (BD_TC_NO_EXACT=1).  Both switches are read per call."""
import ctypes as C
import os

import pytest
import torch
import torch.nn.functional as F

from _fixtures import rel_l2
from demucs_b200 import _lib
from demucs_b200._lib import GemmDesc, ptr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SWITCHES = ("BD_TC_SMEM_A", "BD_TC_NO_EXACT")
TAPS9 = tuple((kt - 1, kf - 1) for kf in range(3) for kt in range(3))
TAPS8 = tuple((0, k - 2) for k in range(8))
# 148 row tiles of 128 (one per SM of a B200): a 192-column tile is then chosen over two 128-column ones, which the
# tile-width choice avoids for problems that would leave SMs idle
WAVE_ROWS = 148 * 128


class Case:
    """One strict-mode bd_conv_gemm launch over x [B, I1, J0, Cin] (channels-last) and W [N, taps * Cin]."""

    def __init__(self, N, Cin, B=2, I1=1, I0=640, taps=((0, 0),), stride4=False, act=_lib.ACT_NONE, resid=False,
                 e_stats=False, rowbias=0, convt=0, stats=None, seed=0):
        g = torch.Generator().manual_seed(seed)
        self.B, self.I1, self.I0, self.taps, self.stride4, self.act, self.convt = B, I1, I0, taps, stride4, act, convt
        self.J0 = 4 * I0 if stride4 else I0
        self.M, K = B * I1 * I0, len(taps) * Cin
        self.x = torch.randn(B, I1, self.J0, Cin, generator=g).to(DEV)
        self.w = (torch.randn(N, K, generator=g) / K ** 0.5).to(DEV)
        self.w_hi = self.w.to(torch.bfloat16)
        self.w_lo = (self.w - self.w_hi.float()).to(torch.bfloat16)
        self.bias = torch.randn(N, generator=g).to(DEV)
        self.n_out = N // 2 if act == _lib.ACT_GLU else (N // 4 if convt else N)
        self.O0 = 4 * I0 - 4
        rows = B * I1 * (self.O0 if convt else I0)
        self.resid = torch.randn(rows, self.n_out, generator=g).to(DEV) if resid else None
        self.scale = torch.randn(self.n_out, generator=g).to(DEV) if resid else None
        slabs = B
        self.e_stats = torch.stack([torch.randn(slabs, generator=g), 0.5 + torch.rand(slabs, generator=g)], 1).to(DEV) \
            if e_stats else None
        self.e_gamma = torch.randn(N, generator=g).to(DEV) if e_stats else None
        self.e_beta = torch.randn(N, generator=g).to(DEV) if e_stats else None
        self.rowbias = torch.randn(rowbias, self.n_out, generator=g).to(DEV) if rowbias else None
        self.stats = stats                      # None, "item" (one slab per item) or "rows" (4 row classes per item)
        d = self.d = GemmDesc()
        d.M, d.N, d.K, d.Cin, d.taps = self.M, N, K, Cin, len(taps)
        d.I1, d.I0, d.m1, d.m0, d.J1, d.J0 = I1, I0, 1, (4 if stride4 else 1), I1, self.J0
        for i, (a, b) in enumerate(taps):
            d.d1[i], d.d0[i] = a, b
        d.xs_b, d.xs_1, d.xs_0, d.xs_c = I1 * self.J0 * Cin, self.J0 * Cin, Cin, 1
        opos = self.O0 if convt else I0
        d.os_b, d.os_1, d.os_0 = I1 * opos * self.n_out, opos * self.n_out, self.n_out
        d.x, d.w, d.bias, d.act = ptr(self.x), ptr(self.w), ptr(self.bias), act
        d.resid, d.scale = ptr(self.resid), ptr(self.scale)
        d.e_stats, d.e_gamma, d.e_beta = ptr(self.e_stats), ptr(self.e_gamma), ptr(self.e_beta)
        d.rowbias, d.rowbias_period = ptr(self.rowbias), rowbias
        d.convt, d.O0 = convt, (self.O0 if convt else 0)
        d.stat_div, d.stat_mul, d.stat_mod = (I1 * I0, 1, 1) if stats != "rows" else (I1 * I0, 4, 4)
        d.math, d.w16_hi, d.w16_lo = _lib.MATH_BF16X3, ptr(self.w_hi), ptr(self.w_lo)
        self.out_rows = rows

    def run(self, **env):
        """(output, stats or None, kernel tile code) with the given switches set for this call only."""
        for k in SWITCHES:
            os.environ.pop(k, None)
        os.environ.update(env)
        try:
            out = torch.full((self.out_rows, self.n_out), float("nan"), device=DEV)
            nslab = self.B * (4 if self.stats == "rows" else 1)
            sums = torch.zeros(nslab, 2, dtype=torch.float64, device=DEV)
            self.d.out = ptr(out)
            self.d.stats_out = ptr(sums) if self.stats else None
            tile = _lib.lib().bd_conv_gemm_arm(C.byref(self.d))
            _lib.call("bd_conv_gemm", C.byref(self.d), 0)
            torch.cuda.synchronize()
        finally:
            for k in SWITCHES:
                os.environ.pop(k, None)
        return out, (sums if self.stats else None), tile

    def reference(self):
        """float64 output rows (plain / GELU / GLU / residual; no e_stats, row bias or transposed conv)."""
        x, w = self.x.double(), self.w.double()
        Cin = x.shape[-1]
        acc = torch.zeros(self.B, self.I1, self.I0, w.shape[0], dtype=torch.float64, device=DEV)
        xp = F.pad(x, (0, 0, 8, 8, 1, 1))      # positions padded by 8, rows by 1: zero padding of every tap
        for t, (d1, d0) in enumerate(self.taps):
            step = 4 if self.stride4 else 1
            sl = xp[:, 1 + d1:1 + d1 + self.I1, 8 + d0:8 + d0 + step * self.I0:step, :]
            acc += sl @ w[:, t * Cin:(t + 1) * Cin].t()
        v = acc.reshape(self.M, -1) + self.bias.double()
        if self.act == _lib.ACT_GELU:
            v = F.gelu(v)
        elif self.act == _lib.ACT_GLU:
            v = v[:, 0::2] * torch.sigmoid(v[:, 1::2])
        if self.resid is not None:
            v = self.resid.double() + self.scale.double() * v
        return v


def bits(t):
    return t.contiguous().view(torch.int32)


@pytest.mark.parametrize("N", [48, 96, 192, 384])
@pytest.mark.parametrize("K", [144, 256])                  # Cin % 32 == 16: 16-deep k-blocks; 256: 32-deep
def test_strict_gemm_vs_fp64(N, K):
    c = Case(N, K, B=1, I0=WAVE_ROWS)
    out, _, tile = c.run()
    assert tile // 1000 == (16 if K % 32 else 32)
    assert tile % 1000 == {48: 64, 96: 96, 192: 192, 384: 128}[N]
    assert not torch.isnan(out).any()
    e = rel_l2(out.cpu(), c.reference().cpu())
    print(f"strict {c.M}x{N}x{K} tile {tile}: rel-L2 {e:.2e}")
    assert e < 2e-5


@pytest.mark.parametrize("kind", ["3x3", "k8s4"])
def test_strict_implicit_conv_vs_fp64(kind):
    if kind == "3x3":       # decoder rewrite: 9 taps over (time, frequency), GLU, N = 192 -> exact 192-wide tiles
        c = Case(192, 96, B=37, I1=8, I0=64, taps=TAPS9, act=_lib.ACT_GLU)
    else:                   # encoder: 8 taps, stride 4 along the position axis, GELU, N = 96 -> exact 96-wide tiles
        c = Case(96, 48, B=2, I1=1, I0=500, taps=TAPS8, stride4=True, act=_lib.ACT_GELU)
    out, _, tile = c.run()
    assert tile % 1000 in (96, 192)
    assert rel_l2(out.cpu(), c.reference().cpu()) < 2e-5


# every compile-time epilogue (ids 0..6 of epi_fast_id) and the generic one (N % 4 != 0), at exact and power-of-two widths
EPILOGUES = {
    "plain": dict(), "resid": dict(resid=True), "gelu": dict(act=_lib.ACT_GELU), "glu": dict(act=_lib.ACT_GLU),
    "glu_gn_resid": dict(act=_lib.ACT_GLU, e_stats=True, resid=True), "rowbias_glu": dict(act=_lib.ACT_GLU, rowbias=7),
    "convt_gelu": dict(act=_lib.ACT_GELU, convt=1), "generic": dict(),
}


@pytest.mark.parametrize("epi", list(EPILOGUES))
@pytest.mark.parametrize("N", [64, 96, 128, 192])
def test_tmem_a_bit_identical_to_smem_a(epi, N):
    """Same hi / lo operands, same MMA order: the tensor-memory A path reproduces the shared-memory one bit for bit."""
    if epi == "generic":
        N -= 2                                               # N % 4 != 0: the scalar epilogue
    c = Case(N, 96, B=2, I1=2, I0=WAVE_ROWS // 4, **EPILOGUES[epi], seed=N)
    new, _, t_new = c.run()
    old, _, t_old = c.run(BD_TC_SMEM_A="1")
    assert t_new == t_old
    assert torch.equal(bits(new), bits(old))
    if epi in ("plain", "resid", "gelu", "glu", "generic"):
        assert rel_l2(new.cpu(), c.reference().cpu()) < 2e-5


@pytest.mark.parametrize("N,Cin", [(96, 48), (192, 96), (90, 48), (176, 32)])
def test_exact_tiles_bit_identical_to_padded(N, Cin):
    """A 96 / 192-column tile computes every output column with the same MMA sequence as the padded 128-column tile."""
    c = Case(N, Cin, B=2, I1=74, I0=96, taps=TAPS9, act=_lib.ACT_GLU if N % 4 == 0 else _lib.ACT_NONE)
    new, _, t_new = c.run()
    old, _, t_old = c.run(BD_TC_SMEM_A="1", BD_TC_NO_EXACT="1")
    assert t_new % 1000 in (96, 192) and t_old % 1000 in (128,)
    assert torch.equal(bits(new), bits(old))


@pytest.mark.parametrize("stats", ["item", "rows"])
@pytest.mark.parametrize("N", [96, 190])
def test_stats_out(stats, N):
    """Per-slab sum / sum of squares of the stored outputs over every chunk of a 96 / 192-column tile."""
    c = Case(N, 64, B=4, I1=1, I0=WAVE_ROWS // 4, stats=stats)
    out, sums, tile = c.run()
    assert tile % 1000 in (96, 192)
    o = out.double().view(c.B, c.I1 * c.I0, -1)
    if stats == "rows":
        o = o.view(c.B, -1, 4, N).transpose(1, 2)
    o = o.reshape(sums.shape[0], -1)
    assert torch.allclose(sums[:, 0], o.sum(1), rtol=1e-6, atol=1e-4)
    assert torch.allclose(sums[:, 1], (o ** 2).sum(1), rtol=1e-6)
