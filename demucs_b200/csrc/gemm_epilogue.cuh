// Epilogue shared by the CUDA-core and the tcgen05 implicit-GEMM kernels: everything that happens
// to an accumulator between the contraction and HBM (see bd_gemm_desc in include/demucs_b200.h).
// Two entry points: bd_epi_apply4 finishes 4 consecutive columns with 128-bit accesses (the hot
// path: every full-size layer qualifies), bd_epi_apply is the scalar form for odd geometries.
#pragma once
#include "common.cuh"
#include "../../include/demucs_b200.h"

struct EpiRow {
  long long obase;   // b*os_b + i1*os_1 + (first output position of the row)*os_0
  int i0;
  int rb_row;        // m % rowbias_period
  float e_mean, e_rstd;
};

__device__ __forceinline__ int bd_stat_slab(const bd_gemm_desc& d, long long m64) {
  const unsigned m = (unsigned)m64;
  return (int)((m / (unsigned)d.stat_div) * (unsigned)d.stat_mul + (m % (unsigned)d.stat_mod));
}

__device__ __forceinline__ EpiRow bd_epi_row(const bd_gemm_desc& d, long long m64) {
  EpiRow r;
  const unsigned m = (unsigned)m64;            // M < 2^31: 32-bit divisions
  const unsigned t = m / (unsigned)d.I0;
  r.i0 = (int)(m - t * (unsigned)d.I0);
  const unsigned b = t / (unsigned)d.I1;
  const int i1 = (int)(t - b * (unsigned)d.I1);
  r.obase = (long long)b * d.os_b + (long long)i1 * d.os_1 +
            (long long)(d.convt ? 4 * r.i0 - (d.convt == 1 ? 2 : 0) : r.i0) * d.os_0;
  r.rb_row = d.rowbias ? (int)(m % (unsigned)d.rowbias_period) : 0;
  r.e_mean = 0.f;
  r.e_rstd = 1.f;
  if (d.e_stats) {
    const int sl = bd_stat_slab(d, m64);
    r.e_mean = __ldg(d.e_stats + 2 * (size_t)sl);
    r.e_rstd = __ldg(d.e_stats + 2 * (size_t)sl + 1);
  }
  return r;
}

// Can every epilogue operand be accessed as aligned float4 (float2 after GLU)?  Uniform per launch.
__host__ __device__ __forceinline__ bool bd_epi_vec_ok(const bd_gemm_desc& d) {
  auto al16 = [](const void* p) { return ((uintptr_t)p & 15) == 0; };
  bool ok = d.N % 4 == 0 && d.os_0 % 4 == 0 && d.os_1 % 4 == 0 && d.os_b % 4 == 0;
  ok = ok && al16(d.out) && al16(d.bias) && al16(d.rowbias) && al16(d.resid) && al16(d.scale) && al16(d.addend) &&
       al16(d.e_gamma) && al16(d.e_beta);
  if (d.convt) ok = ok && ((d.N >> 2) % 4 == 0);
  if (d.oc_split) ok = ok && d.oc_split % 4 == 0 && d.oc_stride % 4 == 0 && d.act != BD_ACT_GLU;
  if (d.act != BD_ACT_GLU && d.rowbias) ok = ok && (d.N % 4 == 0);
  return ok;
}

// offset of output column `no` inside a row (optionally split into channel-group planes)
__device__ __forceinline__ long long bd_col_ofs(const bd_gemm_desc& d, int no) {
  if (d.oc_split == 0) return no;
  const int g = no / d.oc_split;
  return (long long)g * d.oc_stride + (no - g * d.oc_split);
}

// output stores: fp32, or bf16 (round to nearest even) when the descriptor says the output tensor is bf16
__device__ __forceinline__ void bd_store_out4(const bd_gemm_desc& d, long long o, float4 v) {
  if (d.out_bf16)
    *reinterpret_cast<uint2*>(reinterpret_cast<uint16_t*>(d.out) + o) = make_uint2(bd_pack_bf16(v.x, v.y), bd_pack_bf16(v.z, v.w));
  else
    *reinterpret_cast<float4*>(d.out + o) = v;
}
__device__ __forceinline__ void bd_store_out2(const bd_gemm_desc& d, long long o, float2 v) {
  if (d.out_bf16)
    *reinterpret_cast<uint32_t*>(reinterpret_cast<uint16_t*>(d.out) + o) = bd_pack_bf16(v.x, v.y);
  else
    *reinterpret_cast<float2*>(d.out + o) = v;
}
__device__ __forceinline__ void bd_store_out1(const bd_gemm_desc& d, long long o, float v) {
  if (d.out_bf16)
    reinterpret_cast<uint16_t*>(d.out)[o] = (uint16_t)(bd_pack_bf16(v, 0.f) & 0xffffu);
  else
    d.out[o] = v;
}

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float2 ldg2(const float* p) { return __ldg(reinterpret_cast<const float2*>(p)); }

// Column-side operands of a 4-column group (bias, GroupNorm affine, LayerScale, output column offset): they
// depend on n only, so a thread that keeps its column group across rows computes them once.
struct EpiCol {
  float4 bias, gamma, beta, scale;
  long long colofs;  // offset of the first stored element relative to EpiRow::obase
  int no, nout;      // first output channel, channels per output position
  int rr;            // transposed conv: output phase of this column group
};

__device__ __forceinline__ EpiCol bd_epi_cols4(const bd_gemm_desc& d, int n) {
  EpiCol c;
  c.bias = d.bias ? ldg4(d.bias + n) : make_float4(0.f, 0.f, 0.f, 0.f);
  c.gamma = c.beta = make_float4(0.f, 0.f, 0.f, 0.f);
  if (d.e_stats) {
    c.gamma = ldg4(d.e_gamma + n);
    c.beta = ldg4(d.e_beta + n);
  }
  c.rr = 0;
  if (d.act == BD_ACT_GLU) {
    c.no = n >> 1;
    c.nout = d.N >> 1;
    c.colofs = bd_col_ofs(d, c.no);
  } else if (d.convt) {
    c.nout = d.N >> 2;
    c.rr = n / c.nout;
    c.no = n - c.rr * c.nout;
    c.colofs = (long long)c.rr * d.os_0 + bd_col_ofs(d, c.no);
  } else {
    c.no = n;
    c.nout = d.N;
    c.colofs = bd_col_ofs(d, n);
  }
  c.scale = make_float4(1.f, 1.f, 1.f, 1.f);
  if (d.resid && d.scale) {
    if (d.act == BD_ACT_GLU) {
      const float2 t = ldg2(d.scale + c.no);
      c.scale.x = t.x; c.scale.y = t.y;
    } else {
      c.scale = ldg4(d.scale + c.no);
    }
  }
  return c;
}

// Memory-side operands of one 4-column group: output offset plus the residual / skip / embedding
// values, fetched BEFORE any arithmetic so that a caller can put several groups' loads in flight
// (the in-place residual update makes loads and stores alias, which stops the compiler from doing it).
struct EpiMem {
  long long o;       // output offset of the first stored element, -1: nothing to store
  float4 resid, addend, rowbias;
};

__device__ __forceinline__ EpiMem bd_epi_fetch4(const bd_gemm_desc& d, const EpiRow& r, const EpiCol& c) {
  EpiMem e;
  e.resid = e.addend = e.rowbias = make_float4(0.f, 0.f, 0.f, 0.f);
  e.o = r.obase + c.colofs;
  if (d.convt) {
    const int o0 = 4 * r.i0 + c.rr - (d.convt == 1 ? 2 : 0);
    if (o0 < 0 || o0 >= d.O0) {
      e.o = -1;
      return e;
    }
  }
  if (d.act == BD_ACT_GLU) {
    if (d.rowbias) { const float2 t = ldg2(d.rowbias + (size_t)r.rb_row * c.nout + c.no); e.rowbias.x = t.x; e.rowbias.y = t.y; }
    if (d.resid) { const float2 t = ldg2(d.resid + e.o); e.resid.x = t.x; e.resid.y = t.y; }
    if (d.addend) { const float2 t = ldg2(d.addend + e.o); e.addend.x = t.x; e.addend.y = t.y; }
    return e;
  }
  if (d.rowbias) e.rowbias = ldg4(d.rowbias + (size_t)r.rb_row * c.nout + c.no);
  if (d.resid) e.resid = ldg4(d.resid + e.o);
  if (d.addend) e.addend = ldg4(d.addend + e.o);
  return e;
}

// Finish accumulator columns n..n+3 (n % 4 == 0, n + 3 < N) of row r.  Adds the stored values to (s, q).
__device__ __forceinline__ void bd_epi_finish4(const bd_gemm_desc& d, const EpiRow& r, const EpiCol& c, float4 v,
                                               const EpiMem& e, float& s, float& q) {
  if (e.o < 0) return;
  v.x += c.bias.x; v.y += c.bias.y; v.z += c.bias.z; v.w += c.bias.w;
  if (d.e_stats) {
    const float4 g = c.gamma, be = c.beta;
    v.x = fmaf((v.x - r.e_mean) * r.e_rstd, g.x, be.x);
    v.y = fmaf((v.y - r.e_mean) * r.e_rstd, g.y, be.y);
    v.z = fmaf((v.z - r.e_mean) * r.e_rstd, g.z, be.z);
    v.w = fmaf((v.w - r.e_mean) * r.e_rstd, g.w, be.w);
  }
  if (d.act == BD_ACT_GLU) {
    float2 o2 = make_float2(v.x * bd_sigmoid(v.y), v.z * bd_sigmoid(v.w));
    o2.x += e.rowbias.x; o2.y += e.rowbias.y;
    if (d.resid) {
      o2.x = fmaf(c.scale.x, o2.x, e.resid.x); o2.y = fmaf(c.scale.y, o2.y, e.resid.y);
    }
    o2.x += e.addend.x; o2.y += e.addend.y;
    if (d.out) bd_store_out2(d, e.o, o2);
    s += o2.x + o2.y;
    q = fmaf(o2.x, o2.x, fmaf(o2.y, o2.y, q));
    return;
  }
  if (d.act == BD_ACT_GELU) {
    v.x = bd_gelu(v.x); v.y = bd_gelu(v.y); v.z = bd_gelu(v.z); v.w = bd_gelu(v.w);
  }
  v.x += e.rowbias.x; v.y += e.rowbias.y; v.z += e.rowbias.z; v.w += e.rowbias.w;
  if (d.resid) {
    v.x = fmaf(c.scale.x, v.x, e.resid.x); v.y = fmaf(c.scale.y, v.y, e.resid.y);
    v.z = fmaf(c.scale.z, v.z, e.resid.z); v.w = fmaf(c.scale.w, v.w, e.resid.w);
  }
  v.x += e.addend.x; v.y += e.addend.y; v.z += e.addend.z; v.w += e.addend.w;
  if (d.out) bd_store_out4(d, e.o, v);
  s += (v.x + v.y) + (v.z + v.w);
  q = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, q))));
}

__device__ __forceinline__ void bd_epi_apply4(const bd_gemm_desc& d, const EpiRow& r, const EpiCol& c, float4 v,
                                              float& s, float& q) {
  const EpiMem e = bd_epi_fetch4(d, r, c);
  bd_epi_finish4(d, r, c, v, e, s, q);
}

// Scalar form: finish accumulator `acc` of column n (and `acc_gate` of column n+1 for GLU, n even).
// Returns false when nothing is stored (GLU gate column / cropped transposed-conv position).
__device__ __forceinline__ bool bd_epi_apply(const bd_gemm_desc& d, const EpiRow& r, int n, float acc, float acc_gate,
                                             float& stored) {
  float v = acc + (d.bias ? __ldg(d.bias + n) : 0.f);
  if (d.e_stats) v = fmaf((v - r.e_mean) * r.e_rstd, __ldg(d.e_gamma + n), __ldg(d.e_beta + n));
  int no = n;
  int Nout = d.N;
  if (d.act == BD_ACT_GLU) {
    if (n & 1) return false;
    float g = acc_gate + (d.bias ? __ldg(d.bias + n + 1) : 0.f);
    if (d.e_stats) g = fmaf((g - r.e_mean) * r.e_rstd, __ldg(d.e_gamma + n + 1), __ldg(d.e_beta + n + 1));
    v = v * bd_sigmoid(g);
    no = n >> 1;
    Nout = d.N >> 1;
  } else if (d.act == BD_ACT_GELU) {
    v = bd_gelu(v);
  }
  long long o;
  if (d.convt) {
    const int Cout = d.N >> 2;
    const int rr = n / Cout;
    const int o0 = 4 * r.i0 + rr - (d.convt == 1 ? 2 : 0);
    if (o0 < 0 || o0 >= d.O0) return false;
    no = n - rr * Cout;
    Nout = Cout;
    o = r.obase + (long long)rr * d.os_0 + bd_col_ofs(d, no);
  } else {
    o = r.obase + bd_col_ofs(d, no);
  }
  if (d.rowbias) v += __ldg(d.rowbias + (size_t)r.rb_row * Nout + no);
  if (d.resid) v = fmaf(d.scale ? __ldg(d.scale + no) : 1.f, v, __ldg(d.resid + o));
  if (d.addend) v += __ldg(d.addend + o);
  if (d.out) bd_store_out1(d, o, v);
  stored = v;
  return true;
}
