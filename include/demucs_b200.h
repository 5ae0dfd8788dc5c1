/* demucs_b200 -- C ABI of the sm_100a kernel library (libdemucs_b200.so).
 *
 * The reference (DrorT/demucs) is pure Python + PyTorch and has no FFI of its own; its
 * boundary for this path is the Python API (demucs/api.py:53-319, demucs/apply.py:145-322,
 * demucs/htdemucs.py:527-660).  This header declares the entry points the Python host layer
 * (demucs_b200/engine.py) binds with ctypes, each replacing the PyTorch library calls the
 * reference makes at the cited lines.  INTEGRATION.md shows the reference-side binding.
 *
 * Conventions: plain pointers to DEVICE memory owned by the caller, sizes as int / long long,
 * `stream` is a cudaStream_t passed as void*.  No entry point synchronises, allocates or
 * keeps state between calls.  Return value: 0 on success, negative on error
 * (bd_last_error() gives the message; per thread).  All tensors are float32 unless noted.
 *
 * Activation layout ("position-innermost channels-last"): time branch [B, T, C], frequency
 * branch [B, T, F, C]; C is the fastest axis.  DESIGN.md section 3 explains why.
 */
#ifndef DEMUCS_B200_H
#define DEMUCS_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define BD_MAX_TAPS 9

/* A-operand transforms applied while the implicit-GEMM gathers its rows. */
enum { BD_A_NONE = 0, BD_A_GN_GELU = 1, BD_A_ITEM_AFFINE = 2 };
/* Epilogue activations. BD_ACT_GLU expects interleaved (value, gate) output columns. */
enum { BD_ACT_NONE = 0, BD_ACT_GELU = 1, BD_ACT_GLU = 2 };
/* Arithmetic of the contraction. */
/* FP32: CUDA-core FFMA.  TF32: tcgen05 kind::tf32, single pass.  TF32X3: tcgen05, operands split into
 * hi + lo TF32 parts in shared memory, hi*hi + lo*hi + hi*lo (fp32-class accuracy).
 * BF16X3: tcgen05 kind::f16, fp32 activations split into bf16 hi + lo in shared memory, weights pre-split
 * (w16_hi / w16_lo), hi*hi + hi*lo + lo*hi: 16 mantissa bits per operand, ~4e-6 per layer -- the arithmetic of the
 * default mode (per-stem rel-L2 <= 1e-4).  BF16: single bf16 product (the reduced-precision mode, <= 1e-2). */
enum { BD_MATH_FP32 = 0, BD_MATH_TF32 = 1, BD_MATH_TF32X3 = 2, BD_MATH_BF16X3 = 3, BD_MATH_BF16 = 4 };

/* One convolution / linear layer expressed as an implicit GEMM
 *   out[m, n] = epilogue( sum_{tap, ci} A(m, tap, ci) * w[n, tap*Cin + ci] + bias[n] )
 * Row m = (b * I1 + i1) * I0 + i0.  A(m, tap, ci) = x[b*xs_b + j1*xs_1 + j0*xs_0 + ci*xs_c]
 * with j1 = i1*m1 + d1[tap], j0 = i0*m0 + d0[tap]; taps outside [0,J1) x [0,J0) read zero
 * (the zero padding of Conv1d/Conv2d/ConvTranspose).  Covers, in the reference:
 *   Conv1d/Conv2d k=8,s=4 (hdemucs.py:110), 1x1 rewrite (:116), dilated k=3 DConv convs
 *   (demucs.py:138,140), decoder k=3 / 3x3 rewrite (hdemucs.py:294), ConvTranspose k=8,s=4
 *   (hdemucs.py:287, `convt`), channel up/down-samplers (htdemucs.py:369-379) and every
 *   nn.Linear / in_proj / out_proj of the transformer (transformer.py:365,418,506-512). */
typedef struct bd_gemm_desc {
  int M, N, K;
  int Cin, taps;
  int I1, I0;
  int m1, m0, J1, J0;
  int d1[BD_MAX_TAPS], d0[BD_MAX_TAPS];
  long long xs_b, xs_1, xs_0, xs_c;
  const float* x;
  const float* w;      /* [N, K] row-major, K = taps*Cin */
  const float* bias;   /* [N] or NULL */
  /* A prologue */
  int a_mode;
  const float* a_stats; /* GN_GELU: [slab][2] = mean, rstd, slab(m) as below.  ITEM_AFFINE: per item b,
                           a_stats[b*a_stats_stride + 0] = mean, [+2] = 1/(eps+std) */
  int a_stats_stride;
  const float* a_gamma; /* [Cin] (GN_GELU) */
  const float* a_beta;  /* [Cin] */
  /* epilogue, in this order: v = acc + bias; [GroupNorm: v = (v - mean)*rstd*e_gamma[n] + e_beta[n]];
   * v = act(v); v += rowbias[(m % period)*Nout + n]; v = resid + scale[n]*v (scale NULL -> 1);
   * v += addend; store (skipped when out is NULL: statistics-only pass); accumulate stats of v */
  const float* e_stats;  /* [slab][2] = mean, rstd of THIS layer's pre-activation output (slab map below), or NULL */
  const float* e_gamma;  /* [N] */
  const float* e_beta;   /* [N] */
  int act;
  const float* rowbias;
  int rowbias_period;
  const float* resid;
  const float* scale;
  const float* addend;
  float* out;          /* out index = b*os_b + i1*os_1 + o0*os_0 + n_out */
  long long os_b, os_1, os_0;
  int convt;           /* 0: o0 = i0.  Transposed conv k=8,s=4 with N = 4*Cout, r = n / Cout:
                          1: rows = input positions + 1, taps (0,-1): o0 = 4*i0 + r - 2
                          2: rows = input positions, taps (-1,0,+1), zero-extended weights: o0 = 4*i0 + r */
  int O0;              /* convt: valid output positions are 0 <= o0 < O0 */
  int oc_split;        /* 0: output column c lands at + c.  > 0 (multiple of 4): at + (c / oc_split)*oc_stride +
                          c % oc_split -- writes channel groups (e.g. the 4 floats of one source) to separate planes */
  long long oc_stride;
  double* stats_out;   /* [slab][2] += (sum, sumsq) of stored values; or NULL */
  /* GroupNorm slab of row m (for stats_out and for the GN_GELU prologue):
   *   slab(m) = (m / stat_div) * stat_mul + (m % stat_mod)
   * time branch / tokens: one slab per item (stat_div = rows per item, stat_mul = stat_mod = 1);
   * frequency branch [B,T,F,C]: one slab per (b, fr): stat_div = T*F, stat_mul = stat_mod = F. */
  int stat_div, stat_mul, stat_mod;
  int math;            /* BD_MATH_* */
  const void* w16_hi;  /* BD_MATH_BF16X3 / BD_MATH_BF16: bf16 [N, K] = bf16_rn(w) */
  const void* w16_lo;  /* BD_MATH_BF16X3: bf16 [N, K] = bf16_rn(w - w16_hi) */
  /* bf16 storage (the "bf16" mode's transformer: tensors that only ever travel from one GEMM / attention to the next):
   * x_bf16: x is bf16 (element strides as above; BD_MATH_BF16 only, Cin % 64 == 0, read by TMA, no conversion);
   * out_bf16: out is bf16 (same index arithmetic in elements).  resid / addend / rowbias / statistics stay fp32. */
  int x_bf16, out_bf16;
} bd_gemm_desc;

const char* bd_last_error(void);
int bd_version(void);

/* K1 (spec.py:11-27 + htdemucs.py:420-461 + hdemucs.py:23-40): mix [B,2,L] -> spec [B,T,2048,4]
 * (T = ceil(L/1024)); stats[b*4 + {0,1,2,3}] += sum/sumsq of spec and of mix (zero them first). */
int bd_stft_cac(const float* mix, const float* window, const float* twiddle, float* spec, double* stats,
                int B, int A, int L, void* stream);
/* htdemucs.py:545-554: stats -> norm[b*8 + {0..2}] = (mean, std, 1/(1e-5+std)) of spec, [+4..6] of mix. */
int bd_finalize_item_norm(const double* stats, float* norm, int B, double n_freq, double n_time, void* stream);
/* K2a / K2b: the two-kernel form of K2 (frames through HBM).  Diagnostic entry points: the engine uses the fused
 * bd_istft_ola; the parity tests use these to check the inverse FFT and the overlap-add separately.
 * K2a (htdemucs.py:442-471,624-626 + spec.py:30-47): spec [B,T,2048,4S] -> frames [B,S,2,T,4096]. */
int bd_istft_frames(const float* spec, const float* norm, const float* window, const float* twiddle, float* frames,
                    int B, int S, int T, void* stream);
/* K2b (htdemucs.py:449,653-659): out[B,S,2,Lout] = OLA(frames) + xt*stdt + meant; xt [B,Lseg,2S] or NULL. */
int bd_ola_combine(const float* frames, const float* xt, const float* norm, float* out, int B, int S, int T, int Lseg,
                   int Lout, void* stream);

/* K2 fused (same reference lines as K2a + K2b): spec [B,T,S,2048,4] source-major -> out [B,S,2,Lout], with the
 * overlap-add done in shared memory (no frames buffer) and xt [B,Lseg,2S]*stdt+meant added (xt may be NULL). */
int bd_istft_ola(const float* spec, const float* norm, const float* window, const float* twiddle, const float* xt,
                 float* out, int B, int S, int T, int Lseg, int Lout, void* stream);

/* K3/K4/K7: implicit-GEMM convolution / linear layer, see bd_gemm_desc. */
int bd_conv_gemm(const bd_gemm_desc* desc, void* stream);
/* Which arm bd_conv_gemm will use for this descriptor: 0 = fp32 CUDA-core, else 1000*TBK + TBN of the tcgen05
 * kernel template (k-block depth 16/32, tile width 16..256). */
int bd_conv_gemm_arm(const bd_gemm_desc* desc);

/* K5 (GroupNorm(1,C) demucs.py:123, MyGroupNorm transformer.py:258-268): (sum,sumsq) -> (mean, rstd),
 * biased variance, eps 1e-5.  count = elements per slab.  The sums are cleared afterwards, so a buffer that starts
 * at zero needs no fill between one accumulate -> finalize round and the next. */
int bd_finalize_group_stats(double* sums, float* mean_rstd, int slabs, double count, void* stream);
/* DConv tail, diagnostic entry point (the engine fuses it: bd_dconv_expand_update, or the GEMM epilogue)
 * (demucs.py:141-142,151-153): x[m, c] += scale[c] * GLU(GN(u))[m, c]; u [M, 2C] with
 * interleaved (value, gate) columns; GroupNorm slab of row m =
 * (m / rows_per_item) * slabs_per_item + m % slabs_per_item  (time: 1 slab per item; freq: one per bin). */
int bd_dconv_tail(float* x, const float* u, const float* mean_rstd, const float* gamma, const float* beta,
                  const float* scale, long long M, int C, long long rows_per_item, int slabs_per_item, void* stream);
/* DConv expansion stage (demucs.py:138-142,151-153), dedicated HBM-shaped kernels; slab map as bd_dconv_tail.
 *   h [M, ldh] holds the conv3 output (first `hid` columns), w2t [hid, 2C] is the transposed 1x1 weight with
 *   interleaved (value, gate) columns, b2/gamma2/beta2 [2C] interleaved likewise.
 * _stats : sums2[slab] += (sum, sumsq) of u = W2 gelu(gn1(h)) + b2            (u is never stored)
 *          gram_ws: optional workspace of (slabs + 1) * (hid*hid + hid) + hid + 2 doubles, ALL ZERO on entry (it is
 *          returned all zero in its first slabs*(hid*hid+hid) entries).  When given (hid in 6/12/24/48) the sums are
 *          derived from the slab's Gram matrix sum(g g^T): hid^2 instead of hid*2C products per row.
 * _update: x[m, c] += scale[c] * gn2(u)[2c] * sigmoid(gn2(u)[2c+1])            (in place); math = BD_MATH_*:
 *          BD_MATH_TF32 / BD_MATH_BF16 run the expansion on mma.sync tf32 fragments, BD_MATH_TF32X3 / BD_MATH_BF16X3 on
 *          the same fragments with hi/lo split operands (three products), BD_MATH_FP32 in exact fp32 */
/* First encoder layer of a branch (hdemucs.py:110,139-144): out = gelu(conv_{k=8,s=4,p=2}((x - mean_b) * rstd_b) + bias)
 * with the per-item input normalisation (htdemucs.py:545-554) folded into the load; positions outside [0, Jin) are
 * zero AFTER normalisation.  mean_b = norm[b*norm_stride], rstd_b = norm[b*norm_stride + 2] (bd_finalize_item_norm).
 *   channel_major = 0: x [B, I1, Jin, cin] channels-last (spectrogram, cin = 4);  = 1: x [B, cin, Jin] (the mix, cin = 2,
 *   I1 = 1).  w [cout, 8*cin] tap-major, out [B, I1, Io, cout].  mma.sync tf32 fragments: single pass for
 *   math = BD_MATH_TF32 / BD_MATH_BF16, hi/lo split operands and three products (fp32-class) for BD_MATH_TF32X3 /
 *   BD_MATH_BF16X3; only cout = 48 is built. */
int bd_encoder_conv0(const float* x, int channel_major, const float* norm, int norm_stride, const float* w, const float* bias,
                     float* out, int B, int I1, int Io, int Jin, int cin, int cout, int math, void* stream);
/* DConv dilated k=3 convolution of a narrow layer (demucs.py:138, hid = C/8 = 6) with its GroupNorm statistics,
 * on mma.sync tf32 fragments (BD_MATH_TF32 class arithmetic).  x [M, C] rows in memory order, the conv axis is
 * the position t = (m % rows_per_item) / slabs_per_item, neighbours are dilation * slabs_per_item rows away and
 * read as zero outside the item.  w1 [hid, 3*C] tap-major, h [M, ldh = 8] (columns hid.. are written as zero),
 * sums1[slab] += (sum, sumsq) of h; slab map as bd_dconv_tail.  Only hid 6 / C 48 is built.  math as for
 * bd_encoder_conv0. */
int bd_dconv_conv3(const float* x, const float* w1, const float* b1, float* h, int ldh, double* sums1, long long M, int C,
                   int hid, long long rows_per_item, int slabs_per_item, int dilation, int math, void* stream);
int bd_dconv_expand_stats(const float* h, int ldh, int hid, const float* mean_rstd1, const float* gamma1,
                          const float* beta1, const float* w2t, const float* b2, double* sums2, double* gram_ws,
                          long long M, int C, long long rows_per_item, int slabs_per_item, void* stream);
int bd_dconv_expand_update(const float* h, int ldh, int hid, const float* mean_rstd1, const float* gamma1,
                           const float* beta1, const float* w2t, const float* b2, const float* mean_rstd2,
                           const float* gamma2, const float* beta2, const float* scale, float* x, long long M, int C,
                           long long rows_per_item, int slabs_per_item, int math, void* stream);
/* DConv inner activation (demucs.py:138-139): h[m, c] = gelu(GroupNorm(h))[m, c] in place, slab map as
 * bd_dconv_tail.  Used by the tensor-core arm, whose TMA-fed A operand cannot be transformed on the fly. */
int bd_gn_gelu_apply(float* h, const float* mean_rstd, const float* gamma, const float* beta, long long M, int C,
                     long long rows_per_item, int slabs_per_item, void* stream);
/* nn.LayerNorm(C) (transformer.py:434-436,591-592,597-598) with optional additive table
 * pos[(m % pos_period)*C + c] (positional embedding, transformer.py:655-663). y may alias x; y_bf16 != 0: y is a
 * bf16 tensor (it feeds tensor-core GEMMs only). */
int bd_layer_norm(const float* x, void* y, const float* gamma, const float* beta, const float* pos,
                  int pos_period, long long M, int C, int y_bf16, void* stream);
/* (sum, sumsq) per item of x [B, n]: the statistics of a spectrogram handed to forward_core (htdemucs.py:682-692). */
int bd_item_stats(const float* x, double* sums, int B, long long n, void* stream);
/* MyGroupNorm(1) apply: x[b, t, c] = (x - mean_b) * rstd_b * gamma[c] + beta[c], in place. */
int bd_group_norm_apply(float* x, const float* mean_rstd, const float* gamma, const float* beta, int B,
                        long long rows_per_item, int C, void* stream);

/* K6 (nn.MultiheadAttention via _sa_block/_ca_block, transformer.py:365,418,506): softmax(QK^T/8)V,
 * head_dim 64, no mask.  q [B,Tq,ldq] / k,v [B,Tk,ldk] / o [B,Tq,ldo]; head h uses columns [64h, 64h+64).
 * Every arm: pointers 16-byte aligned, leading dims multiples of 4 (of 8 for bd_attention_bf16). */
/* ws: workspace of bd_attention_workspace(...) floats for the tensor-core arms (V^T staging; hi/lo operand
 * splits for BD_MATH_TF32X3), may be NULL when that is 0 (BD_MATH_FP32). */
long long bd_attention_workspace(int B, int H, int Tq, int Tk, int math);
int bd_attention(const float* q, const float* k, const float* v, float* o, int B, int H, int Tq, int Tk,
                 int ldq, int ldk, int ldv, int ldo, int math, float* ws, void* stream);

/* K6 on bf16 tensors (the "bf16" mode): q [B,Tq,ldq] / k,v [B,Tk,ld*] / o [B,Tq,ldo] are bf16, read by TMA with no
 * conversion pass and no workspace; fp32 softmax statistics and accumulation. */
int bd_attention_bf16(const void* q, const void* k, const void* v, void* o, int B, int H, int Tq, int Tk,
                      int ldq, int ldk, int ldv, int ldo, void* stream);

/* K8 (apply.py:257-301 + utils.py:38-54): overlap-add of separated segments.
 * The window of `length` samples is tiled by nseg segments starting at i*stride; the caller holds the
 * forward outputs of segments [seg_first, seg_first+nseg_local) in segs [nseg_local, rows, valid]
 * (all of them on one GPU; a contiguous block plus its left halo when sharded).  Segment i carries
 * n_i = min(length - i*stride, seg_len) samples starting at column (valid - n_i)/2 (centre trim).
 * For window sample n in [max(n_begin,out_shift), min(n_end,length)):
 *   out[r*out_ld + n - out_shift] (+)= alpha * row_alpha[r] * sum_i w[n-i*stride]*seg_i / sum_i w[n-i*stride]
 * out_shift/alpha implement the shift trick (apply.py:253-255), row_alpha the bag weights (apply.py:219-228). */
int bd_overlap_add(const float* segs, const float* weight, float* out, int seg_first, int nseg_local, int nseg,
                   int rows, int valid, int seg_len, int stride, long long length, long long out_ld,
                   long long out_shift, long long n_begin, long long n_end, const float* row_alpha, float alpha,
                   int accumulate, void* stream);

/* Input side of the batcher (apply.py:108-124,278-284: TensorChunk(...).padded(valid) of every segment):
 * batch[(j*B + b), c, :] = the `valid` samples centred on segment seg_first + j of the window [offset0,
 * offset0 + length) of track [B, C, track_len]; real signal where the track has it, zeros beyond its ends. */
int bd_gather_segments(const float* track, float* batch, int B, int C, long long track_len, long long offset0,
                       long long length, int seg_first, int nseg_batch, int seg_len, int stride, int valid,
                       void* stream);

/* ---- Hybrid Demucs v3 only (hdemucs.py:123-157,304-335, demucs.py:20-67,157-216) -------------------------------
 * GroupNorm with G groups over channels-last x [B, rows, C] (norm_groups = 4): sums[(b*G + g)*2 + {0,1}] += (sum, sumsq)
 * of group g of item b; finish with bd_finalize_group_stats(sums, mean_rstd, B*G, rows*C/G). */
int bd_gn_stats(const float* x, double* sums, int B, long long rows, int C, int G, void* stream);
/* y[b*y_item_stride + r*Cout + c] = act(GroupNorm(x)[b, row0 + r, :])[c] (+ addend at the same index, or NULL),
 * r < rows_out: act BD_ACT_NONE / BD_ACT_GELU keep C channels, BD_ACT_GLU gives C/2 = value[c] * sigmoid(gate[c + C/2])
 * in the reference's natural channel order.  The row window lets HDecLayer crop AFTER normalising the full transposed-
 * convolution output (hdemucs.py:326-331); addend carries the next layer's skip connection (hdemucs.py:310). */
int bd_gn_act(const float* x, float* y, const float* mean_rstd, const float* gamma, const float* beta,
              const float* addend, int B, long long rows_in, long long row0, long long rows_out, int C, int G, int act,
              long long y_item_stride, void* stream);
/* BLSTM frame split (demucs.py:41-47, utils.py:20-35): frames[(b*nframes + k), j, c] = x[b, k*stride + j, c], zero past T. */
int bd_lstm_frame(const float* x, float* frames, int B, long long T, int C, int nframes, int width, int stride, void* stream);
/* BLSTM un-framing + skip (demucs.py:52-66): out[b, t] = frames[b*nframes + k(t), t - k(t)*stride] + skip[b, t]. */
int bd_lstm_unframe_add(const float* frames, const float* skip, float* out, int B, long long T, int C, int nframes, int width,
                        int stride, void* stream);
/* One bidirectional nn.LSTM layer from its input projections: pre [N, T, 2, 4H] = x W_ih^T + b_ih + b_hh (direction-major,
 * gates i f g o), whhT [2, H, 4H] = W_hh transposed, out [N, T, 2H] = [forward | backward], ws >= 6*N*H floats. */
int bd_lstm_bidir(const float* pre, const float* whhT, float* out, float* ws, int N, int T, int H, void* stream);
/* LocalState core (demucs.py:186-216, heads x (D/heads), ndecay 4, nfreqs 0): qkc [N, T, 3D] = query | key | content,
 * dq [N, T, heads*4] decay logits -> out [N, T, D] (before the output projection). */
int bd_local_state(const float* qkc, const float* dq, float* out, int N, int T, int D, int heads, void* stream);

/* ---- front / back door of the separator (api.py:265-266, audio.py:143-172,175-265) ------------------------------
 * Channel conversion (audio.py:143-166) of x [items, src_ch, len] -> y [items, dst_ch, len]: copy, downmix to mono,
 * replicate mono, or keep the first dst_ch channels. */
int bd_convert_channels(const float* x, float* y, int items, int src_ch, int dst_ch, long long len, void* stream);
/* convert_audio (audio.py:169-172): channel conversion + julius.resample_frac(old_sr -> new_sr) in one pass.
 * old_sr / new_sr are the rates divided by their gcd; kernel [new_sr, 2*width + old_sr] is the windowed-sinc filter
 * bank (demucs_b200/audio.py builds it as julius 0.2.x does: zeros 24, rolloff 0.945, each phase normalised to unit
 * sum); the input is edge-replicated by `width` samples on the left and width + old_sr on the right;
 * Lout <= ceil(Lin*new_sr/old_sr) (julius' default is the floor). */
int bd_resample_frac(const float* x, float* y, const float* kernel, int items, int src_ch, int dst_ch, long long Lin,
                     long long Lout, int old_sr, int new_sr, int width, void* stream);
/* peak[0] = max |x| over n samples (for prevent_clip's rescale mode, audio.py:223-224). */
int bd_absmax(const float* x, float* peak, long long n, void* stream);
/* prevent_clip (audio.py:218-233) + PCM quantisation (i16_pcm, audio.py:175-180) + planar -> interleaved:
 * x [channels, frames] -> out [frames, channels] as int16 (bits 16: clamp to [-1,1], * 32767, truncate), int32 holding
 * a 24-bit value (bits 24, * 8388607) or float (bits 32).  mode: BD_CLIP_*; rescale divides by max(1.01*peak, 1). */
enum { BD_CLIP_NONE = 0, BD_CLIP_RESCALE = 1, BD_CLIP_CLAMP = 2, BD_CLIP_TANH = 3 };
int bd_clip_pcm(const float* x, void* out, int channels, long long frames, int mode, const float* peak, int bits,
                void* stream);
/* The input side of the same wire format: src [frames, src_ch] interleaved little-endian PCM samples (the bytes of a
 * WAV file's data chunk) -> dst[c * dst_ld + frame0 + t], t < frames, c < dst_ch (planar float; frame0 / dst_ld let
 * the chunks of a long file land in one tensor).  Scaling as torchaudio.load(normalize=True) / ffmpeg's f32 output:
 * u8 (x - 128) / 2^7, s16 x / 2^15, packed 3-byte s24 x / 2^23, s32 float_rn(x) / 2^31, f32 as is, f64 rounded to
 * f32.  The channel rule is bd_convert_channels' (the mono down-mix summed in channel order, then divided by src_ch).
 * src is aligned to the sample size (any alignment for s24); a frame is at most 32768 bytes. */
enum { BD_PCM_U8 = 1, BD_PCM_S16 = 2, BD_PCM_S24 = 3, BD_PCM_S32 = 4, BD_PCM_F32 = 5, BD_PCM_F64 = 6 };
int bd_pcm_decode(const void* src, float* dst, int format, int src_ch, int dst_ch, long long frames, long long dst_ld,
                  long long frame0, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DEMUCS_B200_H */
