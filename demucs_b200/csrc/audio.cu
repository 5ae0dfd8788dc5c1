// Front and back door of the separator on the device (reference demucs/audio.py:143-172,175-265, api.py:265-266):
//   * channel conversion + fractional resampling to the model's rate (convert_audio -> julius.resample_frac): a
//     polyphase windowed-sinc FIR, one output sample per thread, the filter bank [new_sr][2*width + old_sr] read
//     through the read-only cache, input edges replicated as julius pads them;
//   * clip prevention (rescale by the global peak / clamp / tanh) and PCM quantisation fused with the planar ->
//     interleaved transpose, so that stems leave the GPU in wire format (2 bytes per sample instead of 4);
//   * the mirror image for input: interleaved PCM bytes of a WAV file's data chunk -> planar float with the channel
//     conversion fused, so that a file crosses PCIe in its own encoding.
// HBM-bound elementwise / short-FIR kernels; nothing here is on the per-segment hot path.
#include "common.cuh"
#include "../../include/demucs_b200.h"

namespace {

// input channel mix of convert_audio_channels (audio.py:143-166): dst == src: copy; dst == 1: mean of all;
// src == 1: replicate; src > dst: the first dst channels
__device__ __forceinline__ float read_channel(const float* __restrict__ x, int src_ch, int dst_ch, int c, long long len,
                                              long long t) {
  if (src_ch == dst_ch || src_ch > dst_ch && dst_ch != 1) return __ldg(x + (size_t)c * len + t);
  if (src_ch == 1) return __ldg(x + t);
  float s = 0.f;                      // dst_ch == 1: downmix
  for (int k = 0; k < src_ch; ++k) s += __ldg(x + (size_t)k * len + t);
  return s / (float)src_ch;
}

__global__ void convert_channels_kernel(const float* __restrict__ x, float* __restrict__ y, int items, int src_ch,
                                        int dst_ch, long long len) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int c = blockIdx.y % dst_ch, b = blockIdx.y / dst_ch;
  if (t >= len) return;
  y[((size_t)b * dst_ch + c) * len + t] = read_channel(x + (size_t)b * src_ch * len, src_ch, dst_ch, c, len, t);
}

// y[b, c, j*new_sr + i] = sum_k kernel[i][k] * xpad[b, c, j*old_sr + k],  xpad[n] = x[clamp(n - width, 0, Lin-1)]
__global__ void resample_frac_kernel(const float* __restrict__ x, float* __restrict__ y, const float* __restrict__ kern,
                                     int src_ch, int dst_ch, long long Lin, long long Lout, int old_sr, int new_sr,
                                     int width) {
  const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int c = blockIdx.y % dst_ch, b = blockIdx.y / dst_ch;
  if (o >= Lout) return;
  const long long j = o / new_sr;
  const int i = (int)(o - j * new_sr);
  const int klen = 2 * width + old_sr;
  const float* kr = kern + (size_t)i * klen;
  const float* xb = x + (size_t)b * src_ch * Lin;
  const long long base = j * old_sr - width;
  float acc = 0.f;
  for (int k = 0; k < klen; ++k) {
    long long n = base + k;
    n = n < 0 ? 0 : (n >= Lin ? Lin - 1 : n);
    acc = fmaf(__ldg(kr + k), read_channel(xb, src_ch, dst_ch, c, Lin, n), acc);
  }
  y[((size_t)b * dst_ch + c) * Lout + o] = acc;
}

__global__ void absmax_kernel(const float* __restrict__ x, unsigned int* __restrict__ out, long long n) {
  float m = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(__ldg(x + i)));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, __float_as_uint(m));      // non-negative floats order like their bits
}

// x [C, T] planar float -> out [T, C] interleaved: int16 (bits 16), int32 holding a 24-bit value (bits 24), float (bits 32)
__global__ void clip_pcm_kernel(const float* __restrict__ x, void* __restrict__ out, int C, long long T, int mode,
                                const unsigned int* __restrict__ peak_bits, int bits) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  float scale = 1.f;
  if (mode == BD_CLIP_RESCALE) scale = 1.0f / fmaxf(1.01f * __uint_as_float(__ldg(peak_bits)), 1.0f);
  for (int c = 0; c < C; ++c) {
    float v = __ldg(x + (size_t)c * T + t);
    if (mode == BD_CLIP_RESCALE) v = v * scale;
    else if (mode == BD_CLIP_CLAMP) v = fminf(fmaxf(v, -0.99f), 0.99f);
    else if (mode == BD_CLIP_TANH) v = tanhf(v);
    const size_t at = (size_t)t * C + c;
    if (bits == 32) {
      reinterpret_cast<float*>(out)[at] = v;
    } else {
      v = fminf(fmaxf(v, -1.f), 1.f);                                    // i16_pcm (audio.py:175-180): clamp, scale,
      if (bits == 16) reinterpret_cast<short*>(out)[at] = (short)(int)(v * 32767.f);      // truncate toward zero
      else reinterpret_cast<int*>(out)[at] = (int)(v * 8388607.f);
    }
  }
}

// One sample of the input, scaled as torchaudio.load(normalize=True) and ffmpeg's f32 output do: integers divided by
// 2^(bits-1) (u8 offset by 128 first), floats as they are (f64 rounded once).  Every product is by a power of two, so
// it is exact.  `p` is aligned to the sample size (s24: byte-wise).
__device__ __forceinline__ float pcm_sample(const unsigned char* p, int format) {
  switch (format) {
    case BD_PCM_U8: return (float)((int)p[0] - 128) * 0x1p-7f;
    case BD_PCM_S16: return (float)*reinterpret_cast<const short*>(p) * 0x1p-15f;
    case BD_PCM_S24: return (float)((int)((unsigned)p[0] << 8 | (unsigned)p[1] << 16 | (unsigned)p[2] << 24) >> 8) * 0x1p-23f;
    case BD_PCM_S32: return __int2float_rn(*reinterpret_cast<const int*>(p)) * 0x1p-31f;
    case BD_PCM_F32: return *reinterpret_cast<const float*>(p);
    default: return __double2float_rn(*reinterpret_cast<const double*>(p));
  }
}

// read_channel on one interleaved frame: the same channel rule, the down-mix summed in the same order
__device__ __forceinline__ float pcm_channel(const unsigned char* frame, int format, int bps, int src_ch, int dst_ch,
                                             int c) {
  if (src_ch == dst_ch || src_ch > dst_ch && dst_ch != 1) return pcm_sample(frame + c * bps, format);
  if (src_ch == 1) return pcm_sample(frame, format);
  float s = 0.f;
  for (int k = 0; k < src_ch; ++k) s += pcm_sample(frame + k * bps, format);
  return s / (float)src_ch;
}

constexpr int kPcmStage = 32768;        // shared-memory bytes of one CTA's frames
constexpr int kPcmTileFrames = 4096;

// A CTA decodes `tile` consecutive frames.  Their bytes are one contiguous run of the input, staged into shared memory
// with 16-byte loads (byte loads only for the partial 16-byte words at the two ends of the run), so 3-byte samples and
// odd channel counts cost no unaligned global loads.  The run keeps its address phase mod 16 in shared memory, so each
// sample is read there with one load of its natural alignment.  Then one coalesced run of floats per output channel.
__global__ void __launch_bounds__(256) pcm_decode_kernel(const unsigned char* __restrict__ src, float* __restrict__ dst,
                                                         int format, int bps, int src_ch, int dst_ch, long long frames,
                                                         long long dst_ld, long long frame0, int tile) {
  __shared__ __align__(16) unsigned char stage[kPcmStage + 16];
  const long long f0 = (long long)blockIdx.x * tile;
  const int nf = (int)min((long long)tile, frames - f0);
  const int fbytes = src_ch * bps;
  const unsigned char* run = src + f0 * fbytes;
  const int head = (int)((uintptr_t)run & 15), end = head + nf * fbytes;
  const unsigned char* base = run - head;            // 16-byte aligned; the run is stage[head, end)
  const int wa = (head + 15) >> 4, wb = end >> 4;     // words [wa, wb) lie wholly inside the run
#pragma unroll 4
  for (int w = wa + threadIdx.x; w < wb; w += blockDim.x)
    reinterpret_cast<uint4*>(stage)[w] = __ldg(reinterpret_cast<const uint4*>(base) + w);
  const int e0 = min(16 * wa, end), e1 = max(16 * wb, 16 * wa);
  for (int i = head + threadIdx.x; i < e0; i += blockDim.x) stage[i] = __ldg(base + i);
  for (int i = e1 + threadIdx.x; i < end; i += blockDim.x) stage[i] = __ldg(base + i);
  __syncthreads();
  const unsigned char* s = stage + head;
  for (int c = 0; c < dst_ch; ++c) {
    float* out = dst + (size_t)c * dst_ld + frame0 + f0;
    for (int f = threadIdx.x; f < nf; f += blockDim.x) out[f] = pcm_channel(s + f * fbytes, format, bps, src_ch, dst_ch, c);
  }
}

}  // namespace

extern "C" {

int bd_convert_channels(const float* x, float* y, int items, int src_ch, int dst_ch, long long len, void* stream) {
  BD_REQUIRE(items > 0 && src_ch > 0 && dst_ch > 0 && len > 0 && items * dst_ch <= 65535, "bd_convert_channels: bad sizes");
  BD_REQUIRE(src_ch == dst_ch || dst_ch == 1 || src_ch == 1 || src_ch >= dst_ch,
             "The audio file has less channels than requested but is not mono.");
  convert_channels_kernel<<<dim3(bd_cdiv(len, 256), items * dst_ch), 256, 0, (cudaStream_t)stream>>>(x, y, items, src_ch,
                                                                                                    dst_ch, len);
  return bd_check_launch("convert_channels_kernel");
}

int bd_resample_frac(const float* x, float* y, const float* kernel, int items, int src_ch, int dst_ch, long long Lin,
                     long long Lout, int old_sr, int new_sr, int width, void* stream) {
  BD_REQUIRE(items > 0 && src_ch > 0 && dst_ch > 0 && Lin > 0 && Lout > 0 && old_sr > 0 && new_sr > 0 && width > 0 &&
                 items * dst_ch <= 65535, "bd_resample_frac: bad sizes");
  BD_REQUIRE(src_ch == dst_ch || dst_ch == 1 || src_ch == 1 || src_ch >= dst_ch,
             "The audio file has less channels than requested but is not mono.");
  BD_REQUIRE(Lout <= (Lin * new_sr + old_sr - 1) / old_sr, "bd_resample_frac: Lout beyond ceil(Lin * new_sr / old_sr)");
  resample_frac_kernel<<<dim3(bd_cdiv(Lout, 256), items * dst_ch), 256, 0, (cudaStream_t)stream>>>(
      x, y, kernel, src_ch, dst_ch, Lin, Lout, old_sr, new_sr, width);
  return bd_check_launch("resample_frac_kernel");
}

int bd_absmax(const float* x, float* peak, long long n, void* stream) {
  BD_REQUIRE(n > 0 && x && peak, "bd_absmax: bad arguments");
  cudaError_t e = cudaMemsetAsync(peak, 0, sizeof(float), (cudaStream_t)stream);
  if (e != cudaSuccess) {
    bd_set_error("bd_absmax: memset: %s", cudaGetErrorString(e));
    return BD_ERR_CUDA;
  }
  long long g = (n + 256 * 8 - 1) / (256 * 8);
  if (g > 148 * 8) g = 148 * 8;
  absmax_kernel<<<(unsigned)g, 256, 0, (cudaStream_t)stream>>>(x, reinterpret_cast<unsigned int*>(peak), n);
  return bd_check_launch("absmax_kernel");
}

int bd_clip_pcm(const float* x, void* out, int channels, long long frames, int mode, const float* peak, int bits,
                void* stream) {
  BD_REQUIRE(channels > 0 && frames > 0, "bd_clip_pcm: bad sizes");
  BD_REQUIRE(bits == 16 || bits == 24 || bits == 32, "bd_clip_pcm: bits must be 16, 24 or 32 (float)");
  BD_REQUIRE(mode >= BD_CLIP_NONE && mode <= BD_CLIP_TANH, "Invalid mode %d", mode);
  BD_REQUIRE(mode != BD_CLIP_RESCALE || peak, "bd_clip_pcm: rescale needs the peak (bd_absmax)");
  clip_pcm_kernel<<<bd_cdiv(frames, 256), 256, 0, (cudaStream_t)stream>>>(x, out, channels, frames, mode,
                                                                          reinterpret_cast<const unsigned int*>(peak), bits);
  return bd_check_launch("clip_pcm_kernel");
}

int bd_pcm_decode(const void* src, float* dst, int format, int src_ch, int dst_ch, long long frames, long long dst_ld,
                  long long frame0, void* stream) {
  BD_REQUIRE(format >= BD_PCM_U8 && format <= BD_PCM_F64, "bd_pcm_decode: unknown format %d", format);
  BD_REQUIRE(src && dst && src_ch > 0 && dst_ch > 0 && frames > 0 && frame0 >= 0 && dst_ld >= frame0 + frames,
             "bd_pcm_decode: bad sizes");
  BD_REQUIRE(src_ch == dst_ch || dst_ch == 1 || src_ch == 1 || src_ch >= dst_ch,
             "The audio file has less channels than requested but is not mono.");
  const int bps = format == BD_PCM_U8 ? 1 : format == BD_PCM_S16 ? 2 : format == BD_PCM_S24 ? 3 : format == BD_PCM_F64 ? 8 : 4;
  BD_REQUIRE((long long)src_ch * bps <= kPcmStage, "bd_pcm_decode: a frame of %d channels is wider than %d bytes", src_ch,
             kPcmStage);
  BD_REQUIRE(bps == 3 || (uintptr_t)src % bps == 0, "bd_pcm_decode: src is not aligned to the %d-byte sample size", bps);
  const int tile = min(kPcmTileFrames, kPcmStage / (src_ch * bps));
  BD_REQUIRE((frames + tile - 1) / tile <= 0x7fffffffLL, "bd_pcm_decode: too many frames");
  pcm_decode_kernel<<<bd_cdiv(frames, tile), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const unsigned char*>(src), dst, format, bps, src_ch, dst_ch, frames, dst_ld, frame0, tile);
  return bd_check_launch("pcm_decode_kernel");
}

}  // extern "C"
