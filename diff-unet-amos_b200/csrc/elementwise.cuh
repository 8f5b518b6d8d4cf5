// Bandwidth-bound kernels of the Diff-UNet inference path (everything that is not a 3x3x3 convolution).
//
// HBM activation layout ("C8-planar"): act[n][c/8][z][y][x][c%8], bf16.  One 16-byte vector = 8 consecutive channels
// of one voxel; a whole 8-channel plane of a volume is contiguous, so every kernel below reads/writes full 128-byte
// lines with 16-byte vector accesses, and the conv kernel's TMA boxes read x-contiguous runs.
#pragma once
#include <cstdint>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "ptx.cuh"

namespace dunet {

struct alignas(16) BF8 {  // 8 consecutive channels of one voxel: 16 bytes of 16-bit floats (bf16 or fp16, see below)
  __nv_bfloat162 v[4];
};

// 16-bit storage format of activations and packed weights, a compile-time switch `H` on every kernel that converts:
//   H = false: bf16 (8 mantissa bits; also the element type of the hi / lo pairs of fp32x3 mode)
//   H = true : fp16 (11 mantissa bits; DUNET_FLAG_FP16) -- the reference's own reduced precision (torch.autocast fp16,
//              test.py:104,119 with cfg/btcv/test.yaml:16); the tensor cores take it at the bf16 rate (kind::f16)
// Pointers stay typed __nv_bfloat16* in both modes: they are 16-bit storage, the kernels know the format.
template <bool H>
__device__ __forceinline__ void bf8_to_float(const BF8& b, float (&f)[8]) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t;
    if constexpr (H) t = __half22float2(*reinterpret_cast<const __half2*>(&b.v[i]));
    else t = __bfloat1622float2(b.v[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
template <bool H>
__device__ __forceinline__ BF8 float_to_bf8(const float (&f)[8]) {
  BF8 b;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if constexpr (H) *reinterpret_cast<__half2*>(&b.v[i]) = __floats2half2_rn(f[2 * i], f[2 * i + 1]);
    else b.v[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  }
  return b;
}
// two floats -> one 32-bit word of two 16-bit values (low half = first) and back
template <bool H>
__device__ __forceinline__ uint32_t pack_16x2(float lo, float hi) {
  if constexpr (H) {
    __half2 v = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
  } else {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
  }
}
template <bool H>
__device__ __forceinline__ float2 unpack_16x2(uint32_t w) {
  if constexpr (H) return __half22float2(*reinterpret_cast<const __half2*>(&w));
  else return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w));
}
template <bool H>
__device__ __forceinline__ float round_16(float v) {
  if constexpr (H) return __half2float(__float2half_rn(v));
  else return __bfloat162float(__float2bfloat16_rn(v));
}

// fp32x3 ("split-bf16") mode: a tensor is a PAIR of C8-planar bf16 tensors, value = hi + lo, where hi = bf16(v) and
// lo = bf16(v - hi) (v - hi is exact in fp32), so the pair carries ~16 mantissa bits.  `lo == nullptr` is the plain
// 16-bit mode everywhere below (fp16 mode never has a low part).
template <bool H>
__device__ __forceinline__ void store_split(__nv_bfloat16* hi, __nv_bfloat16* lo, long long idx8, const float (&f)[8]) {
  const BF8 h = float_to_bf8<H>(f);
  reinterpret_cast<BF8*>(hi)[idx8] = h;
  if constexpr (!H) {
    if (lo) {
      float hf[8], r[8];
      bf8_to_float<false>(h, hf);
#pragma unroll
      for (int j = 0; j < 8; ++j) r[j] = f[j] - hf[j];
      reinterpret_cast<BF8*>(lo)[idx8] = float_to_bf8<false>(r);
    }
  }
}
template <bool H>
__device__ __forceinline__ void load_split(const __nv_bfloat16* hi, const __nv_bfloat16* lo, long long idx8, float (&f)[8]) {
  bf8_to_float<H>(reinterpret_cast<const BF8*>(hi)[idx8], f);
  if constexpr (!H) {
    if (lo) {
      float g[8];
      bf8_to_float<false>(reinterpret_cast<const BF8*>(lo)[idx8], g);
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] += g[j];
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// pack: fp32 NCDHW (two concatenated sources) -> bf16 C8-planar with c_pad channels (zero padded).
// Used for the denoiser input cat([image, x_t]) (reference denoiser.py:298) and for boundary tensors.
// ---------------------------------------------------------------------------------------------------------------
// triple != 0 (split precision, c0 real channels, c1 == 0, bf16): ONE tensor with channels [hi(c0) | lo(c0) | hi(c0) | 0 ..],
// hi = bf16(v), lo = v - hi -- the operand of a ConvW::triple conv (the encoder's first conv).
template <bool H>
__global__ void pack_c8_kernel(const float* __restrict__ src0, int c0, const float* __restrict__ src1, int c1,
                               __nv_bfloat16* __restrict__ dst, __nv_bfloat16* __restrict__ dst_lo, int c_pad, long long vox,
                               int batch, int triple) {
  pdl_wait();
  const int chunks = c_pad / 8;
  long long total = (long long)batch * chunks * vox;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    long long v = i % vox;
    int ck = (int)((i / vox) % chunks);
    int n = (int)(i / (vox * chunks));
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int c = ck * 8 + j;
      float val = 0.f;
      if (triple) {
        if (c < 3 * c0) {
          const float x = src0[((long long)n * c0 + c % c0) * vox + v];
          const float hi = round_16<false>(x);
          val = (c / c0 == 1) ? x - hi : hi;
        }
      } else if (c < c0) val = src0[((long long)n * c0 + c) * vox + v];
      else if (c < c0 + c1) val = src1[((long long)n * c1 + (c - c0)) * vox + v];
      f[j] = val;
    }
    store_split<H>(dst, triple ? nullptr : dst_lo, i, f);
  }
}

// unpack: bf16 C8-planar (hi [+ lo]) -> fp32 NCDHW (first c_out channels).
template <bool H>
__global__ void unpack_c8_kernel(const __nv_bfloat16* __restrict__ src, const __nv_bfloat16* __restrict__ src_lo, int c_pad,
                                 float* __restrict__ dst, int c_out, long long vox, int batch) {
  const int chunks = c_pad / 8;
  long long total = (long long)batch * chunks * vox;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    long long v = i % vox;
    int ck = (int)((i / vox) % chunks);
    int n = (int)(i / (vox * chunks));
    float f[8];
    load_split<H>(src, src_lo, i, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int c = ck * 8 + j;
      if (c < c_out) dst[((long long)n * c_out + c) * vox + v] = f[j];
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// InstanceNorm statistics: per (n, 8-channel chunk) the plane is contiguous; grid = (nseg, batch*chunks).
// partial[(plane*nseg + seg)*16 + {0..7: sum, 8..15: sum of squares}]  (fp32, fixed order -> deterministic)
// ---------------------------------------------------------------------------------------------------------------
constexpr int STATS_THREADS = 256;

template <bool H>
__global__ void __launch_bounds__(STATS_THREADS) in_stats_kernel(const __nv_bfloat16* __restrict__ raw,
                                                                 float* __restrict__ partial, long long vox, int nseg) {
  const int plane = blockIdx.y, seg = blockIdx.x;
  const BF8* p = reinterpret_cast<const BF8*>(raw) + (long long)plane * vox;
  long long per = (vox + nseg - 1) / nseg;
  long long lo = seg * per, hi = min(vox, lo + per);
  float s[8], q[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = q[j] = 0.f;
  for (long long v = lo + threadIdx.x; v < hi; v += STATS_THREADS) {
    float f[8];
    bf8_to_float<H>(p[v], f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      s[j] += f[j];
      q[j] = fmaf(f[j], f[j], q[j]);
    }
  }
  __shared__ float red[STATS_THREADS / 32][16];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s[j] += __shfl_xor_sync(0xffffffffu, s[j], o);
      q[j] += __shfl_xor_sync(0xffffffffu, q[j], o);
    }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      red[warp][j] = s[j];
      red[warp][8 + j] = q[j];
    }
  }
  __syncthreads();
  if (threadIdx.x < 16) {
    float t = 0.f;
    for (int w = 0; w < STATS_THREADS / 32; ++w) t += red[w][threadIdx.x];
    partial[((long long)plane * nseg + seg) * 16 + threadIdx.x] = t;
  }
}

// Split-K epilogue: sum the fp32 partial tiles of the ksplit CTAs in a fixed order, write the bf16 raw conv output and
// the InstanceNorm partial statistics of the (un-rounded) sums.  partial: [ks][plane][vox][8] fp32.
template <bool H>
__global__ void __launch_bounds__(STATS_THREADS) splitk_reduce_stats_kernel(const float* __restrict__ part, int ksplit,
                                                                            long long split_stride /*floats*/,
                                                                            __nv_bfloat16* __restrict__ raw,
                                                                            __nv_bfloat16* __restrict__ raw_lo,
                                                                            float* __restrict__ partial, long long vox,
                                                                            int nseg) {
  pdl_wait();
  const int plane = blockIdx.y, seg = blockIdx.x;
  const float4* p = reinterpret_cast<const float4*>(part) + (long long)plane * vox * 2;
  long long per = (vox + nseg - 1) / nseg;
  long long lo = seg * per, hi = min(vox, lo + per);
  float s[8], q[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = q[j] = 0.f;
  for (long long v = lo + threadIdx.x; v < hi; v += STATS_THREADS) {
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = 0.f;
    for (int k = 0; k < ksplit; ++k) {
      const float4 a0 = p[(long long)k * (split_stride / 4) + v * 2], a1 = p[(long long)k * (split_stride / 4) + v * 2 + 1];
      f[0] += a0.x; f[1] += a0.y; f[2] += a0.z; f[3] += a0.w;
      f[4] += a1.x; f[5] += a1.y; f[6] += a1.z; f[7] += a1.w;
    }
    store_split<H>(raw, raw_lo, (long long)plane * vox + v, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      s[j] += f[j];
      q[j] = fmaf(f[j], f[j], q[j]);
    }
  }
  __shared__ float red[STATS_THREADS / 32][16];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
#pragma unroll
    for (int o2 = 16; o2 > 0; o2 >>= 1) {
      s[j] += __shfl_xor_sync(0xffffffffu, s[j], o2);
      q[j] += __shfl_xor_sync(0xffffffffu, q[j], o2);
    }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      red[warp][j] = s[j];
      red[warp][8 + j] = q[j];
    }
  }
  __syncthreads();
  if (threadIdx.x < 16) {
    float t = 0.f;
    for (int w = 0; w < STATS_THREADS / 32; ++w) t += red[w][threadIdx.x];
    partial[((long long)plane * nseg + seg) * 16 + threadIdx.x] = t;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Fused normalise pass (reference TwoConv / MONAI ADN "NDA", denoiser.py:56-67, 300-304):
//   y = LeakyReLU_0.1( (x - mean) * rsqrt(var + 1e-5) * gamma + beta )  [+ temb bias_c]  [+ encoder feature]
// and, when POOL, the 2x2x2 max-pool of y for the next level (Down, denoiser.py:105-108) in the same pass.
// One read of the raw conv output, one write of y (+1/8 write of the pooled tensor).
// ---------------------------------------------------------------------------------------------------------------
struct NormActArgs {
  const __nv_bfloat16* raw;
  const float* partial;    // InstanceNorm partial statistics [plane][nseg][16] (8 sums, 8 sums of squares per row)
  int nseg;
  const float* gamma;      // [C]
  const float* beta;       // [C]
  const float* bias;       // [C] additive after activation (temb projection) or nullptr
  int bias_n_stride;       // floats between the bias rows of consecutive samples (0: one row for the whole batch)
  const __nv_bfloat16* add;  // C8-planar tensor added after activation (encoder feature) or nullptr
  __nv_bfloat16* out;
  __nv_bfloat16* pooled;   // POOL only
  const __nv_bfloat16 *raw_lo, *add_lo;  // fp32x3 mode: low parts (all four set, or all nullptr)
  __nv_bfloat16 *out_lo, *pooled_lo;
  int out_single_h;        // fp32x3 kernels only: write `out` as ONE fp16 tensor (out_lo unused) -- the encoder's feature maps in
                           // fp16 mode: computed in split precision, consumed by the fp16 denoiser (pooled stays a hi + lo pair)
  int chunks;              // C/8
  int D, H, W;
  float eps, slope;
};

constexpr int NORM_THREADS = 256;

// Second stage of the InstanceNorm statistics, done by every consumer block for its own 8 channels: fixed-order fp64
// reduction of the partial rows into the affine map of the normalisation (biased variance, eps inside the sqrt, as
// F.instance_norm).  nseg <= a few hundred rows (one per conv CTA / reduction segment), so this is ~10 KB from L2.
// sc/sh: 8 floats each; scratch: 16*16 doubles.  Needs >= 256 threads; ends with __syncthreads().
// One thread's share of the fixed-order reduction: rows g0, g0 + 16, ... of statistic e.  The loads are issued in batches of ten
// before the first add, so the chain is one L2 round trip per 160 rows instead of one per row (measured: the dependent-load loop
// cost every consumer block ~4 us of prologue at 148 rows); missing rows add +0.0, so the sum is the same as the plain loop's.
__device__ __forceinline__ double stats_row_sum(const float* __restrict__ partial, int nseg, int plane, int g0, int e) {
  const float* __restrict__ p = partial + ((long long)plane * nseg) * 16 + e;
  double acc = 0.0;
  for (int base = g0; base < nseg; base += 160) {
    float v[10];
#pragma unroll
    for (int i = 0; i < 10; ++i) {
      const int g = base + 16 * i;
      v[i] = g < nseg ? __ldcg(p + (long long)g * 16) : 0.f;  // L2: rows written by the kernel this one was pre-launched behind
    }
#pragma unroll
    for (int i = 0; i < 10; ++i) acc += (double)v[i];
  }
  return acc;
}
// second stage for one plane: 16 x 16 partial sums in scratch -> scale / shift of its 8 channels (threads 0..7)
__device__ __forceinline__ void stats_finish(const double* scratch, int plane, const float* __restrict__ gamma,
                                             const float* __restrict__ beta, int chunks, double count, float eps, float* sc,
                                             float* sh, int j) {
  double s = 0.0, q = 0.0;
  for (int g = 0; g < 16; ++g) {
    s += scratch[g * 16 + j];
    q += scratch[g * 16 + 8 + j];
  }
  const int c = (plane % chunks) * 8 + j;
  const double mean = s / count;
  double var = q / count - mean * mean;
  if (var < 0.0) var = 0.0;
  const float rstd = (float)(1.0 / sqrt(var + (double)eps));
  const float scale = rstd * gamma[c];
  sc[j] = scale;
  sh[j] = beta[c] - (float)mean * scale;
}
__device__ __forceinline__ void stats_to_affine(const float* __restrict__ partial, int nseg, int plane,
                                                const float* __restrict__ gamma, const float* __restrict__ beta,
                                                int chunks, double count, float eps, float* sc, float* sh,
                                                double* scratch) {
  if (threadIdx.x < 256) {
    const int e = threadIdx.x & 15, g0 = threadIdx.x >> 4;
    scratch[g0 * 16 + e] = stats_row_sum(partial, nseg, plane, g0, e);
  }
  __syncthreads();
  if (threadIdx.x < 8) stats_finish(scratch, plane, gamma, beta, chunks, count, eps, sc, sh, threadIdx.x);
  __syncthreads();
}
// The same for `np` consecutive planes (the final kernel needs all 64 channels of its sample): four planes per pass, their
// row loads all in flight together.  sc / sh: np * 8 floats; scratch: 4 * 256 doubles.  Same arithmetic, same order per plane.
__device__ __forceinline__ void stats_to_affine_planes(const float* __restrict__ partial, int nseg, int plane0, int np,
                                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                                       int chunks, double count, float eps, float* sc, float* sh,
                                                       double* scratch) {
  for (int k0 = 0; k0 < np; k0 += 4) {
    if (threadIdx.x < 256) {
      const int e = threadIdx.x & 15, g0 = threadIdx.x >> 4;
      if (nseg <= 160) {
        float v[4][10];
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
          for (int i = 0; i < 10; ++i) {
            const int g = g0 + 16 * i;
            v[k][i] = (k0 + k < np && g < nseg) ? __ldcg(partial + ((long long)(plane0 + k0 + k) * nseg + g) * 16 + e) : 0.f;
          }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          double acc = 0.0;
#pragma unroll
          for (int i = 0; i < 10; ++i) acc += (double)v[k][i];
          scratch[k * 256 + g0 * 16 + e] = acc;
        }
      } else {
        for (int k = 0; k < 4 && k0 + k < np; ++k) scratch[k * 256 + g0 * 16 + e] = stats_row_sum(partial, nseg, plane0 + k0 + k, g0, e);
      }
    }
    __syncthreads();
    if (threadIdx.x < 32 && k0 + (threadIdx.x >> 3) < np) {
      const int k = threadIdx.x >> 3, j = threadIdx.x & 7;
      stats_finish(scratch + k * 256, plane0 + k0 + k, gamma, beta, chunks, count, eps, sc + (k0 + k) * 8, sh + (k0 + k) * 8, j);
    }
    __syncthreads();
  }
}

// The affine map alone, for consumers that normalise on load (conv3d_tc64 FUSE): out[plane][16] = scale[8], shift[8].
__global__ void __launch_bounds__(256) in_affine_kernel(const float* __restrict__ partial, int nseg,
                                                        const float* __restrict__ gamma, const float* __restrict__ beta,
                                                        int chunks, double count, float eps, float* __restrict__ out) {
  __shared__ float sc[8], sh[8];
  __shared__ double scratch[256];
  pdl_wait();
  stats_to_affine(partial, nseg, blockIdx.x, gamma, beta, chunks, count, eps, sc, sh, scratch);
  if (threadIdx.x < 8) {
    out[blockIdx.x * 16 + threadIdx.x] = sc[threadIdx.x];
    out[blockIdx.x * 16 + 8 + threadIdx.x] = sh[threadIdx.x];
  }
}

__device__ __forceinline__ void norm_prologue(const NormActArgs& a, int plane, float* sc, float* sh, float* bi,
                                              double* scratch) {
  if (threadIdx.x < 8)
    bi[threadIdx.x] = a.bias ? a.bias[(long long)(plane / a.chunks) * a.bias_n_stride + (plane % a.chunks) * 8 + threadIdx.x] : 0.f;
  stats_to_affine(a.partial, a.nseg, plane, a.gamma, a.beta, a.chunks, (double)a.D * a.H * a.W, a.eps, sc, sh, scratch);
}

__device__ __forceinline__ void norm_apply(float (&f)[8], const float* sc, const float* sh, const float* bi,
                                           float slope) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float y = fmaf(f[j], sc[j], sh[j]);
    y = fmaxf(y, y * slope);  // LeakyReLU for 0 < slope < 1
    f[j] = y + bi[j];
  }
}

// ADD: the encoder-feature residual is present (in the tensor's own format).  MODE: 0 = bf16, 1 = fp32x3 (hi + lo pairs in
// and out; with out_single_h the output is one fp16 tensor instead), 2 = fp16.
// All variants keep 4 independent 16-byte loads per tensor in flight per thread; __launch_bounds__ asks for 3-4 resident
// blocks per SM so ~64 KB of loads are outstanding per SM.
constexpr int MODE_BF16 = 0, MODE_FP32X3 = 1, MODE_FP16 = 2;

template <bool ADD, int MODE>
__global__ void __launch_bounds__(NORM_THREADS, (ADD || MODE == MODE_FP32X3) ? 3 : 4) norm_act_kernel(NormActArgs a) {
  constexpr bool PREC = MODE == MODE_FP32X3, H = MODE == MODE_FP16;
  constexpr bool ADD_PAIR = ADD && PREC, ADD_H = H;
  __shared__ float sc[8], sh[8], bi[8];
  __shared__ double scratch[256];
  const int plane = blockIdx.y;  // n*chunks + chunk
  pdl_wait();
  norm_prologue(a, plane, sc, sh, bi, scratch);
  const long long vox = (long long)a.D * a.H * a.W;
  const BF8* __restrict__ in = reinterpret_cast<const BF8*>(a.raw) + plane * vox;
  const BF8* __restrict__ add = reinterpret_cast<const BF8*>(a.add) + plane * vox;
  const BF8* __restrict__ in_lo = reinterpret_cast<const BF8*>(a.raw_lo) + plane * vox;
  const BF8* __restrict__ add_lo = reinterpret_cast<const BF8*>(a.add_lo) + plane * vox;
  constexpr int U = PREC ? 2 : 4;
  const long long stride = (long long)gridDim.x * NORM_THREADS;
  for (long long v0 = blockIdx.x * (long long)NORM_THREADS + threadIdx.x; v0 < vox; v0 += stride * U) {
    BF8 xin[U], ain[U], xlo[U], alo[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long v = v0 + u * stride;
      if (v < vox) {
        xin[u] = in[v];
        if constexpr (PREC) xlo[u] = in_lo[v];
        if constexpr (ADD) ain[u] = add[v];
        if constexpr (ADD_PAIR) alo[u] = add_lo[v];
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const long long v = v0 + u * stride;
      if (v < vox) {
        float f[8];
        bf8_to_float<H>(xin[u], f);
        if constexpr (PREC) {
          float g[8];
          bf8_to_float<false>(xlo[u], g);
#pragma unroll
          for (int j = 0; j < 8; ++j) f[j] += g[j];
        }
        norm_apply(f, sc, sh, bi, a.slope);
        if constexpr (ADD) {
          float g[8];
          bf8_to_float<ADD_H>(ain[u], g);
          if constexpr (ADD_PAIR) {
            float h[8];
            bf8_to_float<false>(alo[u], h);
#pragma unroll
            for (int j = 0; j < 8; ++j) g[j] += h[j];
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) f[j] += g[j];
        }
        if (PREC && a.out_single_h) reinterpret_cast<BF8*>(a.out)[plane * vox + v] = float_to_bf8<true>(f);
        else store_split<H>(a.out, PREC ? a.out_lo : nullptr, plane * vox + v, f);
      }
    }
  }
}

// Same pass + the 2x2x2 max-pool of the result (Down, denoiser.py:105-108).  thread = (x, y/2, z/2): it handles the four
// (dz, dy) voxels at its x (lanes run along x: every load/store instruction covers 512 contiguous bytes) and completes
// the pool with its x^1 neighbour through a shuffle; the pooled tensor is built from the ROUNDED outputs (16-bit, or the
// hi + lo sum in fp32x3 mode) so that pooled == maxpool(out) exactly.
// with the residual the kernel holds 8 independent 16-byte loads per thread: at 3 blocks / SM (<= 85 registers) ptxas spills
// 40-52 bytes into the hot loop; 2 blocks / SM (96 registers, no spills, still 64 KB of loads in flight per SM) measured
// 4.68 vs 4.24 TB/s on the 96^3 launches
#ifndef DUNET_NORM_POOL_ADD_MINB
#define DUNET_NORM_POOL_ADD_MINB 2
#endif
template <bool ADD, int MODE>
__global__ void __launch_bounds__(NORM_THREADS, MODE == MODE_FP32X3 ? 2 : (ADD ? DUNET_NORM_POOL_ADD_MINB : 3)) norm_act_pool_kernel(NormActArgs a) {
  constexpr bool PREC = MODE == MODE_FP32X3, H = MODE == MODE_FP16;
  constexpr bool ADD_PAIR = ADD && PREC, ADD_H = H;
  __shared__ float sc[8], sh[8], bi[8];
  __shared__ double scratch[256];
  const int plane = blockIdx.y;
  pdl_wait();
  norm_prologue(a, plane, sc, sh, bi, scratch);
  const long long vox = (long long)a.D * a.H * a.W;
  const BF8* __restrict__ in = reinterpret_cast<const BF8*>(a.raw) + plane * vox;
  const BF8* __restrict__ add = reinterpret_cast<const BF8*>(a.add) + plane * vox;
  const BF8* __restrict__ in_lo = reinterpret_cast<const BF8*>(a.raw_lo) + plane * vox;
  const BF8* __restrict__ add_lo = reinterpret_cast<const BF8*>(a.add_lo) + plane * vox;
  BF8* __restrict__ out = reinterpret_cast<BF8*>(a.out) + plane * vox;
  BF8* __restrict__ out_lo = reinterpret_cast<BF8*>(a.out_lo) + plane * vox;
  const int D2 = a.D / 2, H2 = a.H / 2, W2 = a.W / 2;
  const long long pvox = (long long)D2 * H2 * W2;
  const long long total = (long long)D2 * H2 * a.W;  // even: W is even
  const int lane = threadIdx.x & 31;
  for (long long p = blockIdx.x * (long long)NORM_THREADS + threadIdx.x; p - lane < total;
       p += (long long)gridDim.x * NORM_THREADS) {
    const bool valid = p < total;
    const int x = (int)(p % a.W), y2 = (int)((p / a.W) % H2), z2 = (int)(p / ((long long)a.W * H2));
    BF8 xin[4], ain[4], xlo[4], alo[4];
    unsigned vv[4];  // voxel offsets inside one 8-channel plane (< 2^31: checked on the host), 32-bit to save registers
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      vv[k] = ((unsigned)(2 * z2 + (k >> 1)) * (unsigned)a.H + (unsigned)(2 * y2 + (k & 1))) * (unsigned)a.W + (unsigned)x;
      if (valid) {
        xin[k] = in[vv[k]];
        if constexpr (PREC) xlo[k] = in_lo[vv[k]];
        if constexpr (ADD) ain[k] = add[vv[k]];
        if constexpr (ADD_PAIR) alo[k] = add_lo[vv[k]];
      }
    }
    float m[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) m[j] = -INFINITY;
    if (valid) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float f[8];
        bf8_to_float<H>(xin[k], f);
        if constexpr (PREC) {
          float g[8];
          bf8_to_float<false>(xlo[k], g);
#pragma unroll
          for (int j = 0; j < 8; ++j) f[j] += g[j];
        }
        norm_apply(f, sc, sh, bi, a.slope);
        if constexpr (ADD) {
          float g[8];
          bf8_to_float<ADD_H>(ain[k], g);
          if constexpr (ADD_PAIR) {
            float h[8];
            bf8_to_float<false>(alo[k], h);
#pragma unroll
            for (int j = 0; j < 8; ++j) g[j] += h[j];
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) f[j] += g[j];
        }
        const bool single_h = PREC && a.out_single_h;  // warp-uniform
        const BF8 o = single_h ? float_to_bf8<true>(f) : float_to_bf8<H>(f);
        out[vv[k]] = o;
        float r[8];
        if (single_h) {  // the pooled pair is formed from the un-rounded values (the reference pools fp32 activations)
#pragma unroll
          for (int j = 0; j < 8; ++j) r[j] = f[j];
        } else {
          bf8_to_float<H>(o, r);
        }
        if (PREC && !single_h) {
          float d[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) d[j] = f[j] - r[j];
          const BF8 ol = float_to_bf8<false>(d);
          out_lo[vv[k]] = ol;
          float rl[8];
          bf8_to_float<false>(ol, rl);
#pragma unroll
          for (int j = 0; j < 8; ++j) r[j] += rl[j];
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) m[j] = fmaxf(m[j], r[j]);
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) m[j] = fmaxf(m[j], __shfl_xor_sync(0xffffffffu, m[j], 1));
    if (valid && !(x & 1))
      store_split<H>(a.pooled, PREC ? a.pooled_lo : nullptr, plane * pvox + ((long long)z2 * H2 + y2) * W2 + (x >> 1), m);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Split-K epilogue FUSED with the normalise pass, for the deepest levels (<= 2048 voxels per sample: 12^3, 6^3 of a 96^3
// window).  One block owns one (sample, 8-channel plane): it sums the fp32 K-split partial tiles in a fixed order into
// registers, reduces the InstanceNorm statistics of the plane on the spot (the whole plane is in this block), and writes
// y = LeakyReLU(norm(x)) [+ temb bias] [+ encoder feature] (and its 2x2x2 max-pool) directly -- replacing
// splitk_reduce_stats_kernel + norm_act(_pool)_kernel and the 16-bit round trip of the raw conv output between them
// (two launch-latency-bound launches per layer; same reference lines as norm_act_kernel).
// ---------------------------------------------------------------------------------------------------------------
struct SplitkNormArgs {
  const float* part;        // [ks][plane][vox][8] fp32
  int ksplit;
  long long split_stride;   // floats between consecutive K-split buffers
  NormActArgs n;            // raw / partial / nseg unused
};
constexpr int SKN_VPT = 8;                  // voxels per thread
constexpr int SKN_MAX_VOX = 256 * SKN_VPT;  // 2048

template <bool ADD, bool POOL, bool H>
__global__ void __launch_bounds__(256) splitk_norm_kernel(SplitkNormArgs a) {
  __shared__ float sc[8], sh[8], bi[8];
  __shared__ double red[8][16];
  __shared__ BF8 tile[POOL ? SKN_MAX_VOX : 1];
  const int plane = blockIdx.x;
  const int vox = a.n.D * a.n.H * a.n.W;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  pdl_wait();
  if (threadIdx.x < 8)
    bi[threadIdx.x] = a.n.bias ? a.n.bias[(long long)(plane / a.n.chunks) * a.n.bias_n_stride + (plane % a.n.chunks) * 8 + threadIdx.x] : 0.f;
  const float4* __restrict__ p = reinterpret_cast<const float4*>(a.part) + (long long)plane * vox * 2;
  const long long kstride = a.split_stride / 4;
  float f[SKN_VPT][8];
  float s[8], q[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = q[j] = 0.f;
#pragma unroll
  for (int u = 0; u < SKN_VPT; ++u) {
    const int v = threadIdx.x + u * 256;
#pragma unroll
    for (int j = 0; j < 8; ++j) f[u][j] = 0.f;
    if (v < vox) {
      for (int k = 0; k < a.ksplit; ++k) {
        const float4 a0 = __ldcg(p + k * kstride + v * 2), a1 = __ldcg(p + k * kstride + v * 2 + 1);
        f[u][0] += a0.x; f[u][1] += a0.y; f[u][2] += a0.z; f[u][3] += a0.w;
        f[u][4] += a1.x; f[u][5] += a1.y; f[u][6] += a1.z; f[u][7] += a1.w;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        s[j] += f[u][j];
        q[j] = fmaf(f[u][j], f[u][j], q[j]);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
#pragma unroll
    for (int o2 = 16; o2 > 0; o2 >>= 1) {
      s[j] += __shfl_xor_sync(0xffffffffu, s[j], o2);
      q[j] += __shfl_xor_sync(0xffffffffu, q[j], o2);
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      red[warp][j] = (double)s[j];
      red[warp][8 + j] = (double)q[j];
    }
  }
  __syncthreads();
  if (threadIdx.x < 8) {
    double ts = 0.0, tq = 0.0;
    for (int w = 0; w < 8; ++w) {
      ts += red[w][threadIdx.x];
      tq += red[w][8 + threadIdx.x];
    }
    const int c = (plane % a.n.chunks) * 8 + threadIdx.x;
    const double mean = ts / (double)vox;
    double var = tq / (double)vox - mean * mean;
    if (var < 0.0) var = 0.0;
    const float rstd = (float)(1.0 / sqrt(var + (double)a.n.eps));
    const float scale = rstd * a.n.gamma[c];
    sc[threadIdx.x] = scale;
    sh[threadIdx.x] = a.n.beta[c] - (float)mean * scale;
  }
  __syncthreads();
  const BF8* __restrict__ add = reinterpret_cast<const BF8*>(a.n.add) + (long long)plane * vox;
  BF8* __restrict__ out = reinterpret_cast<BF8*>(a.n.out) + (long long)plane * vox;
#pragma unroll
  for (int u = 0; u < SKN_VPT; ++u) {
    const int v = threadIdx.x + u * 256;
    if (v < vox) {
      norm_apply(f[u], sc, sh, bi, a.n.slope);
      if constexpr (ADD) {
        float g[8];
        bf8_to_float<H>(add[v], g);
#pragma unroll
        for (int j = 0; j < 8; ++j) f[u][j] += g[j];
      }
      const BF8 o = float_to_bf8<H>(f[u]);
      out[v] = o;
      if constexpr (POOL) tile[v] = o;
    }
  }
  if constexpr (POOL) {  // pooled == maxpool(out) of the ROUNDED outputs, as in norm_act_pool_kernel
    __syncthreads();
    const int D2 = a.n.D / 2, H2 = a.n.H / 2, W2 = a.n.W / 2;
    const int pvox = D2 * H2 * W2;
    for (int pv = threadIdx.x; pv < pvox; pv += 256) {
      const int x2 = pv % W2, y2 = (pv / W2) % H2, z2 = pv / (W2 * H2);
      float m[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) m[j] = -INFINITY;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        float r[8];
        bf8_to_float<H>(tile[((2 * z2 + (k >> 2)) * a.n.H + 2 * y2 + ((k >> 1) & 1)) * a.n.W + 2 * x2 + (k & 1)], r);
#pragma unroll
        for (int j = 0; j < 8; ++j) m[j] = fmaxf(m[j], r[j]);
      }
      store_split<H>(a.n.pooled, nullptr, (long long)plane * pvox + pv, m);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// ConvTranspose3d k=2 s=2 + bias (MONAI UpSample "deconv", denoiser.py:161-170,181).  CUDA-core version:
// thread = (input voxel, tap, 8 output channels).  weights packed [tap][cin][cout] bf16.
// ---------------------------------------------------------------------------------------------------------------
template <bool HF>
__global__ void __launch_bounds__(256) deconv2_kernel(const __nv_bfloat16* __restrict__ in, int cin,
                                                      const __nv_bfloat16* __restrict__ w, const float* __restrict__ b,
                                                      __nv_bfloat16* __restrict__ out, int cout, int D, int H, int W,
                                                      int batch) {
  const long long vox = (long long)D * H * W;
  const int och = cout / 8, ich = cin / 8;
  const long long total = (long long)batch * och * 8 * vox;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long v = i % vox;
    const int tap = (int)((i / vox) % 8);
    const int oc = (int)((i / (vox * 8)) % och);
    const int n = (int)(i / (vox * 8 * och));
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = b[oc * 8 + j];
    const BF8* ip = reinterpret_cast<const BF8*>(in) + (long long)n * ich * vox + v;
    const BF8* wp = reinterpret_cast<const BF8*>(w) + ((long long)tap * cin) * och + oc;
    for (int ic = 0; ic < ich; ++ic) {
      float xi[8];
      bf8_to_float<HF>(ip[(long long)ic * vox], xi);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        float wk[8];
        bf8_to_float<HF>(wp[(long long)(ic * 8 + k) * och], wk);
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = fmaf(xi[k], wk[j], acc[j]);
      }
    }
    const int x = (int)(v % W), y = (int)((v / W) % H), z = (int)(v / ((long long)W * H));
    const int dz = tap >> 2, dy = (tap >> 1) & 1, dx = tap & 1;
    const long long ov = ((long long)(2 * z + dz) * (2 * H) + (2 * y + dy)) * (2 * W) + (2 * x + dx);
    reinterpret_cast<BF8*>(out)[((long long)n * och + oc) * (vox * 8) + ov] = float_to_bf8<HF>(acc);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// final 1x1x1 conv (denoiser.py:282,311) fused with
//   * the InstanceNorm + LeakyReLU of its input (the last TwoConv's normalise pass: u1 never goes to HBM),
//   * the DDIM update (gaussian_diffusion.py:292-297 clamp, :345-349 eps, :566-584 eta = 0 step),
//   * the ensemble accumulation (models/diffusion/diffusion.py:94-98),
//   * the re-pack of the next step's bf16 conv input.
// The [voxels x F] x [F x C] product runs on warp-level bf16 MMAs (m16n8k16) with the fp32 weights split into
// hi + lo bf16 parts (two MMAs) so the weights keep ~16 mantissa bits; everything else is plain fp32.
// The kernel is HBM-bound (reads the 64-channel feature map once, reads/writes the fp32 state once).
//
// Packed denoiser-input channel order: [x_0 .. x_{C-1}, image_0 .. image_{in_ch-1}, 0 ...]  (the reference's
// cat([image, x]) order is restored by permuting the first conv's input channels when its weights are packed), so a
// thread's two adjacent classes form one aligned 4-byte store.  The re-pack rewrites the class tiles (channels < 8 * NT)
// only: image channels inside them are rewritten every step, those past them keep what ddim_init_kernel wrote.
// MC (in_ch > 1) reads each image channel where it is stored; MC = false keeps the single-channel path's one
// hoisted image load per voxel.
// ---------------------------------------------------------------------------------------------------------------
struct FinalDdimArgs {
  const __nv_bfloat16* feat;  // RAW output of the last conv (or, with partial == nullptr, the activated u1), C8-planar
  const __nv_bfloat16* feat_lo;  // fp32x3 mode: low part of feat
  __nv_bfloat16* next_in_lo;     // fp32x3 mode: low part of next_in
  int F;                      // feature channels (multiple of 16, <= 128)
  const float* partial;       // InstanceNorm partial statistics of `feat` [n*F/8 + chunk][nseg][16] or nullptr
  int nseg;
  const float* gamma;
  const float* beta;
  float eps, slope;
  const float* w;             // [C][F] fp32
  const float* b;             // [C]
  int C;
  const float* image;         // [B][in_ch][vox] fp32
  float* x_t;                 // DDIM state, VOXEL-MAJOR fp32 [B][vox][8*NT], updated in place (nullptr: logits only)
  float* acc;                 // sum of clamped x0, same voxel-major layout, += clamp(logits)
  float* logits_out;          // optional [B][C][vox]
  __nv_bfloat16* next_in;     // optional packed [x_prev, image.., 0..] with in_pad channels
  int in_pad;
  long long vox;
  int batch;
  float r, m, abp;            // sqrt_recip_alphas_cumprod[i], sqrt_recipm1_alphas_cumprod[i], alphas_cumprod_prev[i]
  int in_ch;                  // image channels (1 unless MC)
};

constexpr int FINAL_MAX_C = 32;
constexpr int FINAL_MAX_F = 128;
constexpr int FINAL_THREADS = 256;

template <bool H>
__device__ __forceinline__ void mma_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  if constexpr (H)
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  else
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// NT = number of 8-class column tiles (C <= 8 * NT); NKS = F / 16 k-steps; MC = more than one image channel
template <int NT, int NKS, int MODE, bool MC>
__global__ void __launch_bounds__(FINAL_THREADS) final_ddim_kernel(FinalDdimArgs a) {
  constexpr bool PREC = MODE == MODE_FP32X3, H = MODE == MODE_FP16;
  // B fragments of the weights: [k-step][n-tile][hi|lo][b0|b1][lane]
  __shared__ uint32_t wfrag[(FINAL_MAX_F / 16) * NT * 2 * 2 * 32];
  __shared__ float sbias[NT * 8];
  __shared__ __align__(8) float nsc[FINAL_MAX_F], nsh[FINAL_MAX_F];
  __shared__ double scratch[4 * 256];
  constexpr int nks = NKS;
  const int fch = a.F / 8;
  const int n = blockIdx.y;
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  for (int i = threadIdx.x; i < nks * NT * 32; i += FINAL_THREADS) {
    const int l = i & 31, nt = (i >> 5) % NT, ks = i / (32 * NT);
    const int cls = nt * 8 + (l >> 2), k0 = ks * 16 + 2 * (l & 3);
    float wv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + (j & 1) + (j >> 1) * 8;
      wv[j] = cls < a.C ? a.w[cls * a.F + k] : 0.f;
    }
    float hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      hi[j] = round_16<H>(wv[j]);
      lo[j] = wv[j] - hi[j];
    }
    uint32_t* dst = wfrag + ((ks * NT + nt) * 4) * 32 + l;
    dst[0] = pack_16x2<H>(hi[0], hi[1]);
    dst[32] = pack_16x2<H>(hi[2], hi[3]);
    dst[64] = pack_16x2<H>(lo[0], lo[1]);
    dst[96] = pack_16x2<H>(lo[2], lo[3]);
  }
  for (int i = threadIdx.x; i < NT * 8; i += FINAL_THREADS) sbias[i] = i < a.C ? a.b[i] : 0.f;
  pdl_wait();  // the weight fragments above are plan constants; everything below depends on the previous kernels
  if (a.partial) stats_to_affine_planes(a.partial, a.nseg, n * fch, fch, a.gamma, a.beta, fch, (double)a.vox, a.eps, nsc, nsh, scratch);
  __syncthreads();

  const float s_abp = sqrtf(a.abp), s_1mabp = sqrtf(1.f - a.abp - 0.f);
  // All per-sample bases are formed once (64-bit); inside the loop only 32-bit element offsets are computed.
  // (voxels per window < 2^26 and every per-sample tensor < 2^31 elements: checked on the host.)
  const unsigned vox = (unsigned)a.vox;
  const uint32_t* __restrict__ fw = reinterpret_cast<const uint32_t*>(a.feat) + (size_t)n * fch * vox * 4 + t;
  const uint32_t* __restrict__ fw_lo = reinterpret_cast<const uint32_t*>(a.feat_lo) + (size_t)n * fch * vox * 4 + t;
  const float* __restrict__ img_n = a.image ? a.image + (size_t)n * (MC ? a.in_ch : 1) * vox : nullptr;
  // voxel-major state: a quad of lanes (t = 0..3) covers 8 consecutive classes of one voxel with float2 accesses, so
  // the 8 voxels x NT*8 classes a warp touches per access form one contiguous run
  float2* xt_n = a.x_t ? reinterpret_cast<float2*>(a.x_t) + (size_t)n * vox * (NT * 4) + t : nullptr;
  float2* acc_n = a.acc ? reinterpret_cast<float2*>(a.acc) + (size_t)n * vox * (NT * 4) + t : nullptr;
  float* lg_n = a.logits_out ? a.logits_out + (size_t)n * a.C * vox : nullptr;
  uint32_t* np_n = a.next_in ? reinterpret_cast<uint32_t*>(a.next_in) + (size_t)n * (a.in_pad / 8) * vox * 4 + t : nullptr;
  uint32_t* np_lo_n = (PREC && a.next_in) ? reinterpret_cast<uint32_t*>(a.next_in_lo) + (size_t)n * (a.in_pad / 8) * vox * 4 + t : nullptr;
  unsigned cls_off[NT][2];
  bool cls_ok[NT][2], cls_img[NT][2];
#pragma unroll
  for (int nt = 0; nt < NT; ++nt)
#pragma unroll
    for (int b = 0; b < 2; ++b) {
      const int cls = nt * 8 + 2 * t + b;
      cls_ok[nt][b] = cls < a.C;
      cls_img[nt][b] = MC ? (cls >= a.C && cls < a.C + a.in_ch) : cls == a.C;
      cls_off[nt][b] = (unsigned)cls * vox;
    }
  const unsigned warps = gridDim.x * (FINAL_THREADS / 32);
  const unsigned warp_id = blockIdx.x * (FINAL_THREADS / 32) + (threadIdx.x >> 5);
  const unsigned ngroups = (vox + 15) / 16;
  for (unsigned grp = warp_id; grp < ngroups; grp += warps) {
    const unsigned v0 = grp * 16 + g, v1 = v0 + 8;
    const bool ok0 = v0 < vox, ok1 = v1 < vox;
    // ---- issue every load of this group up front: state (independent of the MMAs), image, features
    float2 xt[NT][2], ac[NT][2];  // [class tile][voxel v0 | v1] = classes (2t, 2t+1)
    if (xt_n) {
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        xt[nt][0] = ok0 ? xt_n[v0 * (NT * 4) + nt * 4] : make_float2(0.f, 0.f);
        xt[nt][1] = ok1 ? xt_n[v1 * (NT * 4) + nt * 4] : make_float2(0.f, 0.f);
        ac[nt][0] = ok0 ? acc_n[v0 * (NT * 4) + nt * 4] : make_float2(0.f, 0.f);
        ac[nt][1] = ok1 ? acc_n[v1 * (NT * 4) + nt * 4] : make_float2(0.f, 0.f);
      }
    }
    const float img0 = (!MC && np_n && ok0) ? img_n[v0] : 0.f;
    const float img1 = (!MC && np_n && ok1) ? img_n[v1] : 0.f;
    // A fragments: rows (voxels) v0 / v1, channel pairs (2t, 2t+1) of chunk 2ks and of chunk 2ks+1
    uint32_t af[NKS][4], al[PREC ? NKS : 1][4];
#pragma unroll
    for (int ks = 0; ks < NKS; ++ks) {
      const unsigned c0 = (2 * ks) * vox, c1 = c0 + vox;
      af[ks][0] = ok0 ? __ldg(fw + (c0 + v0) * 4) : 0u;
      af[ks][1] = ok1 ? __ldg(fw + (c0 + v1) * 4) : 0u;
      af[ks][2] = ok0 ? __ldg(fw + (c1 + v0) * 4) : 0u;
      af[ks][3] = ok1 ? __ldg(fw + (c1 + v1) * 4) : 0u;
      if constexpr (PREC) {
        al[ks][0] = ok0 ? __ldg(fw_lo + (c0 + v0) * 4) : 0u;
        al[ks][1] = ok1 ? __ldg(fw_lo + (c0 + v1) * 4) : 0u;
        al[ks][2] = ok0 ? __ldg(fw_lo + (c1 + v0) * 4) : 0u;
        al[ks][3] = ok1 ? __ldg(fw_lo + (c1 + v1) * 4) : 0u;
      }
    }
    float d[NT][4];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      d[nt][0] = d[nt][2] = sbias[nt * 8 + 2 * t];
      d[nt][1] = d[nt][3] = sbias[nt * 8 + 2 * t + 1];
    }
#pragma unroll
    for (int ks = 0; ks < NKS; ++ks) {
      if (a.partial) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int c = ks * 16 + (j >> 1) * 8 + 2 * t;
          float2 x = unpack_16x2<H>(af[ks][j]);
          if constexpr (PREC) {
            const float2 xl = unpack_16x2<false>(al[ks][j]);
            x.x += xl.x; x.y += xl.y;
          }
          const float2 sc2 = *reinterpret_cast<const float2*>(nsc + c), sh2 = *reinterpret_cast<const float2*>(nsh + c);
          float y0 = fmaf(x.x, sc2.x, sh2.x), y1 = fmaf(x.y, sc2.y, sh2.y);
          y0 = fmaxf(y0, y0 * a.slope);  // LeakyReLU with 0 < slope < 1
          y1 = fmaxf(y1, y1 * a.slope);
          af[ks][j] = pack_16x2<H>(y0, y1);
          if constexpr (PREC) {
            const float2 h = unpack_16x2<false>(af[ks][j]);
            al[ks][j] = pack_16x2<false>(y0 - h.x, y1 - h.y);
          }
        }
      }
#pragma unroll
      for (int nt = 0; nt < NT; ++nt) {
        const uint32_t* wf = wfrag + ((ks * NT + nt) * 4) * 32 + lane;
        mma_16816<H>(d[nt], af[ks], wf[0], wf[32]);
        mma_16816<H>(d[nt], af[ks], wf[64], wf[96]);
        if constexpr (PREC) mma_16816<false>(d[nt], al[ks], wf[0], wf[32]);
      }
    }
    // d[nt][0..1]: voxel v0, classes nt*8 + 2t, +1 ; d[nt][2..3]: voxel v1, same classes
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      float nxt[4];
      float xp4[4], ac4[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const bool okv = (j >> 1) ? ok1 : ok0;
        const float xin = (j & 1) ? xt[nt][j >> 1].y : xt[nt][j >> 1].x;
        const float ain = (j & 1) ? ac[nt][j >> 1].y : ac[nt][j >> 1].x;
        float val;
        if constexpr (MC)  // image channel cls - C of this voxel
          val = (cls_img[nt][j & 1] && np_n && okv) ? img_n[(unsigned)(nt * 8 + 2 * t + (j & 1) - a.C) * vox + ((j >> 1) ? v1 : v0)] : 0.f;
        else
          val = cls_img[nt][j & 1] ? ((j >> 1) ? img1 : img0) : 0.f;
        xp4[j] = 0.f;
        ac4[j] = 0.f;
        if (cls_ok[nt][j & 1] && okv) {
          const float lg = d[nt][j];
          if (lg_n) lg_n[cls_off[nt][j & 1] + ((j >> 1) ? v1 : v0)] = lg;
          if (xt_n) {
            const float x0 = fminf(fmaxf(lg, -1.f), 1.f);
            const float eps = (a.r * xin - x0) / a.m;
            const float xp = x0 * s_abp + s_1mabp * eps;
            xp4[j] = xp;
            ac4[j] = ain + x0;
            val = xp;
          }
        }
        nxt[j] = val;
      }
      if (xt_n) {
        if (ok0) { xt_n[v0 * (NT * 4) + nt * 4] = make_float2(xp4[0], xp4[1]); acc_n[v0 * (NT * 4) + nt * 4] = make_float2(ac4[0], ac4[1]); }
        if (ok1) { xt_n[v1 * (NT * 4) + nt * 4] = make_float2(xp4[2], xp4[3]); acc_n[v1 * (NT * 4) + nt * 4] = make_float2(ac4[2], ac4[3]); }
      }
      if (np_n && nt * 8 < a.in_pad) {
        const uint32_t h0 = pack_16x2<H>(nxt[0], nxt[1]), h1 = pack_16x2<H>(nxt[2], nxt[3]);
        if (ok0) np_n[(nt * vox + v0) * 4] = h0;
        if (ok1) np_n[(nt * vox + v1) * 4] = h1;
        if constexpr (PREC) {
          const float2 f0 = unpack_16x2<false>(h0), f1 = unpack_16x2<false>(h1);
          if (ok0) np_lo_n[(nt * vox + v0) * 4] = pack_16x2<false>(nxt[0] - f0.x, nxt[1] - f0.y);
          if (ok1) np_lo_n[(nt * vox + v1) * 4] = pack_16x2<false>(nxt[2] - f1.x, nxt[3] - f1.y);
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// DDIM state layout conversion: voxel-major fp32 [B][vox][CP] -> planar fp32 [B][C][vox] (the reference's NCDHW) for the
// entry points that return planar tensors (the other direction is part of ddim_init_kernel).   thread = (voxel, 4 classes)
// ---------------------------------------------------------------------------------------------------------------
// dst = (accumulate ? dst : 0) + scale * src   (ensemble averaging over independent noise draws)
__global__ void state_from_vm_kernel(const float* __restrict__ src, float* __restrict__ dst, int C, int CP, long long vox, int batch,
                                     float scale, int accumulate) {
  pdl_wait();
  const int q4 = CP / 4;
  const long long total = (long long)batch * vox * q4;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int qd = (int)(i % q4);
    const long long v = (i / q4) % vox;
    const int n = (int)(i / (q4 * vox));
    const float4 f4 = reinterpret_cast<const float4*>(src)[i];
    const float f[4] = {f4.x, f4.y, f4.z, f4.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = qd * 4 + j;
      if (c < C) {
        float* o = dst + ((long long)n * C + c) * vox + v;
        *o = accumulate ? fmaf(scale, f[j], *o) : scale * f[j];
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Start of a DDIM window (gaussian_diffusion.py:690-693 `img = noise or th.randn(shape)`): ONE pass that writes
//   x_t  = the initial noise, voxel-major fp32 [B][vox][CP]      (state read/written by final_ddim_kernel)
//   acc  = 0 (same layout; skipped when `zero_acc == 0`: ensemble draws keep accumulating)
//   next = the packed 16-bit input of the first denoiser conv [x_0 .. x_{C-1}, image_0 .. image_{in_ch-1}, 0 ..]
//          (C8-planar, in_pad channels)
// The noise is either the caller's tensor (planar fp32 [B][C][vox], parity runs) or generated here: Philox4x32-10 keyed by
// `seed`, counter = (element index / 4, window id), Box-Muller -> N(0,1).  Counter-based: a window's noise depends only
// on (seed, window id), not on batching, rank or launch order (multi-GPU runs give identical volumes).
// thread = (sample, voxel, 8-channel chunk).
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
    c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
}
// two uniform 32-bit words -> two independent standard normals (Box-Muller; u1 in (0, 1])
__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float& z0, float& z1) {
  const float u1 = ((float)(a >> 8) + 1.0f) * (1.0f / 16777216.0f);
  const float u2 = (float)(b >> 8) * (1.0f / 16777216.0f);
  const float r = sqrtf(-2.0f * __logf(u1));
  float sn, cs;
  __sincosf(6.283185307179586f * u2, &sn, &cs);
  z0 = r * cs;
  z1 = r * sn;
}
constexpr int INIT_MAX_B = 16;
struct DdimInitArgs {
  const float* noise;      // [B][C][vox] or nullptr (generate)
  const float* image;      // [B][in_ch][vox]
  float* x_t;              // [B][vox][CP]
  float* acc;              // [B][vox][CP]
  __nv_bfloat16* next_in;  // [B][in_pad/8][vox][8]
  __nv_bfloat16* next_in_lo;  // fp32x3 mode or nullptr
  int C, CP, in_pad, batch, zero_acc, in_ch;
  long long vox;
  unsigned long long seed;
  long long ids[INIT_MAX_B];  // noise stream id of each window of the batch
};
template <bool H>
__global__ void __launch_bounds__(256) ddim_init_kernel(DdimInitArgs a) {
  pdl_wait();
  const int nch = (a.CP > a.in_pad ? a.CP : a.in_pad) / 8;
  const long long total = (long long)a.batch * a.vox * nch;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int ck = (int)(i % nch);
    const long long v = (i / nch) % a.vox;
    const int n = (int)(i / (nch * a.vox));
    float f[8];
    if (a.noise) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int c = ck * 8 + j;
        f[j] = c < a.C ? a.noise[((long long)n * a.C + c) * a.vox + v] : 0.f;
      }
    } else {
      const unsigned long long e = (unsigned long long)v * (unsigned)(a.CP / 4) + (unsigned)(ck * 2);  // 4-element group index
      const unsigned long long id = (unsigned long long)a.ids[n];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t c4[4] = {(uint32_t)(e + h), (uint32_t)((e + h) >> 32), (uint32_t)id, (uint32_t)(id >> 32)};
        philox4x32_10(c4, (uint32_t)a.seed, (uint32_t)(a.seed >> 32));
        box_muller(c4[0], c4[1], f[4 * h + 0], f[4 * h + 1]);
        box_muller(c4[2], c4[3], f[4 * h + 2], f[4 * h + 3]);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (ck * 8 + j >= a.C) f[j] = 0.f;
    }
    if (ck * 8 < a.CP) {
      float4* xs = reinterpret_cast<float4*>(a.x_t + ((long long)n * a.vox + v) * a.CP + ck * 8);
      xs[0] = make_float4(f[0], f[1], f[2], f[3]);
      xs[1] = make_float4(f[4], f[5], f[6], f[7]);
      if (a.zero_acc) {
        float4* as = reinterpret_cast<float4*>(a.acc + ((long long)n * a.vox + v) * a.CP + ck * 8);
        as[0] = make_float4(0.f, 0.f, 0.f, 0.f);
        as[1] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    if (ck * 8 < a.in_pad) {
      if (a.C < ck * 8 + 8 && a.C + a.in_ch > ck * 8) {  // packed order [x.., image.., 0..]
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int ic = ck * 8 + j - a.C;
          if (ic >= 0 && ic < a.in_ch) f[j] = a.image[((long long)n * a.in_ch + ic) * a.vox + v];
        }
      }
      store_split<H>(a.next_in, a.next_in_lo, ((long long)n * (a.in_pad / 8) + ck) * a.vox + v, f);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// q(x_t | x_0) of the training forward (GaussianDiffusion.q_sample, gaussian_diffusion.py:187-205, called from
// Diffusion.q_sample, models/diffusion/diffusion.py:65-69):
//   x_t = sqrt_alphas_cumprod[t_n] * x_0 + sqrt_one_minus_alphas_cumprod[t_n] * noise       (per sample n)
// fp32, multiplies and add kept separate (no FMA contraction) so the result is bit-identical to the torch expression.
// noise_in == nullptr: the noise is drawn here (same Philox stream as ddim_init_kernel, id = id0 + n) and written to
// noise_out (the reference returns it: `return sample, t, noise`).
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) q_sample_kernel(const float* __restrict__ x0, const float* __restrict__ noise_in,
                                                       float* __restrict__ noise_out, const long long* __restrict__ t,
                                                       const float* __restrict__ sqrt_ac, const float* __restrict__ sqrt_1mac,
                                                       float* __restrict__ out, long long per_sample, int batch,
                                                       unsigned long long seed, long long id0) {
  const long long groups = (per_sample + 3) / 4;
  const long long total = groups * batch;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i / groups);
    const long long g = i % groups;
    const float a = sqrt_ac[t[n]], b = sqrt_1mac[t[n]];
    float z[4];
    if (!noise_in) {
      const unsigned long long id = (unsigned long long)(id0 + n);
      uint32_t c4[4] = {(uint32_t)g, (uint32_t)((unsigned long long)g >> 32), (uint32_t)id, (uint32_t)(id >> 32)};
      philox4x32_10(c4, (uint32_t)seed, (uint32_t)(seed >> 32));
      box_muller(c4[0], c4[1], z[0], z[1]);
      box_muller(c4[2], c4[3], z[2], z[3]);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const long long e = g * 4 + j;
      if (e < per_sample) {
        const long long o = (long long)n * per_sample + e;
        const float nz = noise_in ? noise_in[o] : z[j];
        if (noise_out) noise_out[o] = nz;
        out[o] = __fadd_rn(__fmul_rn(a, x0[o]), __fmul_rn(b, nz));
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Window crop for a whole batch in one launch (MONAI: `torch.cat([inputs[win_slice] for ...])`, engine.py:173-177 driver):
// patches[b][c] = volume[c][start_b : start_b + roi]   (volume [nc][VD][VH][VW], patches [batch][nc][roi])
// ---------------------------------------------------------------------------------------------------------------
struct CropArgs {
  const float* vol;
  float* patches;
  int VD, VH, VW, PD, PH, PW, batch, nc;
  int start[INIT_MAX_B][3];
};
__global__ void crop_windows_kernel(CropArgs a) {
  pdl_wait();
  const long long pv = (long long)a.PD * a.PH * a.PW;
  const long long total = pv * a.nc * a.batch;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int bc = (int)(i / pv);  // window * nc + channel
    const int b = bc / a.nc, c = bc % a.nc;
    const long long r = i % pv;
    const int x = (int)(r % a.PW), y = (int)((r / a.PW) % a.PH), z = (int)(r / ((long long)a.PW * a.PH));
    a.patches[i] = a.vol[(((long long)c * a.VD + a.start[b][0] + z) * a.VH + a.start[b][1] + y) * a.VW + a.start[b][2] + x];
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Stitching straight from the voxel-major DDIM accumulator (no planar [C][roi] intermediate):
//   out[:, start : start + roi] += scale * acc[n]            (constant blend; scale = 1: exactly `out[slices] += pred`)
//   out += w * (scale * acc[n]); count += w                  (gaussian blend, `weights` != nullptr)
// One launch per window, in MONAI's window order: fp32 sums are formed in the oracle's order, no atomics.
// thread = one window voxel: reads its CP classes (contiguous), writes class by class (lanes run along x: coalesced).
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) stitch_from_vm_kernel(float* __restrict__ vol, float* __restrict__ cnt,
                                                             const float* __restrict__ acc_vm, const float* __restrict__ w,
                                                             int C, int CP, int VD, int VH, int VW, int PD, int PH, int PW,
                                                             int sz, int sy, int sx, float scale) {
  pdl_wait();
  const long long pv = (long long)PD * PH * PW, vv = (long long)VD * VH * VW;
  for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v < pv; v += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(v % PW), y = (int)((v / PW) % PH), z = (int)(v / ((long long)PW * PH));
    const long long o = ((long long)(sz + z) * VH + sy + y) * VW + sx + x;
    const float4* src = reinterpret_cast<const float4*>(acc_vm + v * CP);
    const float wv = w ? w[v] : 1.f;
    for (int q = 0; q < CP / 4; ++q) {
      const float4 f4 = src[q];
      const float f[4] = {f4.x, f4.y, f4.z, f4.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = q * 4 + j;
        if (c < C) {
          const float pred = scale == 1.f ? f[j] : __fmul_rn(scale, f[j]);
          float* dst = vol + c * vv + o;
          *dst = w ? __fadd_rn(*dst, __fmul_rn(wv, pred)) : __fadd_rn(*dst, pred);
        }
      }
    }
    if (w) cnt[o] = __fadd_rn(cnt[o], wv);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Time-embedding bias table (models/diffusion/utils.py:6-54 + denoiser.py:51-52,65):
//   bias[step][block][c] = temb_proj_block( swish( dense1( swish( dense0( sinusoid(t_step) ) ) ) ) )
// Only the N respaced timesteps ever occur, so this runs once per plan, one CTA per step.
// ---------------------------------------------------------------------------------------------------------------
struct TembArgs {
  const float *w0, *b0, *w1, *b1;  // dense.0 [512,128], dense.1 [512,512]
  const float* pw[9];              // temb_proj weights [cout, 512]
  const float* pb[9];
  int pc[9];                       // cout per block
  int poff[9];                     // offset of the block inside one step's row
  int row;                         // floats per step
  const int* tmap;                 // [steps] original timesteps
  float* table;                    // [steps][row]
};

__global__ void __launch_bounds__(512) temb_table_kernel(TembArgs a) {
  __shared__ float e[128], h[512], g[512];
  const int tid = threadIdx.x;
  const float t = (float)a.tmap[blockIdx.x];
  if (tid < 64) {
    const float fr = expf((float)tid * -(logf(10000.f) / 63.f));
    const float arg = t * fr;
    e[tid] = sinf(arg);
    e[64 + tid] = cosf(arg);
  }
  __syncthreads();
  {
    float s = a.b0[tid];
    for (int k = 0; k < 128; ++k) s = fmaf(a.w0[tid * 128 + k], e[k], s);
    h[tid] = s / (1.f + expf(-s));  // swish
  }
  __syncthreads();
  {
    float s = a.b1[tid];
    for (int k = 0; k < 512; ++k) s = fmaf(a.w1[tid * 512 + k], h[k], s);
    g[tid] = s / (1.f + expf(-s));  // swish(temb), consumed by every temb_proj
  }
  __syncthreads();
  for (int blk = 0; blk < 9; ++blk) {
    for (int c = tid; c < a.pc[blk]; c += blockDim.x) {
      float s = a.pb[blk][c];
      const float* wr = a.pw[blk] + (long long)c * 512;
      for (int k = 0; k < 512; ++k) s = fmaf(wr[k], g[k], s);
      a.table[(long long)blockIdx.x * a.row + a.poff[blk] + c] = s;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Sliding-window stitching (MONAI sliding_window_inference, constant blend; reference call engine.py:173-177).
// One launch per window in MONAI's window order -> fp32 sums are formed in exactly the oracle's order, no atomics.
// ---------------------------------------------------------------------------------------------------------------
__global__ void stitch_add_kernel(float* __restrict__ vol, const float* __restrict__ patch, int C, int VD, int VH,
                                  int VW, int PD, int PH, int PW, int sz, int sy, int sx) {
  const long long pv = (long long)PD * PH * PW;
  const long long total = (long long)C * pv;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(i % PW), y = (int)((i / PW) % PH), z = (int)((i / ((long long)PW * PH)) % PD);
    const int c = (int)(i / pv);
    vol[(((long long)c * VD + sz + z) * VH + sy + y) * VW + sx + x] += patch[i];
  }
}

// Weighted variant for MONAI's mode="gaussian" blend (SURVEY 8f-4; not used by the reference's own call, engine.py:173-177):
//   out[slices] += w * pred ; count[slices] += w      with w the clamped gaussian importance map of the window.
// Multiply and add are kept separate (no FMA contraction) so the fp32 result matches torch's `importance_map * pred` then `+=`.
__global__ void stitch_add_weighted_kernel(float* __restrict__ vol, float* __restrict__ cnt, const float* __restrict__ patch,
                                           const float* __restrict__ w, int C, int VD, int VH, int VW, int PD, int PH, int PW,
                                           int sz, int sy, int sx) {
  const long long pv = (long long)PD * PH * PW;
  const long long total = (long long)C * pv;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long v = i % pv;
    const int x = (int)(v % PW), y = (int)((v / PW) % PH), z = (int)(v / ((long long)PW * PH));
    const int c = (int)(i / pv);
    const long long o = ((long long)(sz + z) * VH + sy + y) * VW + sx + x;
    const long long oc = (long long)c * VD * VH * VW + o;
    vol[oc] = __fadd_rn(vol[oc], __fmul_rn(w[v], patch[i]));
    if (c == 0) cnt[o] = __fadd_rn(cnt[o], w[v]);
  }
}

// The reference's binarisation (sigmoid(o) > 0.5, engine.py:179-180) of every class of voxel v and its argmax label (first
// maximum, engine.py:187).  logit(c) returns class c's fp32 logit; binary is [C][vv], argmax [vv], either may be NULL.
template <typename Logit>
__device__ __forceinline__ void binarise_voxel(Logit logit, int C, long long vv, long long v, uint8_t* __restrict__ binary,
                                               uint8_t* __restrict__ argmax) {
  float best = -INFINITY;
  int bi = 0;
  for (int c = 0; c < C; ++c) {
    const float o = logit(c);
    if (binary) binary[c * vv + v] = (1.f / (1.f + expf(-o)) > 0.5f) ? 1 : 0;
    if (o > best) {
      best = o;
      bi = c;
    }
  }
  if (argmax) argmax[v] = (uint8_t)bi;
}

// out /= count_map (fp32 volume), then the same binarisation / argmax as finalize_kernel
__global__ void finalize_weighted_kernel(float* __restrict__ vol, const float* __restrict__ cnt, uint8_t* __restrict__ binary,
                                         uint8_t* __restrict__ argmax, int C, long long vv) {
  for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v < vv; v += (long long)gridDim.x * blockDim.x) {
    const float cn = cnt[v];
    binarise_voxel([&](int c) {
      const float o = vol[c * vv + v] / cn;
      vol[c * vv + v] = o;
      return o;
    }, C, vv, v, binary, argmax);
  }
}

// MONAI ScaleIntensityRange (reference val/test transform, utils.py:167-170: a_min=-175, a_max=250, b_min=0, b_max=1, clip):
//   y = (x - a_min) / (a_max - a_min) ; y = y * (b_max - b_min) + b_min ; clip to [b_min, b_max]
// same op order in fp32, no FMA contraction -> bit-exact with the torch/numpy evaluation.
__global__ void scale_intensity_kernel(const float* __restrict__ in, float* __restrict__ out, long long n, float a_min,
                                       float a_max, float b_min, float b_max, int clip) {
  const float den = __fsub_rn(a_max, a_min), span = __fsub_rn(b_max, b_min);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float y = __fdiv_rn(__fsub_rn(in[i], a_min), den);
    y = __fadd_rn(__fmul_rn(y, span), b_min);
    if (clip) y = fminf(fmaxf(y, b_min), b_max);
    out[i] = y;
  }
}

// crop a window out of the (padded) input volume: [1][VD][VH][VW] -> [PD][PH][PW]
__global__ void crop_window_kernel(const float* __restrict__ vol, float* __restrict__ patch, int VD, int VH, int VW,
                                   int PD, int PH, int PW, int sz, int sy, int sx) {
  const long long total = (long long)PD * PH * PW;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(i % PW), y = (int)((i / PW) % PH), z = (int)(i / ((long long)PW * PH));
    patch[i] = vol[((long long)(sz + z) * VH + sy + y) * VW + sx + x];
  }
}

// out /= count (count = product of per-axis integer window counts: the grid is a Cartesian product), then the
// reference's binarisation (sigmoid(out) > 0.5), engine.py:179-180, and optionally the argmax label (engine.py:187).
__global__ void finalize_kernel(float* __restrict__ vol, const int* __restrict__ cd, const int* __restrict__ ch,
                                const int* __restrict__ cw, uint8_t* __restrict__ binary, uint8_t* __restrict__ argmax,
                                int C, int VD, int VH, int VW) {
  const long long vv = (long long)VD * VH * VW;
  for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v < vv;
       v += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(v % VW), y = (int)((v / VW) % VH), z = (int)(v / ((long long)VW * VH));
    const float cnt = (float)(cd[z] * ch[y] * cw[x]);
    binarise_voxel([&](int c) {
      const float o = vol[c * vv + v] / cnt;
      vol[c * vv + v] = o;
      return o;
    }, C, vv, v, binary, argmax);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Input-side pre-pass of the reference's val transforms (utils.py:165-181) after ScaleIntensityRanged:
//   CropForegroundd(source_key="image")     bounding box of image > 0 (MONAI generate_spatial_bounding_box, select_fn =
//                                           is_positive, margin 0), then the same crop of image and label
//   Spacingd(pixdim=(1.5, 1.5, 2.0), mode=("bilinear", "nearest"))   resample to the new voxel spacing
// ---------------------------------------------------------------------------------------------------------------
// bbox[0..2] = min index with a positive voxel per axis, bbox[3..5] = max index + 1 (caller initialises to {D,H,W,0,0,0});
// the box is over all channels.  Integer atomics: exact, order-independent.
__global__ void bbox_init_kernel(int* __restrict__ bbox, int D, int H, int W) {
  if (threadIdx.x == 0) { bbox[0] = D; bbox[1] = H; bbox[2] = W; bbox[3] = bbox[4] = bbox[5] = 0; }
}
__global__ void __launch_bounds__(256) foreground_bbox_kernel(const float* __restrict__ img, int C, int D, int H, int W,
                                                              int* __restrict__ bbox) {
  const long long vox = (long long)D * H * W, total = vox * C;
  int lo[3] = {D, H, W}, hi[3] = {0, 0, 0};
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    if (img[i] > 0.f) {
      const long long v = i % vox;
      const int x = (int)(v % W), y = (int)((v / W) % H), z = (int)(v / ((long long)W * H));
      lo[0] = min(lo[0], z); lo[1] = min(lo[1], y); lo[2] = min(lo[2], x);
      hi[0] = max(hi[0], z + 1); hi[1] = max(hi[1], y + 1); hi[2] = max(hi[2], x + 1);
    }
  }
#pragma unroll
  for (int d = 0; d < 3; ++d) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lo[d] = min(lo[d], __shfl_xor_sync(0xffffffffu, lo[d], o));
      hi[d] = max(hi[d], __shfl_xor_sync(0xffffffffu, hi[d], o));
    }
  }
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      atomicMin(bbox + d, lo[d]);
      atomicMax(bbox + 3 + d, hi[d]);
    }
  }
}
// out[c] = in[c][s0 : s0 + OD, s1 : s1 + OH, s2 : s2 + OW]   (SpatialCrop of every channel)
__global__ void crop_box_kernel(const float* __restrict__ in, float* __restrict__ out, int C, int D, int H, int W, int OD, int OH,
                                int OW, int s0, int s1, int s2) {
  const long long ov = (long long)OD * OH * OW, total = ov * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i / ov);
    const long long r = i % ov;
    const int x = (int)(r % OW), y = (int)((r / OW) % OH), z = (int)(r / ((long long)OW * OH));
    out[i] = in[(((long long)c * D + s0 + z) * H + s1 + y) * W + s2 + x];
  }
}
// Spacing resample for axis-aligned affines: output voxel (i, j, k) samples the input at index (i*rz, j*ry, k*rx) with
// r = new spacing / old spacing (voxel 0 stays on voxel 0, MONAI compute_shape_offset with scale_extent = False), border
// clamped.  mode 0: trilinear (image), weights and lerps in fp32 in a fixed order (x, then y, then z); mode 1: nearest
// (label), index = rint(coordinate) (round half to even, like grid_sample's nearest).  Coordinates are formed in fp64.
// The sample point of grid voxel (z, y, x) on a D x H x W source; shared by resample_spacing_kernel and invert_labels_kernel.
struct ResamplePoint {
  int z0, y0, x0, z1, y1, x1;  // nearest: (z0, y0, x0) only
  float fz, fy, fx;
};
__device__ __forceinline__ ResamplePoint resample_point(int z, int y, int x, double rz, double ry, double rx, int D, int H, int W,
                                                        bool nearest) {
  const double cz = fmin(fmax(z * rz, 0.0), (double)(D - 1)), cy = fmin(fmax(y * ry, 0.0), (double)(H - 1)),
               cx = fmin(fmax(x * rx, 0.0), (double)(W - 1));
  ResamplePoint p;
  if (nearest) {
    p.z0 = (int)rint(cz); p.y0 = (int)rint(cy); p.x0 = (int)rint(cx);
    return p;
  }
  p.z0 = (int)floor(cz); p.y0 = (int)floor(cy); p.x0 = (int)floor(cx);
  p.z1 = min(p.z0 + 1, D - 1); p.y1 = min(p.y0 + 1, H - 1); p.x1 = min(p.x0 + 1, W - 1);
  p.fz = (float)(cz - p.z0); p.fy = (float)(cy - p.y0); p.fx = (float)(cx - p.x0);
  return p;
}
// src: one channel, element (z, y, x) at src[(z * SH + y) * SW + x] (SH, SW: row strides of the volume src lies in)
__device__ __forceinline__ float resample_sample(const float* __restrict__ src, int SH, int SW, const ResamplePoint& p, bool nearest) {
  auto at = [&](int zz, int yy, int xx) { return src[((long long)zz * SH + yy) * SW + xx]; };
  if (nearest) return at(p.z0, p.y0, p.x0);
  auto lerp = [](float a, float b, float t) { return __fadd_rn(a, __fmul_rn(t, __fsub_rn(b, a))); };
  const float c00 = lerp(at(p.z0, p.y0, p.x0), at(p.z0, p.y0, p.x1), p.fx), c01 = lerp(at(p.z0, p.y1, p.x0), at(p.z0, p.y1, p.x1), p.fx);
  const float c10 = lerp(at(p.z1, p.y0, p.x0), at(p.z1, p.y0, p.x1), p.fx), c11 = lerp(at(p.z1, p.y1, p.x0), at(p.z1, p.y1, p.x1), p.fx);
  return lerp(lerp(c00, c01, p.fy), lerp(c10, c11, p.fy), p.fz);
}
__global__ void __launch_bounds__(256) resample_spacing_kernel(const float* __restrict__ in, float* __restrict__ out, int C, int D,
                                                               int H, int W, int OD, int OH, int OW, double rz, double ry,
                                                               double rx, int mode) {
  const long long ov = (long long)OD * OH * OW, total = ov * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i / ov);
    const long long r = i % ov;
    const int x = (int)(r % OW), y = (int)((r / OW) % OH), z = (int)(r / ((long long)OW * OH));
    const ResamplePoint p = resample_point(z, y, x, rz, ry, rx, D, H, W, mode == 1);
    out[i] = resample_sample(in + (long long)c * D * H * W, H, W, p, mode == 1);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Labels on the input volume's grid: MONAI Invertd of the val transforms' Spacingd + CropForegroundd, then AsDiscreted
// (sigmoid > 0.5, engine.py:179-180), fused.  blended: the finalised fp32 [C][VD][VH][VW] volume of the window driver (padded
// to the roi when the resampled volume was smaller); the resampled volume [RD][RH][RW] sits at `offset` inside it.  For each
// voxel p of the [D0][H0][W0] output: outside the foreground box [box_start, box_start + box_dims) the logits are the zeros
// MONAI's inverse BorderPad inserts (binary 0, argmax 0); inside, j = p - box_start samples the resampled volume at
// clamp(j * ratio, 0, res - 1) with ratio = spacing_in / pixdim -- the exact inverse of resample_spacing_kernel's mapping, with
// the same sample point and lerp order -- and each class is binarised as in finalize_kernel.  One thread per output voxel
// (consecutive threads along W: coalesced byte stores per class plane), looping over the classes.
// ---------------------------------------------------------------------------------------------------------------
struct InvertLabelsArgs {
  const float* blended;
  int C, VH, VW;               // classes, row strides of the driver volume
  long long vol_vox;           // VD * VH * VW
  int off[3], res[3], box_start[3], box_dims[3], out[3];
  double ratio[3];
  int nearest;
  uint8_t* binary;             // [C][D0][H0][W0] or NULL
  uint8_t* argmax;             // [D0][H0][W0] or NULL
};
__global__ void __launch_bounds__(256) invert_labels_kernel(InvertLabelsArgs a) {
  const long long vv = (long long)a.out[0] * a.out[1] * a.out[2];
  const float* base = a.blended + ((long long)a.off[0] * a.VH + a.off[1]) * a.VW + a.off[2];
  for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v < vv; v += (long long)gridDim.x * blockDim.x) {
    const int jz = (int)(v / ((long long)a.out[2] * a.out[1])) - a.box_start[0];
    const int jy = (int)((v / a.out[2]) % a.out[1]) - a.box_start[1];
    const int jx = (int)(v % a.out[2]) - a.box_start[2];
    if ((unsigned)jz >= (unsigned)a.box_dims[0] || (unsigned)jy >= (unsigned)a.box_dims[1] || (unsigned)jx >= (unsigned)a.box_dims[2]) {
      binarise_voxel([](int) { return 0.f; }, a.C, vv, v, a.binary, a.argmax);
      continue;
    }
    const ResamplePoint p = resample_point(jz, jy, jx, a.ratio[0], a.ratio[1], a.ratio[2], a.res[0], a.res[1], a.res[2], a.nearest);
    binarise_voxel([&](int c) { return resample_sample(base + c * a.vol_vox, a.VH, a.VW, p, a.nearest); }, a.C, vv, v, a.binary,
                   a.argmax);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Uncertainty-weighted fusion of the DDIM steps of R independent runs (upstream Diff-UNet's test-time fusion; NOT used
// by this reference, whose ddim_sample returns the plain sum, models/diffusion/diffusion.py:94-98; SURVEY 8f-4):
//   for every step k (loop order, t high -> low):  m = mean_r(model_output[r][k]);  p = max(sigmoid(m), 0.001)
//     u = -p * log(p);   w = exp(sigmoid((k + 1) / N) * (1 - u));   out += w * sum_r clamp(model_output[r][k], -1, 1)
// steps: [R][N][n] fp32 raw model outputs (dunet_ddim_sample's per_step_logits of each run).
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) uncertainty_fuse_kernel(const float* __restrict__ steps, float* __restrict__ out, int R, int N,
                                                               long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float acc = 0.f;
    for (int k = 0; k < N; ++k) {
      float m = 0.f, sx0 = 0.f;
      for (int r = 0; r < R; ++r) {
        const float v = steps[((long long)r * N + k) * n + i];
        m += v;
        sx0 += fminf(fmaxf(v, -1.f), 1.f);
      }
      m /= (float)R;
      const float p = fmaxf(1.f / (1.f + expf(-m)), 0.001f);
      const float u = -p * logf(p);
      const float sg = 1.f / (1.f + expf(-(float)(k + 1) / (float)N));
      acc += expf(sg * (1.f - u)) * sx0;
    }
    out[i] = acc;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Multi-GPU exchange fused with the finalize step, over NVLink peer memory (no NCCL on the data): rank r owns channels
// [c_lo, c_hi) of a volume.  It READS the partial stitched sums of those channels straight out of every contributing
// rank's buffer (peer pointers: plain ld.global over NVLink / NVSwitch; a rank only contributes the slab of dim-0 rows
// its windows touch, the others are skipped), adds them in rank order, divides by the coverage counts, binarises
// (sigmoid > 0.5, engine.py:179-180) and WRITES the uint8 labels into the destination rank's volume (peer store).
// Replaces reduce-scatter + local finalize + gather: the fp32 sums cross NVLink once, only where they are non-zero.
// thread = 4 consecutive voxels along x (16-byte loads, 4-byte stores); W % 4 == 0 required.
// ---------------------------------------------------------------------------------------------------------------
constexpr int PEER_MAX_SRC = 16;
struct FinalizePeersArgs {
  const float* src[PEER_MAX_SRC];  // [C][D][H][W] fp32 partial sums of source k (local or peer memory)
  int lo[PEER_MAX_SRC], hi[PEER_MAX_SRC];  // dim-0 rows [lo, hi) source k has contributed to
  int n_src;
  const int *cd, *ch, *cw;         // per-axis coverage counts (device, local)
  uint8_t* binary;                 // [C][D][H][W] destination labels (local or peer memory)
  float* blended;                  // optional [C][D][H][W] fp32 destination of the normalised logits, or nullptr
  int c_lo, c_hi, D, H, W;
};
__global__ void __launch_bounds__(256) finalize_peers_kernel(FinalizePeersArgs a) {
  const long long vv = (long long)a.D * a.H * a.W, q = vv / 4;
  const long long total = q * (a.c_hi - a.c_lo);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = a.c_lo + (int)(i / q);
    const long long v = (i % q) * 4;
    const int x = (int)(v % a.W), y = (int)((v / a.W) % a.H), z = (int)(v / ((long long)a.W * a.H));
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    bool first = true;
#pragma unroll 1
    for (int k = 0; k < a.n_src; ++k) {
      if (z < a.lo[k] || z >= a.hi[k]) continue;
      const float4 t = *reinterpret_cast<const float4*>(a.src[k] + c * vv + v);
      if (first) { s = t; first = false; }   // the first contribution is taken as is (0 + t would lose the sign of -0)
      else { s.x += t.x; s.y += t.y; s.z += t.z; s.w += t.w; }
    }
    const float czy = (float)(a.cd[z] * a.ch[y]);
    const float o[4] = {s.x / (czy * (float)a.cw[x]), s.y / (czy * (float)a.cw[x + 1]), s.z / (czy * (float)a.cw[x + 2]),
                        s.w / (czy * (float)a.cw[x + 3])};
    uchar4 lab;
    lab.x = (1.f / (1.f + expf(-o[0])) > 0.5f) ? 1 : 0;
    lab.y = (1.f / (1.f + expf(-o[1])) > 0.5f) ? 1 : 0;
    lab.z = (1.f / (1.f + expf(-o[2])) > 0.5f) ? 1 : 0;
    lab.w = (1.f / (1.f + expf(-o[3])) > 0.5f) ? 1 : 0;
    *reinterpret_cast<uchar4*>(a.binary + c * vv + v) = lab;
    if (a.blended) *reinterpret_cast<float4*>(a.blended + c * vv + v) = make_float4(o[0], o[1], o[2], o[3]);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Per-class Dice inputs (reference metric.py:3-49 dice_coeff as used by Tester.validation_step, test.py:143-151):
// counts[c] = { |pred_c & label_c|, |pred_c|, |label_c| } as exact 64-bit integers.  pred: uint8 {0,1} [C][vox] (the
// binary volume finalize_kernel writes); label: uint8 or fp32 one-hot [C][vox], non-zero = foreground.
// grid = (blocks, C); integer atomics -> order-independent, exact.
// ---------------------------------------------------------------------------------------------------------------
template <typename LabelT>
__global__ void __launch_bounds__(256) dice_counts_kernel(const uint8_t* __restrict__ pred, const LabelT* __restrict__ label,
                                                          long long vox, unsigned long long* __restrict__ counts) {
  const int c = blockIdx.y;
  const uint8_t* p = pred + (long long)c * vox;
  const LabelT* l = label + (long long)c * vox;
  unsigned int inter = 0, np = 0, nl = 0;  // < 2^32 per thread: vox / threads is far below that
  for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v < vox; v += (long long)gridDim.x * blockDim.x) {
    const bool a = p[v] != 0, b = l[v] != LabelT(0);
    inter += (a && b) ? 1u : 0u;
    np += a ? 1u : 0u;
    nl += b ? 1u : 0u;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    inter += __shfl_xor_sync(0xffffffffu, inter, o);
    np += __shfl_xor_sync(0xffffffffu, np, o);
    nl += __shfl_xor_sync(0xffffffffu, nl, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(counts + c * 3 + 0, (unsigned long long)inter);
    atomicAdd(counts + c * 3 + 1, (unsigned long long)np);
    atomicAdd(counts + c * 3 + 2, (unsigned long long)nl);
  }
}

}  // namespace dunet
