// Debug-only direct 3x3x3 convolution on CUDA cores.  NOT on the product path: it exists so the tcgen05 kernel
// (conv3d_tc.cuh) and the weight packing can be bisected on the GPU against an independent implementation that reads
// the ORIGINAL fp32 [Cout][Cin][3][3][3] weights.  Selected only by DUNET_DEBUG_REF_CONV (tests).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "elementwise.cuh"

namespace dunet {

template <bool HF>
__global__ void __launch_bounds__(128) conv3d_ref_kernel(const __nv_bfloat16* __restrict__ src0, int c0, int chunks0,
                                                         const __nv_bfloat16* __restrict__ src1, int c1, int chunks1,
                                                         const float* __restrict__ w /*[cout][c0+c1][27]*/,
                                                         __nv_bfloat16* __restrict__ out, int cout, int out_chunks,
                                                         int D, int H, int W, int batch, int rot) {
  // cout = REAL output channels; out_chunks = chunk stride of the (padded) output tensor, padded chunks untouched
  const long long vox = (long long)D * H * W;
  const int och = (cout + 7) / 8;
  const int cin = c0 + c1;
  const long long total = (long long)batch * och * vox;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long v = i % vox;
    const int oc = (int)((i / vox) % och);
    const int n = (int)(i / (vox * och));
    const int x = (int)(v % W), y = (int)((v / W) % H), z = (int)(v / ((long long)W * H));
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    for (int tz = 0; tz < 3; ++tz) {
      const int zz = z + tz - 1;
      if (zz < 0 || zz >= D) continue;
      for (int ty = 0; ty < 3; ++ty) {
        const int yy = y + ty - 1;
        if (yy < 0 || yy >= H) continue;
        for (int tx = 0; tx < 3; ++tx) {
          const int xx = x + tx - 1;
          if (xx < 0 || xx >= W) continue;
          const int tap = (tz * 3 + ty) * 3 + tx;
          const long long sv = ((long long)zz * H + yy) * W + xx;
          for (int ci = 0; ci < cin; ci += 8) {
            const bool second = ci >= c0;  // c0 is a multiple of 8 whenever c1 > 0
            const BF8* sp = second ? reinterpret_cast<const BF8*>(src1) + ((long long)n * chunks1 + (ci - c0) / 8) * vox
                                   : reinterpret_cast<const BF8*>(src0) + ((long long)n * chunks0 + ci / 8) * vox;
            float xi[8];
            bf8_to_float<HF>(sp[sv], xi);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              if (ci + k < cin) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  if (oc * 8 + j >= cout) continue;
                  const float wv =
                      round_16<HF>(w[((long long)(oc * 8 + j) * cin + (rot ? (ci + k + rot) % c0 : ci + k)) * 27 + tap]);
                  acc[j] = fmaf(xi[k], wv, acc[j]);
                }
              }
            }
          }
        }
      }
    }
    reinterpret_cast<BF8*>(out)[((long long)n * out_chunks + oc) * vox + v] = float_to_bf8<HF>(acc);
  }
}

}  // namespace dunet
