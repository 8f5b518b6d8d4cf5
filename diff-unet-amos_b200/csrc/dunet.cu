// libdunet_b200.so -- C ABI (include/dunet.h) + host-side plan for the Diff-UNet DDIM inference path on B200.
// Host code here only sequences kernels on the caller's stream; all arithmetic is in the sm_100a kernels.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <set>
#include <string>
#include <unordered_map>
#include <vector>

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "../../include/dunet.h"
#include "conv3d_ref.cuh"
#include "conv3d_tc.cuh"
#include "conv3d_tc64.cuh"
#include "conv3d_flat.cuh"
#include "deconv2_tc.cuh"
#include "elementwise.cuh"
#include "surface.cuh"

using namespace dunet;
typedef __nv_bfloat16 bf16;

// ------------------------------------------------------------------------------------------------ errors / utils
static thread_local std::string g_err;
static std::atomic<uint64_t> g_launches{0};

static int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
#define CUDA_TRY(expr)                                                                                   \
  do {                                                                                                   \
    cudaError_t e__ = (expr);                                                                            \
    if (e__ != cudaSuccess) return fail(DUNET_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), \
                                        __FILE__, __LINE__);                                             \
  } while (0)
#define LAUNCH_CHECK()                                                                                   \
  do {                                                                                                   \
    g_launches.fetch_add(1, std::memory_order_relaxed);                                                  \
    cudaError_t e__ = cudaGetLastError();                                                                \
    if (e__ != cudaSuccess) return fail(DUNET_E_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(e__), \
                                        __FILE__, __LINE__);                                             \
  } while (0)
#define TRY(expr)            \
  do {                       \
    int r__ = (expr);        \
    if (r__ != 0) return r__; \
  } while (0)

// ---- optional live profiling of the launches of ONE plan (bench.py roofline): CUDA events around every launch ----
struct ProfRec { cudaEvent_t a, b; int tag; };
// PROF_CONV_SPLIT: 3x3x3 convs that run in split precision inside a 16-bit plan (the encoder in fp16 mode): 3 MMAs per
// algorithmic product, reported apart from the 16-bit convs whose roofline is the tensor peak
enum { PROF_CONV = 0, PROF_NORM = 1, PROF_FINAL = 2, PROF_DECONV = 3, PROF_SPLITK = 4, PROF_OTHER = 5, PROF_NORM_SMALL = 6, PROF_GLUE = 7,
       PROF_CONV_SPLIT = 8, PROF_DECONV_SMALL = 9, PROF_TAGS = 12 };
struct Prof {
  bool on = false;
  std::vector<ProfRec> recs;       // event pool, reused across enable() calls
  size_t used = 0;
  double flops = 0.0;
  double bytes[PROF_TAGS] = {};  // ALGORITHMIC HBM bytes per kernel family; for the two conv families: ALGORITHMIC FLOPs
};
struct dunet_plan;
static Prof* prof_of(const dunet_plan* p);
static int prof_begin_(Prof* pr, int tag, cudaStream_t st) {
  if (!pr || !pr->on) return 0;
  if (pr->used == pr->recs.size()) {
    ProfRec rec;
    CUDA_TRY(cudaEventCreate(&rec.a));
    CUDA_TRY(cudaEventCreate(&rec.b));
    pr->recs.push_back(rec);
  }
  pr->recs[pr->used].tag = tag;
  CUDA_TRY(cudaEventRecord(pr->recs[pr->used].a, st));
  return 0;
}
static int prof_end_(Prof* pr, cudaStream_t st) {
  if (!pr || !pr->on) return 0;
  CUDA_TRY(cudaEventRecord(pr->recs[pr->used].b, st));
  ++pr->used;
  return 0;
}
// the launchers below all have the plan in scope as `p`
#define prof_begin(tag, st) prof_begin_(prof_of(p), tag, st)
#define prof_end(st) prof_end_(prof_of(p), st)
#define PROF_ON (prof_of(p)->on)

// Launch with programmatic stream serialization (see pdl_sync() in ptx.cuh): only for kernels that call pdl_sync().
template <typename... KArgs, typename... Args>
static void launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  (void)cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);  // the error is picked up by LAUNCH_CHECK()
}

static inline int pad_to(int v, int m) { return (v + m - 1) / m * m; }
static inline int grid_for(long long total, int threads, int cap = 148 * 16) {
  long long b = (total + threads - 1) / threads;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}
static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ------------------------------------------------------------------------------------------------ TMA descriptors
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;

static int load_driver_entry() {
  if (g_encode) return 0;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult q;
  CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
  if (!fn || q != cudaDriverEntryPointSuccess) return fail(DUNET_E_CUDA, "cuTensorMapEncodeTiled not available");
  g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  return 0;
}

// Tensor map over a C8-planar activation: dims (x*8+c8 : W*8, y : H, z : D, plane : batch*chunks), box = one halo plane.
static int make_act_tmap(CUtensorMap* m, const bf16* base, int planes, int D, int H, int W, int kch, int halo) {
  TRY(load_driver_entry());
  cuuint64_t dims[4] = {(cuuint64_t)W * 8, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)planes};
  cuuint64_t strides[3] = {(cuuint64_t)W * 16, (cuuint64_t)H * W * 16, (cuuint64_t)D * H * W * 16};
  cuuint32_t box[4] = {(cuuint32_t)(CONV_TX + 2 * halo) * 8, (cuuint32_t)(CONV_TY + 2 * halo), 1, (cuuint32_t)kch};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<bf16*>(base), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(DUNET_E_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d (W=%d H=%d D=%d planes=%d)",
                                     (int)r, W, H, D, planes);
  return 0;
}

// Tensor map for the flattened-plane kernel (conv3d_flat.cuh): box = (W + 2 positions, ty + 2 rows, one z, 8 chunks)
static int make_flat_tmap(CUtensorMap* m, const bf16* base, int planes, int D, int H, int W, int hx, int ty, int halo = 1) {
  TRY(load_driver_entry());
  cuuint64_t dims[4] = {(cuuint64_t)W * 8, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)planes};
  cuuint64_t strides[3] = {(cuuint64_t)W * 16, (cuuint64_t)H * W * 16, (cuuint64_t)D * H * W * 16};
  cuuint32_t box[4] = {(cuuint32_t)hx * 8, (cuuint32_t)(ty + 2 * halo), 1, 8};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<bf16*>(base), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(DUNET_E_CUDA, "cuTensorMapEncodeTiled (flat) failed with CUresult %d (W=%d H=%d D=%d planes=%d hx=%d ty=%d)",
                                     (int)r, W, H, D, planes, hx, ty);
  return 0;
}

// ------------------------------------------------------------------------------------------------ weight packing
// conv weights fp32 [coutr][cinr][27] -> bf16 [n_tile][cin block][tap][k chunk][N_TILE][8]   (see conv3d_tc.cuh)
// fp32x3 mode (parts == 3): the block list is [W.hi | W.hi | W.lo] (ncb = 3 x the logical blocks), matching the activation
// segments [A.hi | A.lo | A.hi] of ConvSegs.
__device__ __forceinline__ bf16 weight_part(float v, int part, int fp16) {
  if (fp16) {  // fp16 storage behind the 16-bit pointer type (DUNET_FLAG_FP16; never combined with the hi/lo split)
    const __half h = __float2half_rn(v);
    return *reinterpret_cast<const bf16*>(&h);
  }
  const bf16 hi = __float2bfloat16_rn(v);
  return part < 2 ? hi : __float2bfloat16_rn(v - __bfloat162float(hi));
}
__global__ void pack_conv_w_kernel(const float* __restrict__ w, bf16* __restrict__ out, int coutr, int cinr, int c0r,
                                   int c0p, int c1r, int cb_ch, int n_tile, int ncb, int n_tiles, int rot, int parts, int fp16, int triple) {
  const int kch = cb_ch / 8;
  const int ncb1 = ncb / parts;
  const long long total = (long long)n_tiles * ncb * 27 * kch * n_tile * 8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    long long t = i;
    const int j = (int)(t % 8); t /= 8;
    const int col = (int)(t % n_tile); t /= n_tile;
    const int k = (int)(t % kch); t /= kch;
    const int tap = (int)(t % 27); t /= 27;
    const int cbg = (int)(t % ncb); t /= ncb;
    const int nt = (int)t;
    const int co = nt * n_tile + col;
    const int cb = cbg % ncb1, part = parts == 1 ? 0 : cbg / ncb1;
    const int lc = cb * cb_ch + k * 8 + j;
    int ci = -1, wpart = part;
    if (triple) {  // one block holds [A.hi | A.lo | A.hi] of the c0r real channels against [W.hi | W.hi | W.lo] (see ConvW::triple)
      if (lc < 3 * c0r) { ci = lc % c0r; wpart = lc / c0r == 2 ? 2 : 0; }
    } else if (lc < c0p) { if (lc < c0r) ci = rot ? (lc + rot) % c0r : lc; }  // rot: packed order is [x.., image..], reference [image.., x..]
    else { const int l1 = lc - c0p; if (l1 < c1r) ci = c0r + l1; }
    float v = 0.f;
    if (co < coutr && ci >= 0) v = w[((long long)co * cinr + ci) * 27 + tap];
    out[i] = weight_part(v, wpart, fp16);
  }
}
// conv weights for the Cout = 64 z-stacked kernel (conv3d_tc64.cuh): bf16 [cin block][ty*3+tx][k chunk][192][8] with
// row = (2 - tz) * 64 + cout
__global__ void pack_conv_w64_kernel(const float* __restrict__ w, bf16* __restrict__ out, int coutr, int cinr, int c0r,
                                     int c0p, int c1r, int cb_ch, int ncb, int rot, int parts, int fp16, int triple) {
  const int kch = cb_ch / 8;
  const int ncb1 = ncb / parts;
  const long long total = (long long)ncb * 9 * kch * 192 * 8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    long long t = i;
    const int j = (int)(t % 8); t /= 8;
    const int row = (int)(t % 192); t /= 192;
    const int k = (int)(t % kch); t /= kch;
    const int tyx = (int)(t % 9); t /= 9;
    const int cbg = (int)t;
    const int cb = cbg % ncb1, part = parts == 1 ? 0 : cbg / ncb1;
    const int tz = 2 - row / 64, co = row % 64;
    const int tap = tz * 9 + tyx;
    const int lc = cb * cb_ch + k * 8 + j;
    int ci = -1, wpart = part;
    if (triple) {  // one block holds [A.hi | A.lo | A.hi] of the c0r real channels against [W.hi | W.hi | W.lo] (see ConvW::triple)
      if (lc < 3 * c0r) { ci = lc % c0r; wpart = lc / c0r == 2 ? 2 : 0; }
    } else if (lc < c0p) { if (lc < c0r) ci = rot ? (lc + rot) % c0r : lc; }  // rot: packed order is [x.., image..], reference [image.., x..]
    else { const int l1 = lc - c0p; if (l1 < c1r) ci = c0r + l1; }
    float v = 0.f;
    if (co < coutr && ci >= 0) v = w[((long long)co * cinr + ci) * 27 + tap];
    out[i] = weight_part(v, wpart, fp16);
  }
}
// transposed-conv weights fp32 [cinr][coutr][8] -> bf16 [tap][cinp][coutp]
__global__ void pack_deconv_w_kernel(const float* __restrict__ w, bf16* __restrict__ out, int cinr, int coutr, int cinp,
                                     int coutp, int fp16) {
  const long long total = 8LL * cinp * coutp;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int co = (int)(i % coutp);
    const int ci = (int)((i / coutp) % cinp);
    const int tap = (int)(i / ((long long)coutp * cinp));
    float v = 0.f;
    if (ci < cinr && co < coutr) v = w[((long long)ci * coutr + co) * 8 + tap];
    out[i] = weight_part(v, 0, fp16);
  }
}
// transposed-conv weights fp32 [cinr][coutr][8] -> tensor-core B operand bf16 [n_tile][cin block][k chunk][128][8] where
// 128-column block nt = (dz*2 + dy) * (coutp/64) + cout/64, column inside it = dx * 64 + cout % 64  (tap = dz*4 + dy*2 + dx)
__global__ void pack_deconv_tc_w_kernel(const float* __restrict__ w, bf16* __restrict__ out, int cinr, int coutr, int cinp,
                                        int coutp, int parts, int fp16) {
  const int n_tile = 128, kch = 8, ncb1 = cinp / 64, ncb = ncb1 * parts, n_tiles = 8 * coutp / n_tile;
  const long long total = (long long)n_tiles * ncb * kch * n_tile * 8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    long long t = i;
    const int j = (int)(t % 8); t /= 8;
    const int col = (int)(t % n_tile); t /= n_tile;
    const int k = (int)(t % kch); t /= kch;
    const int cbg = (int)(t % ncb); t /= ncb;
    const int nt = (int)t;
    const int cb = cbg % ncb1, part = parts == 1 ? 0 : cbg / ncb1;
    const int nblk = coutp / 64, dzdy = nt / nblk;
    const int tap = dzdy * 2 + col / 64, co = (nt - dzdy * nblk) * 64 + col % 64;
    const int ci = cb * 64 + k * 8 + j;
    float v = 0.f;
    if (ci < cinr && co < coutr) v = w[((long long)ci * coutr + co) * 8 + tap];
    out[i] = weight_part(v, part, fp16);
  }
}
// copy `n` floats into a zero-padded buffer of n_pad floats, optionally strided rows: dst[r][0..cols_pad) <- src[r][0..cols)
__global__ void copy_pad_rows_kernel(const float* __restrict__ src, float* __restrict__ dst, int rows, int cols,
                                     int rows_pad, int cols_pad) {
  const long long total = (long long)rows_pad * cols_pad;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % cols_pad), r = (int)(i / cols_pad);
    dst[i] = (r < rows && c < cols) ? src[(long long)r * cols + c] : 0.f;
  }
}

// ------------------------------------------------------------------------------------------------ plan
struct ConvW {
  int c0r = 0, c1r = 0, c0p = 0, c1p = 0, coutr = 0, coutp = 0;
  int cb_ch = 64, n_tile = 64, nb0 = 0, nb1 = 0, n_tiles = 1;
  int parts = 1;  // 3 in split precision: weight block list [W.hi | W.hi | W.lo]
  bool split = false;   // this conv reads and writes hi + lo bf16 pairs (fp32x3 mode; the encoder in fp16 mode)
  // split precision with very few real input channels (the encoder's first conv, Cin = 1): the three products hi*hi + lo*hi +
  // hi*lo fit into ONE input-channel block -- packed activation channels [A.hi | A.lo | A.hi] (3 * c0r of the 32) against
  // weights [W.hi | W.hi | W.lo] -- instead of three mostly-zero 32-channel blocks: a third of the MMAs, a single source tensor
  bool triple = false;
  bf16* packed = nullptr;
  bf16* packed64 = nullptr;  // z-stacked layout for the Cout = 64 kernel (coutp == 64 only)
  float* w32 = nullptr;  // debug copy of the original fp32 weight
  float *gamma = nullptr, *beta = nullptr;
  int rot = 0;  // > 0: packed input channel j holds reference channel (j + rot) % c0r (denoiser input [x.., image..], rot = in_channels)
  bool have_w = false, have_cb = false, have_g = false, have_b = false;
  void shape(int c0r_, int c0p_, int c1r_, int c1p_, int coutr_, int parts_ = 1, int cb64_ = 32) {
    c0r = c0r_; c0p = c0p_; c1r = c1r_; c1p = c1p_; coutr = coutr_; parts = parts_;
    split = parts_ == 3;
    triple = false;
    cb64 = (c1p == 0 && c0p == 32) ? 32 : cb64_;
    coutp = pad_to(coutr, 64);
    cb_ch = (c1p == 0 && c0p == 32) ? 32 : 64;
    n_tile = (coutp % 128 == 0) ? 128 : 64;
    n_tiles = coutp / n_tile;
    nb0 = c0p / cb_ch; nb1 = c1p / cb_ch;
  }
  int ncb() const { return (nb0 + nb1) * parts; }  // input-channel blocks the kernels walk
  size_t packed_elems() const { return (size_t)n_tiles * ncb() * 27 * cb_ch * n_tile; }
  // the Cout = 64 z-stacked kernel walks 32-channel blocks (its plane ring then holds two blocks, conv3d_tc64.cuh)
  int cb64 = 32;
  int ncb64() const { return (c0p + c1p) / cb64 * parts; }
  size_t packed64_elems() const { return (size_t)ncb64() * 9 * cb64 * 192; }
};
struct Act {  // an activation tensor: C8-planar bf16, plus its low part in fp32x3 mode
  bf16* hi = nullptr;
  bf16* lo = nullptr;
};
struct TwoConvW {
  ConvW a, b;
  float *tp_w = nullptr, *tp_b = nullptr;  // temb_proj [coutr][512], [coutr]
  bool has_temb = false, have_tpw = false, have_tpb = false;
};
struct DeconvW {
  int cinr = 0, cinp = 0, coutr = 0, coutp = 0, parts = 1;
  bf16* packed = nullptr;     // CUDA-core debug kernel layout [tap][cinp][coutp]
  bf16* packed_tc = nullptr;  // tensor-core layout, see pack_deconv_tc_w_kernel
  float* bias = nullptr;
  bool have_w = false, have_b = false;
};

enum SlotKind { K_CONV_W, K_CONV_B, K_IN_G, K_IN_B, K_TP_W, K_TP_B, K_DENSE, K_DECONV_W, K_DECONV_B, K_FINAL_W, K_FINAL_B };
struct Slot {
  SlotKind kind;
  void* obj;
  int idx;  // K_DENSE: 0..3
  std::vector<int64_t> shape;
  bool seen = false;
};

struct WsLayout {
  size_t in_pack, raw, mid, partial, ss, splitk, affine, x_t, acc, image, total;
  size_t emb[5], epool[5], x[5], dpool[5], up[5], u[5];
};

struct dunet_plan {
  dunet_cfg cfg;
  int C, D[5], H[5], W[5];
  long long V[5];
  int fr[6], fp[6];       // real / padded features
  int upr[5], upp[5];     // upsampled channels of upcat_l (index l = 4..1)
  int uoutr[5], uoutp[5]; // output channels of upcat_l
  int in_pad = 32;
  TwoConvW enc[5], den[5], upc[5];  // upc index = l (1..4)
  DeconvW dec[5];
  float* dense[4] = {nullptr, nullptr, nullptr, nullptr};  // temb dense.0 w,b ; dense.1 w,b
  float *final_w = nullptr, *final_b = nullptr;            // [C][f5p], [C]
  std::unordered_map<std::string, Slot> slots;
  // schedule
  int n_steps = 0;
  std::vector<int> tmap;
  std::vector<float> sr, srm1, acp;
  int* d_tmap = nullptr;
  // temb bias table [n_steps + 1][row]; the extra row is scratch for timesteps outside the schedule
  float* temb_table = nullptr;
  int temb_row = 0, temb_off[9];
  bool committed = false;
  // layout the embeddings currently held in a workspace were written with: (batch, dual-stream halves or not).  A later
  // dunet_ddim_sample(run_encoder = 0) must read them back through the same layout.
  int emb_B = 0;
  bool emb_dual = false;
  std::vector<void*> owned;
  // two internal streams: the two halves of a window batch run out of phase so that the HBM-bound kernels of one half
  // (normalise, final/DDIM, transposed conv) overlap the tensor-core-bound convolutions of the other
  cudaStream_t half_stream[2] = {nullptr, nullptr};
  cudaEvent_t ev_fork = nullptr, ev_join[2] = {nullptr, nullptr};
  int num_sms = 0;
  mutable Prof prof;  // per-plan launch profiler (dunet_profile_*)
  // timesteps passed to dunet_denoise_step that are not one shared schedule entry (training-style calls, per-sample t):
  // a [batch_max][temb_row] bias table built per call; the timesteps are staged through a small ring of pinned host
  // slots (an event per slot says when its copy has been consumed) -- all allocated in dunet_plan_commit
  static constexpr int T_RING = 8;
  int* h_t = nullptr;          // pinned [T_RING][batch_max]
  int* d_t = nullptr;          // device [batch_max]
  float* temb_scratch = nullptr;  // device [batch_max][temb_row]
  cudaEvent_t t_ev[T_RING] = {};
  int t_slot = 0;
};
static Prof* prof_of(const dunet_plan* p) { return &p->prof; }

static int dev_alloc(dunet_plan* p, void** out, size_t bytes) {
  CUDA_TRY(cudaMalloc(out, bytes ? bytes : 16));
  p->owned.push_back(*out);
  return 0;
}

static void add_slot(dunet_plan* p, const std::string& key, SlotKind kind, void* obj, std::vector<int64_t> shape, int idx = 0) {
  Slot s; s.kind = kind; s.obj = obj; s.idx = idx; s.shape = std::move(shape);
  p->slots[key] = s;
}
static void add_convblock_slots(dunet_plan* p, const std::string& pre, ConvW* c) {
  add_slot(p, pre + ".conv.weight", K_CONV_W, c, {c->coutr, c->c0r + c->c1r, 3, 3, 3});
  add_slot(p, pre + ".conv.bias", K_CONV_B, c, {c->coutr});
  add_slot(p, pre + ".adn.N.weight", K_IN_G, c, {c->coutr});
  add_slot(p, pre + ".adn.N.bias", K_IN_B, c, {c->coutr});
}
static void add_twoconv_slots(dunet_plan* p, const std::string& pre, TwoConvW* t) {
  if (t->has_temb) {
    add_slot(p, pre + ".temb_proj.weight", K_TP_W, t, {t->a.coutr, 512});
    add_slot(p, pre + ".temb_proj.bias", K_TP_B, t, {t->a.coutr});
  }
  add_convblock_slots(p, pre + ".conv_0", &t->a);
  add_convblock_slots(p, pre + ".conv_1", &t->b);
}

constexpr int CONV_ZT = 4;

// Geometry of the flattened-plane kernel (conv3d_flat.cuh) on a level of D x H x W voxels per sample: strips of ty rows of
// hx = W + 2 * halo positions (N = npos of them, at most 256), zt z-slabs per work item (a divisor of D, zt * npos <= 512
// TMEM columns), and the plane and weight rings that fit the shared memory.
struct FlatGeom {
  int hx = 0, ty = 0, npos = 0, lbo = 0, a_slots = 0, w_slots = 0, smem = 0, zt = 0, tiles_y = 0, tiles_z = 0;
};
// 3x3x3 conv: halo 1, >= 160 accumulator columns, a plane ring of 2 x (zt + 2) slots.  Transposed conv: halo 0, >= 128
// columns, 3 x zt slots.  False (g untouched) when the row does not fit one TMA box (hx > 32) or the weight ring would get
// fewer than two slots.
static bool flat_geom(FlatGeom* g, int D, int H, int W, int halo, int min_cols, int slots_per_plane) {
  const int hx = W + 2 * halo;
  if (hx > 32) return false;
  const int ty_max = std::max(1, (256 + 2 * halo) / hx);  // the last 2 * halo positions of a strip are not outputs
  const int tiles_y = (H + ty_max - 1) / ty_max, ty = (H + tiles_y - 1) / tiles_y;
  const int npos = pad_to(std::max(ty * hx - 2 * halo, 1), 16);
  // ZT: the SMALLEST slab count (dividing D) whose ZT * npos accumulator columns keep the weight stream affordable -- a
  // 16 KB weight tile feeds ZT * npos / 2 MMA clocks; at >= 160 columns (<= ~50 B/clk/SM; measured at 24^3 with 144 CTAs
  // streaming concurrently: no slowdown, L2 serves CTAs that walk the same tiles in step) more items beat more re-use:
  // 24^3 at ZT = 1 has 72 items per sample instead of 36 and the four layers take 132 us instead of 200 (2 windows).
  int zt = 0;
  for (int cand : {1, 2, 3, 4, 6})
    if (cand * npos <= 512 && cand <= D && D % cand == 0 && cand * npos >= min_cols) { zt = cand; break; }
  if (!zt) {  // min_cols out of reach: the largest feasible slab count
    zt = 1;
    for (int cand : {2, 3, 4, 6}) if (cand * npos <= 512 && cand <= D && D % cand == 0) zt = cand;
  }
  const int planes = zt + 2 * halo, lbo = (ty + 2 * halo) * hx * 16, plane_bytes = 8 * lbo;
  const int budget = FLAT_SMEM_MAX - 1024 - 512 - FLAT_EPI_SMEM - FLAT_A_SLACK;
  const int a_slots = std::max(planes, std::min(std::min(16, slots_per_plane * planes), (budget - 4 * FLAT_W_BYTES) / plane_bytes));
  const int w_slots = std::min(8, (budget - a_slots * plane_bytes) / FLAT_W_BYTES);
  if (w_slots < 2) return false;
  g->hx = hx; g->ty = ty; g->npos = npos; g->lbo = lbo; g->a_slots = a_slots; g->w_slots = w_slots; g->zt = zt;
  g->smem = 1024 + a_slots * plane_bytes + FLAT_A_SLACK + w_slots * FLAT_W_BYTES + FLAT_EPI_SMEM + 512;
  g->tiles_y = tiles_y; g->tiles_z = D / zt;
  return true;
}

enum ConvKernel {
  CONV_REF,      // CUDA-core reference kernel (DUNET_FLAG_REF_CONV); it reads none of the tiling below
  CONV_TC64,     // Cout = 64 z-stacked kernel (conv3d_tc64.cuh), ZT = 4, never split
  CONV_FLAT,     // flattened-plane kernel of the deep levels (conv3d_flat.cuh)
  CONV_GENERIC,  // generic voxel-as-M kernel (conv3d_tc.cuh)
};
// How one 3x3x3 conv runs: everything run_conv launches with and everything its callers size or decide from it.
struct ConvPlan {
  ConvKernel kernel = CONV_GENERIC;
  int cb = 0;                                       // input-channel block of the kernel and its tensor maps
  int zt = 0, tiles_x = 0, tiles_y = 0, tiles_z = 0;
  int tiles = 0;                                    // work items (= statistics rows) per sample and cout tile
  int ksplit = 1, ksub = 1;                         // K split ksplit ways, in units of 1/ksub of a 64-channel block
  bool fuse_input = false;                          // the conv may take its input normalised on load (FuseIn)
  FlatGeom flat;                                    // kernel == CONV_FLAT
};

// The one decision of which kernel runs a conv layer at U-Net level `lvl`, with which tiling and K split.  It depends on
// PER-SAMPLE shapes and the plan flags only, never on the batch: a window's result is bit-identical whatever it is batched
// with.  may_split = false never splits K (dunet_op_conv3x3x3 has no partial-tile buffers).
static ConvPlan conv_plan(const dunet_plan* p, const ConvW& c, int lvl, bool may_split) {
  const uint32_t flags = p->cfg.flags;
  ConvPlan g;
  g.cb = c.cb_ch;
  g.tiles_x = (p->W[lvl] + CONV_TX - 1) / CONV_TX;
  g.tiles_y = (p->H[lvl] + CONV_TY - 1) / CONV_TY;
  // ZT (z-slabs per work item) trades weight re-use (each streamed weight tile feeds ZT slabs) against parallelism, and
  // split-K trades parallelism against an fp32 partial round trip + a reduce launch.  Both are tuned for the way the path is
  // actually driven: 2-4 windows per launch (dual-stream half batches), so ~24+ work items per sample already fill the GPU.
  // Round 1 split K whenever a sample had < 96 items: at batch 4 that doubled the 24^3 / 12^3 launches into two waves of
  // half-K items, each still streaming its weights from L2, plus the reduce kernels (measured 0.31-0.38 of the tensor peak).
  // The Cout = 64 z-stacked kernel always uses ZT = 4.  ZT = 2 below 24 items per sample; split-K below 20.
  {
    const int tz4 = (p->D[lvl] + CONV_ZT - 1) / CONV_ZT;
    const int items4 = g.tiles_x * g.tiles_y * tz4 * c.n_tiles;
    g.zt = (items4 < 24 && !(c.coutp == 64 && c.cb_ch == 32)) ? 2 : CONV_ZT;
  }
  g.tiles_z = (p->D[lvl] + g.zt - 1) / g.zt;
  g.tiles = g.tiles_x * g.tiles_y * g.tiles_z;
  const int ctas = g.tiles * c.n_tiles, ncb = c.ncb();
  if (may_split && ncb >= 2 && ctas < 20) g.ksplit = std::max(1, std::min(ncb, 96 / ctas));
  if (flags & DUNET_FLAG_REF_CONV) {
    g.kernel = CONV_REF;
  } else if (flags & DUNET_FLAG_GENERIC_CONV) {
    g.kernel = CONV_GENERIC;
  } else if (c.coutp == 64 && g.ksplit == 1 && g.zt == CONV_ZT) {
    g.kernel = CONV_TC64;
    g.cb = c.cb64;
    // normalise-on-load needs a single 16-bit source (a split-precision conv, every conv in fp32x3 mode, reads hi + lo)
    g.fuse_input = !(flags & DUNET_FLAG_NO_FUSED_NORM) && !c.split && c.nb1 == 0;
  } else if (c.cb_ch == 64 && c.n_tile == 128 && flat_geom(&g.flat, p->D[lvl], p->H[lvl], p->W[lvl], 1, 160, 2)) {
    // Deep levels (row of at most 30 voxels, Cout a multiple of 128): swapped-operand flattened-plane kernel, split-K when a
    // sample has fewer than 36 items, until it has ~48
    g.kernel = CONV_FLAT;
    g.zt = g.flat.zt; g.tiles_x = 1; g.tiles_y = g.flat.tiles_y; g.tiles_z = g.flat.tiles_z;
    g.tiles = g.tiles_y * g.tiles_z;
    const int items1 = g.tiles * c.n_tiles;
    g.ksplit = 1;
    if (may_split && items1 < 36) {
      // K is split in units of 64-channel blocks; when a sample still has too few items, in units of one tz slice of a
      // block (9 taps), up to 16 ways
      const int want = (48 + items1 - 1) / items1;
      if (want > ncb) { g.ksub = 3; g.ksplit = std::max(1, std::min(std::min(3 * ncb, 16), want)); }
      else g.ksplit = std::max(1, std::min(ncb, want));
    }
  }
  return g;
}

enum DeconvKernel {
  DECONV_REF,      // CUDA-core reference kernel (DUNET_FLAG_REF_CONV)
  DECONV_TC,       // persistent deconv2_tc kernel (deconv2_tc.cuh)
  DECONV_FLAT,     // flattened-plane kernel in transposed-conv mode
  DECONV_GENERIC,  // generic voxel-as-M kernel in MODE_DECONV2
};
struct DeconvPlan {
  DeconvKernel kernel = DECONV_GENERIC;
  FlatGeom flat;  // kernel == DECONV_FLAT
};

// The one decision of which kernel runs the k2 s2 transposed conv d on U-Net level lvl_in (its input level)
static DeconvPlan deconv_plan(const dunet_plan* p, const DeconvW& d, int lvl_in) {
  DeconvPlan g;
  if (p->cfg.flags & DUNET_FLAG_REF_CONV) g.kernel = DECONV_REF;
  else if (d.parts == 3 || (p->cfg.flags & DUNET_FLAG_GENERIC_CONV)) g.kernel = DECONV_GENERIC;
  // Cin <= 128: the persistent, HBM-write-bound kernel (the flattened-plane kernel measured 37 vs 19 us on the 24 -> 48
  // up-conv, 2 windows)
  else if (d.cinp <= 128) g.kernel = DECONV_TC;
  // deep levels (Cin > 128): the flattened-plane kernel in transposed-conv mode (rows = (tap, cout), positions as N, no halo)
  else if (flat_geom(&g.flat, p->D[lvl_in], p->H[lvl_in], p->W[lvl_in], 0, 128, 3)) g.kernel = DECONV_FLAT;
  return g;
}

static int stats_nseg(long long vox) {
  long long n = (vox + 8191) / 8192;
  return (int)std::min<long long>(std::max<long long>(n, 1), 128);
}

static inline bool is_prec(const dunet_plan* p) { return (p->cfg.flags & DUNET_FLAG_FP32X3) != 0; }
static inline bool is_fp16(const dunet_plan* p) { return (p->cfg.flags & DUNET_FLAG_FP16) != 0; }
// dispatch a statement templated on the 16-bit storage format: DUNET_FMT(is_fp16(p), f<..., HF>(args))
#define DUNET_FMT(cond, ...)                               \
  do {                                                     \
    if (cond) { constexpr bool HF = true; __VA_ARGS__; }   \
    else { constexpr bool HF = false; __VA_ARGS__; }       \
  } while (0)
// a per-channel bias row (time-embedding projection), optionally one row per sample (n_stride floats apart)
struct BiasRef {
  const float* p = nullptr;
  int n_stride = 0;
  BiasRef at(int off) const { BiasRef r; r.p = p ? p + off : nullptr; r.n_stride = n_stride; return r; }
};
// activation of `ch` (padded) channels at U-Net level `lvl`, batch B, stored at workspace offset `off`: in fp32x3 mode the
// low part follows the high part
static inline Act ws_act_x(const dunet_plan* p, uint8_t* ws, size_t off, int ch, int lvl, int B, bool prec) {
  Act a;
  a.hi = reinterpret_cast<bf16*>(ws + off);
  a.lo = prec ? a.hi + (size_t)B * ch * (size_t)p->V[lvl] : nullptr;
  return a;
}
static inline Act ws_act(const dunet_plan* p, uint8_t* ws, size_t off, int ch, int lvl, int B) {
  return ws_act_x(p, ws, off, ch, lvl, B, is_prec(p));
}
// The ENCODER runs in split precision in fp32x3 mode and ALSO in fp16 mode: its feature maps are added into the denoiser
// at every level of every DDIM step, so its rounding error is the one error source that repeats identically N times
// (measured on a 96^3 window: 2/3 of the fp16 error variance; argmax agreement 99.90 % -> 99.94 % with an exact encoder).
// It is 2.6 % of the FLOPs, so 3x its MMAs costs ~5 %.  DUNET_FLAG_PLAIN_ENCODER switches this off (A-B measurements).
static inline bool enc_prec(const dunet_plan* p) {
  return is_prec(p) || (is_fp16(p) && !(p->cfg.flags & (DUNET_FLAG_PLAIN_ENCODER | DUNET_FLAG_REF_CONV)));
}
// 16-bit storage format of a tensor: fp16 in fp16 mode unless it is (part of) a split hi/lo bf16 pair
static inline bool fmt_h(const dunet_plan* p, bool prec) { return is_fp16(p) && !prec; }

static WsLayout ws_layout(const dunet_plan* p, int B) {
  WsLayout L;
  size_t off = 0;
  const size_t pm = is_prec(p) ? 2 : 1, pme = enc_prec(p) ? 2 : 1;  // denoiser / encoder tensors: 1 or 2 (hi + lo) parts
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
  auto act_m = [&](int ch, int lvl, size_t m) -> size_t { return (size_t)(m * (size_t)B * ch * (size_t)p->V[lvl] * sizeof(bf16)); };
  auto act = [&](int ch, int lvl) -> size_t { return act_m(ch, lvl, pm); };
  L.in_pack = take(act_m(p->in_pad, 0, std::max(pm, pme)));
  size_t raw_max = 0, part_max = 0, ss_max = 0, split_max = 0;
  auto upd = [&](const ConvW& c, int lvl) {
    raw_max = std::max(raw_max, act_m(c.coutp, lvl, c.split ? 2 : 1));
    const ConvPlan g = conv_plan(p, c, lvl, /*may_split=*/true);
    const size_t planes = (size_t)B * (c.coutp / 8);
    part_max = std::max(part_max, planes * std::max(g.tiles, 160) * 16 * sizeof(float));  // rows: tiles, reduction segments (<= 128) or persistent CTAs (<= #SMs)
    ss_max = std::max(ss_max, planes * 16 * sizeof(float));
    if (g.ksplit > 1) split_max = std::max(split_max, (size_t)g.ksplit * B * c.coutp * (size_t)p->V[lvl] * sizeof(float));
  };
  for (int l = 0; l < 5; ++l) { upd(p->enc[l].a, l); upd(p->enc[l].b, l); upd(p->den[l].a, l); upd(p->den[l].b, l); }
  for (int l = 4; l >= 1; --l) { upd(p->upc[l].a, l - 1); upd(p->upc[l].b, l - 1); }
  L.raw = take(raw_max);
  L.mid = take(raw_max);
  L.partial = take(part_max);
  L.ss = take(ss_max);
  L.splitk = take(split_max);
  L.affine = take(ss_max);  // [plane][16] affine maps for the normalise-on-load convs
  const int CP = p->C <= 8 ? 8 : (p->C <= 16 ? 16 : 32);  // voxel-major DDIM state, classes padded to the MMA column tiles
  L.x_t = take((size_t)B * CP * p->V[0] * sizeof(float));
  L.acc = take((size_t)B * CP * p->V[0] * sizeof(float));
  L.image = take((size_t)B * p->cfg.in_channels * p->V[0] * sizeof(float));  // cropped windows (dunet_infer_windows)
  for (int l = 0; l < 5; ++l) {
    L.emb[l] = take(act(p->fp[l], l));
    L.x[l] = take(act(p->fp[l], l));
    L.epool[l] = l ? take(act_m(p->fp[l - 1], l, pme)) : 0;
    L.dpool[l] = l ? take(act(p->fp[l - 1], l)) : 0;
    L.up[l] = l ? take(act(p->upp[l], l - 1)) : 0;
    L.u[l] = l ? take(act(p->uoutp[l], l - 1)) : 0;
  }
  L.total = off;
  return L;
}

// ------------------------------------------------------------------------------------------------ layer launchers
// optional per-CTA timeline buffer of the generic conv / transposed conv kernels (tools only; process-global by design:
// dunet_debug_set_conv_timeline is a debugging hook, see include/dunet.h)
static long long* g_conv_dbg = nullptr;
static int g_conv_dbg_count = 0;

// every tcgen05 kernel instantiation that exists: X(kernel, dynamic shared memory bytes)
#define DUNET_TC_KERNELS_H(X, H)                                                                  \
  X((conv3d_tc_kernel<32, 64, CONV_ZT, MODE_CONV3, H>), (ConvTc<32, 64, CONV_ZT, MODE_CONV3>::SMEM_BYTES))     \
  X((conv3d_tc_kernel<32, 128, CONV_ZT, MODE_CONV3, H>), (ConvTc<32, 128, CONV_ZT, MODE_CONV3>::SMEM_BYTES))   \
  X((conv3d_tc_kernel<64, 64, 2, MODE_CONV3, H>), (ConvTc<64, 64, 2, MODE_CONV3>::SMEM_BYTES))                 \
  X((conv3d_tc_kernel<64, 128, 2, MODE_CONV3, H>), (ConvTc<64, 128, 2, MODE_CONV3>::SMEM_BYTES))               \
  X((conv3d_tc_kernel<64, 64, CONV_ZT, MODE_CONV3, H>), (ConvTc<64, 64, CONV_ZT, MODE_CONV3>::SMEM_BYTES))     \
  X((conv3d_tc_kernel<64, 128, CONV_ZT, MODE_CONV3, H>), (ConvTc<64, 128, CONV_ZT, MODE_CONV3>::SMEM_BYTES))   \
  X((conv3d_tc_kernel<64, 128, 2, MODE_DECONV2, H>), (ConvTc<64, 128, 2, MODE_DECONV2>::SMEM_BYTES))           \
  X((conv3d_tc64_kernel<32, CONV_ZT, false, H>), (ConvTc64<32, CONV_ZT>::SMEM_BYTES))                          \
  X((conv3d_tc64_kernel<32, CONV_ZT, true, H>), (ConvTc64<32, CONV_ZT>::SMEM_BYTES))                           \
  X((conv3d_tc64_kernel<64, CONV_ZT, false, H>), (ConvTc64<64, CONV_ZT>::SMEM_BYTES))                          \
  X((conv3d_tc64_kernel<64, CONV_ZT, true, H>), (ConvTc64<64, CONV_ZT>::SMEM_BYTES))                           \
  X((deconv2_tc_kernel<1, 2, H>), (DeconvTc<1, 2>::SMEM_BYTES))                                                \
  X((deconv2_tc_kernel<2, 2, H>), (DeconvTc<2, 2>::SMEM_BYTES))                                                \
  X((conv3d_flat_kernel<1, H>), FLAT_SMEM_MAX)                                                                 \
  X((conv3d_flat_kernel<2, H>), FLAT_SMEM_MAX)                                                                 \
  X((conv3d_flat_kernel<3, H>), FLAT_SMEM_MAX)                                                                 \
  X((conv3d_flat_kernel<4, H>), FLAT_SMEM_MAX)                                                                 \
  X((conv3d_flat_kernel<6, H>), FLAT_SMEM_MAX)

// Per-DEVICE one-time setup (the dynamic shared memory opt-in of a kernel is a per-device attribute): keyed by device
// id, mutex-protected.  Called from dunet_plan_create and the standalone dunet_op_* entry points, never on the per-step
// path.  Returns the SM count of the current device.
static std::mutex g_dev_mu;
static std::unordered_map<int, int> g_dev_sms;
static int dev_prepare(int* sms_out) {
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(g_dev_mu);
  auto it = g_dev_sms.find(dev);
  if (it == g_dev_sms.end()) {
    int sms = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
#define DUNET_SET_SMEM(K, BYTES) CUDA_TRY(cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, BYTES));
    DUNET_TC_KERNELS_H(DUNET_SET_SMEM, false)
    DUNET_TC_KERNELS_H(DUNET_SET_SMEM, true)
#undef DUNET_SET_SMEM
    it = g_dev_sms.emplace(dev, sms).first;
  }
  if (sms_out) *sms_out = it->second;
  return 0;
}

template <int CB_CH, int N_TILE, int ZT, int MODE, bool H>
static int launch_conv_tc(const dunet_plan* p, const CUtensorMap (&t)[4], const ConvTcArgs& a, cudaStream_t st, int conv_tag = PROF_CONV) {
  using Cfg = ConvTc<CB_CH, N_TILE, ZT, MODE>;
  auto kern = conv3d_tc_kernel<CB_CH, N_TILE, ZT, MODE, H>;
  const long long items = (long long)a.tiles_x * a.tiles_y * a.tiles_z * a.n_tiles * a.ksplit * a.batch;
  // persistent: one CTA per SM (each may own all 512 TMEM columns) walking the work items round-robin
  const long long grid = std::min<long long>(items, (long long)p->num_sms);
  TRY(prof_begin(conv_tag, st));  // MODE_DECONV2 callers pass their PROF_DECONV / PROF_DECONV_SMALL tag
  launch_k(kern, dim3((unsigned)grid), dim3(CONV_TC_THREADS), Cfg::SMEM_BYTES, st, t[0], t[1], t[2], t[3], a);
  LAUNCH_CHECK();
  TRY(prof_end(st));
  return 0;
}

template <int CB_CH, bool FUSE, bool H>
static int launch_conv_tc64(const dunet_plan* p, const CUtensorMap (&t)[4], const ConvTc64Args& a, unsigned* grid_out, cudaStream_t st,
                            int conv_tag = PROF_CONV) {
  using Cfg = ConvTc64<CB_CH, CONV_ZT>;
  auto kern = conv3d_tc64_kernel<CB_CH, CONV_ZT, FUSE, H>;
  const long long tiles = (long long)a.tiles_x * a.tiles_y * a.tiles_z * a.batch;
  const unsigned grid = (unsigned)std::min<long long>(tiles, p->num_sms);
  *grid_out = grid;
  TRY(prof_begin(conv_tag, st));
  launch_k(kern, dim3(grid), dim3(FUSE ? Cfg::THREADS_FUSED : CONV_THREADS), Cfg::SMEM_BYTES, st, t[0], t[1], t[2], t[3], a);
  LAUNCH_CHECK();
  TRY(prof_end(st));
  return 0;
}

// the flattened-plane kernel (3x3x3 conv, or transposed conv with f.deconv) on geometry g; h: fp16 storage
static int launch_flat(const dunet_plan* p, const CUtensorMap (&t)[4], ConvFlatArgs f, const FlatGeom& g, bool h, int tag, cudaStream_t st) {
  f.hx = g.hx; f.ty = g.ty; f.tiles_y = g.tiles_y; f.tiles_z = g.tiles_z;
  f.npos = g.npos; f.lbo = g.lbo; f.a_slots = g.a_slots; f.w_slots = g.w_slots;
  const long long items = (long long)f.tiles_y * f.tiles_z * f.n_tiles * f.ksplit * f.batch;
  const unsigned grid = (unsigned)std::min<long long>(items, p->num_sms);
  TRY(prof_begin(tag, st));
  DUNET_FMT(h, {
    switch (g.zt) {
      case 1: launch_k(conv3d_flat_kernel<1, HF>, dim3(grid), dim3(FLAT_THREADS), (size_t)g.smem, st, t[0], t[1], t[2], t[3], f); break;
      case 2: launch_k(conv3d_flat_kernel<2, HF>, dim3(grid), dim3(FLAT_THREADS), (size_t)g.smem, st, t[0], t[1], t[2], t[3], f); break;
      case 3: launch_k(conv3d_flat_kernel<3, HF>, dim3(grid), dim3(FLAT_THREADS), (size_t)g.smem, st, t[0], t[1], t[2], t[3], f); break;
      case 4: launch_k(conv3d_flat_kernel<4, HF>, dim3(grid), dim3(FLAT_THREADS), (size_t)g.smem, st, t[0], t[1], t[2], t[3], f); break;
      default: launch_k(conv3d_flat_kernel<6, HF>, dim3(grid), dim3(FLAT_THREADS), (size_t)g.smem, st, t[0], t[1], t[2], t[3], f); break;
    }
  });
  LAUNCH_CHECK();
  TRY(prof_end(st));
  return 0;
}

// tools: the timeline buffer for this generic / flattened-plane conv launch -- only the DUNET_DBG_LAUNCH-th one since the
// buffer was set (default: every launch)
static long long* conv_dbg_stamp() {
  static const int target = [] { const char* e = getenv("DUNET_DBG_LAUNCH"); return e ? atoi(e) : -1; }();
  long long* dbg = (g_conv_dbg && (target < 0 || g_conv_dbg_count == target)) ? g_conv_dbg : nullptr;
  if (g_conv_dbg) ++g_conv_dbg_count;
  return dbg;
}

// block list of a conv: bf16 mode [S0, S1]; fp32x3 mode [S0.hi, S1.hi | S0.lo, S1.lo | S0.hi, S1.hi] (tensor maps 0..3 =
// S0.hi, S1.hi, S0.lo, S1.lo), matching the packed weight blocks [W.hi | W.hi | W.lo]
static ConvSegs make_segs(int nb0, int chunks0, int nb1, int chunks1, bool prec) {
  ConvSegs sg;
  memset(&sg, 0, sizeof sg);
  auto add = [&](int tm, int nb, int chunks) {
    if (nb > 0) { sg.s[sg.n].tmap = tm; sg.s[sg.n].nblocks = nb; sg.s[sg.n].chunks = chunks; ++sg.n; sg.ncb += nb; }
  };
  add(0, nb0, chunks0); add(1, nb1, chunks1);
  if (prec) { add(2, nb0, chunks0); add(3, nb1, chunks1); add(0, nb0, chunks0); add(1, nb1, chunks1); }
  return sg;
}

// normalise-on-load request for run_conv: src0 is the RAW output of the previous conv, to be seen through
// LeakyReLU(x * scale + shift) + bias (in_affine_kernel output + optional time-embedding bias row)
struct FuseIn {
  const float* affine = nullptr;
  BiasRef bias;
};

// 3x3x3 conv as planned by conv_plan -> raw output (bf16, or hi + lo in fp32x3 mode) + InstanceNorm partial statistics
// [plane][*nseg_out][16].  With `pending_split` a K-split conv of a small level may leave its fp32 partial tiles un-reduced
// (*pending_split = ksplit): the caller's run_norm then sums, normalises and activates them in one launch (splitk_norm_kernel).
static bool splitk_norm_ok(const dunet_plan* p, bool prec, int lvl) {
  return !prec && p->V[lvl] <= SKN_MAX_VOX && p->D[lvl] % 2 == 0 && p->H[lvl] % 2 == 0 && p->W[lvl] % 2 == 0;
}
static int run_conv(const dunet_plan* p, const ConvW& c, const ConvPlan& cp, Act src0, Act src1, Act out, float* partial,
                    float* splitk, int* nseg_out, int lvl, int B, cudaStream_t st, const FuseIn* fuse = nullptr,
                    int* pending_split = nullptr) {
  if (pending_split) *pending_split = 0;
  const int D = p->D[lvl], H = p->H[lvl], W = p->W[lvl];
  const int planes = B * (c.coutp / 8);
  const bool prec = c.split, pairs_in = prec && !c.triple;  // triple: one packed source tensor already holds hi, lo, hi
  if (prec && (!out.lo || (pairs_in && (!src0.lo || (c.nb1 > 0 && !src1.lo))))) return fail(DUNET_E_STATE, "split-precision conv needs hi + lo tensors");
  if (fuse && !cp.fuse_input) return fail(DUNET_E_STATE, "normalise-on-load requested for a conv that cannot take it");
  if (cp.ksplit > 1 && (!partial || !splitk)) return fail(DUNET_E_STATE, "K-split conv without partial-tile buffers");
  if (cp.kernel == CONV_REF) {
    if (prec) return fail(DUNET_E_UNSUPPORTED, "DUNET_FLAG_REF_CONV and DUNET_FLAG_FP32X3 are mutually exclusive");
    if (!c.w32) return fail(DUNET_E_STATE, "DUNET_FLAG_REF_CONV needs DUNET_FLAG_KEEP_FP32_WEIGHTS");
    // the debug kernel writes only the chunks holding real output channels; padded chunks must still be zero
    CUDA_TRY(cudaMemsetAsync(out.hi, 0, (size_t)B * c.coutp * p->V[lvl] * sizeof(bf16), st));
    DUNET_FMT(fmt_h(p, prec), conv3d_ref_kernel<HF><<<grid_for((long long)B * ((c.coutr + 7) / 8) * p->V[lvl], 128, 148 * 64), 128, 0, st>>>(
        src0.hi, c.c0r, c.c0p / 8, src1.hi, c.c1r, c.c1p / 8, c.w32, out.hi, c.coutr, c.coutp / 8, D, H, W, B, c.rot));
    LAUNCH_CHECK();
    if (partial) {
      const int nseg = stats_nseg(p->V[lvl]);
      DUNET_FMT(fmt_h(p, prec), in_stats_kernel<HF><<<dim3(nseg, planes), STATS_THREADS, 0, st>>>(out.hi, partial, p->V[lvl], nseg));
      LAUNCH_CHECK();
      *nseg_out = nseg;
    }
    return 0;
  }
  const int conv_tag = (prec && !is_prec(p)) ? PROF_CONV_SPLIT : PROF_CONV;
  if (PROF_ON) {
    const double fl = 2.0 * B * (double)p->V[lvl] * c.coutr * 27.0 * (c.c0r + c.c1r);
    prof_of(p)->bytes[conv_tag] += fl;
    if (conv_tag == PROF_CONV) prof_of(p)->flops += fl;
  }
  const ConvSegs segs = make_segs(c.c0p / cp.cb, c.c0p / 8, c.c1p / cp.cb, c.c1p / 8, pairs_in);
  auto tmap = [&](CUtensorMap* m, const bf16* base, int ch) {
    return cp.kernel == CONV_FLAT ? make_flat_tmap(m, base, B * (ch / 8), D, H, W, cp.flat.hx, cp.flat.ty)
                                  : make_act_tmap(m, base, B * (ch / 8), D, H, W, cp.cb / 8, 1);
  };
  CUtensorMap t[4];  // S0.hi, S1.hi, S0.lo, S1.lo (see make_segs); the unused ones repeat map 0
  TRY(tmap(&t[0], src0.hi, c.c0p));
  t[1] = t[2] = t[3] = t[0];
  if (c.nb1 > 0) TRY(tmap(&t[1], src1.hi, c.c1p));
  if (pairs_in) {
    TRY(tmap(&t[2], src0.lo, c.c0p));
    if (c.nb1 > 0) TRY(tmap(&t[3], src1.lo, c.c1p));
  }
  switch (cp.kernel) {
    case CONV_TC64: {
      if (!c.packed64) return fail(DUNET_E_STATE, "conv weights not packed for the Cout = 64 kernel");
      ConvTc64Args b;
      memset(&b, 0, sizeof b);
      b.w = c.packed64; b.out = out.hi; b.out_lo = out.lo; b.stats = partial; b.segs = segs;
      b.D = D; b.H = H; b.W = W; b.tiles_x = cp.tiles_x; b.tiles_y = cp.tiles_y; b.tiles_z = cp.tiles_z; b.batch = B;
      unsigned grid = 0;
      if (fuse) {
        b.in_affine = fuse->affine; b.in_bias = fuse->bias.p; b.in_bias_n_stride = fuse->bias.n_stride; b.slope = 0.1f;
        DUNET_FMT(fmt_h(p, prec), TRY(cp.cb == 32 ? (launch_conv_tc64<32, true, HF>(p, t, b, &grid, st, conv_tag)) : (launch_conv_tc64<64, true, HF>(p, t, b, &grid, st, conv_tag))));
      } else {
        DUNET_FMT(fmt_h(p, prec), TRY(cp.cb == 32 ? (launch_conv_tc64<32, false, HF>(p, t, b, &grid, st, conv_tag)) : (launch_conv_tc64<64, false, HF>(p, t, b, &grid, st, conv_tag))));
      }
      if (partial) *nseg_out = (int)grid;  // one statistics row per persistent CTA and sample
      return 0;
    }
    case CONV_FLAT: {
      ConvFlatArgs f;
      memset(&f, 0, sizeof f);
      f.w = c.packed; f.out = out.hi; f.out_lo = out.lo; f.segs = segs;
      f.cout = c.coutp; f.D = D; f.H = H; f.W = W; f.n_tiles = c.n_tiles; f.batch = B;
      f.ksplit = cp.ksplit; f.ksub = cp.ksub;
      f.dbg = conv_dbg_stamp();
      if (cp.ksplit > 1) f.out_partial = splitk;
      else f.stats = partial;
      TRY(launch_flat(p, t, f, cp.flat, fmt_h(p, prec), conv_tag, st));
      break;
    }
    default: {  // CONV_GENERIC
      ConvTcArgs a;
      memset(&a, 0, sizeof a);
      a.w = c.packed; a.out = out.hi; a.out_lo = out.lo; a.segs = segs;
      a.cout = c.coutp; a.D = D; a.H = H; a.W = W;
      a.tiles_x = cp.tiles_x; a.tiles_y = cp.tiles_y; a.tiles_z = cp.tiles_z; a.n_tiles = c.n_tiles; a.batch = B;
      a.ksplit = cp.ksplit;
      a.dbg = conv_dbg_stamp();
      if (cp.ksplit > 1) a.out_partial = splitk;
      else a.stats = partial;
      int rc = 0;
      DUNET_FMT(fmt_h(p, prec), {
        if (c.cb_ch == 32 && c.n_tile == 64) rc = launch_conv_tc<32, 64, CONV_ZT, MODE_CONV3, HF>(p, t, a, st, conv_tag);
        else if (c.cb_ch == 32 && c.n_tile == 128) rc = launch_conv_tc<32, 128, CONV_ZT, MODE_CONV3, HF>(p, t, a, st, conv_tag);
        else if (c.cb_ch == 64 && c.n_tile == 64 && cp.zt == 2) rc = launch_conv_tc<64, 64, 2, MODE_CONV3, HF>(p, t, a, st, conv_tag);
        else if (c.cb_ch == 64 && c.n_tile == 128 && cp.zt == 2) rc = launch_conv_tc<64, 128, 2, MODE_CONV3, HF>(p, t, a, st, conv_tag);
        else if (c.cb_ch == 64 && c.n_tile == 64) rc = launch_conv_tc<64, 64, CONV_ZT, MODE_CONV3, HF>(p, t, a, st, conv_tag);
        else if (c.cb_ch == 64 && c.n_tile == 128) rc = launch_conv_tc<64, 128, CONV_ZT, MODE_CONV3, HF>(p, t, a, st, conv_tag);
        else rc = fail(DUNET_E_UNSUPPORTED, "no conv instantiation for cb_ch=%d n_tile=%d", c.cb_ch, c.n_tile);
      });
      TRY(rc);
      break;
    }
  }
  // flattened-plane and generic kernels: one statistics row per tile, or K-split partial tiles to sum
  if (cp.ksplit == 1) {
    if (partial) *nseg_out = cp.tiles;
    return 0;
  }
  if (pending_split && splitk_norm_ok(p, prec, lvl)) {
    *pending_split = cp.ksplit;
    *nseg_out = 0;
    return 0;
  }
  const int nseg = (int)std::min<long long>(std::max<long long>((p->V[lvl] + 255) / 256, 1), 128);
  if (PROF_ON) prof_of(p)->bytes[PROF_SPLITK] += (double)B * c.coutp * (double)p->V[lvl] * (4.0 * cp.ksplit + (prec ? 4.0 : 2.0));
  TRY(prof_begin(PROF_SPLITK, st));
  DUNET_FMT(fmt_h(p, prec), launch_k(splitk_reduce_stats_kernel<HF>, dim3(nseg, planes), dim3(STATS_THREADS), 0, st, (const float*)splitk, cp.ksplit,
           (long long)B * c.coutp * p->V[lvl], out.hi, out.lo, partial, (long long)p->V[lvl], nseg));
  LAUNCH_CHECK();
  TRY(prof_end(st));
  *nseg_out = nseg;
  return 0;
}

// statistics (reduced in the kernel prologue) -> fused normalise/activation(/bias/add/pool)
static int run_norm(const dunet_plan* p, const ConvW& c, Act raw, const float* partial, int nseg, BiasRef bias, Act add,
                    Act out, Act pooled, int lvl, int B, cudaStream_t st, int pending_split = 0, const float* splitk = nullptr) {
  const int planes = B * (c.coutp / 8);
  const bool prec = raw.lo != nullptr;
  NormActArgs a;
  memset(&a, 0, sizeof a);
  a.raw = raw.hi; a.partial = partial; a.nseg = nseg; a.gamma = c.gamma; a.beta = c.beta; a.bias = bias.p; a.bias_n_stride = bias.n_stride; a.add = add.hi;
  a.out = out.hi; a.pooled = pooled.hi; a.raw_lo = raw.lo; a.add_lo = add.lo; a.out_lo = out.lo; a.pooled_lo = pooled.lo;
  a.chunks = c.coutp / 8; a.D = p->D[lvl]; a.H = p->H[lvl]; a.W = p->W[lvl];
  a.eps = 1e-5f; a.slope = 0.1f;
  if (pending_split > 1) {
    // the conv left its K-split partial tiles un-reduced: sum + statistics + normalise (+ pool) in one launch
    if (prec || !splitk || add.lo || p->V[lvl] > SKN_MAX_VOX) return fail(DUNET_E_STATE, "fused split-K normalise: unsupported configuration");
    SplitkNormArgs k;
    k.part = splitk; k.ksplit = pending_split; k.split_stride = (long long)B * c.coutp * p->V[lvl]; k.n = a;
    if (PROF_ON) prof_of(p)->bytes[PROF_NORM_SMALL] += (double)B * c.coutp * (double)p->V[lvl] * (4.0 * pending_split + 2.0 + (add.hi ? 2.0 : 0.0) + (pooled.hi ? 0.25 : 0.0));
    TRY(prof_begin(PROF_NORM_SMALL, st));
#define DUNET_SKN(ADDF, POOLF) DUNET_FMT(is_fp16(p), launch_k(splitk_norm_kernel<ADDF, POOLF, HF>, dim3(planes), dim3(256), 0, st, k))
    if (add.hi && pooled.hi) DUNET_SKN(true, true);
    else if (add.hi) DUNET_SKN(true, false);
    else if (pooled.hi) DUNET_SKN(false, true);
    else DUNET_SKN(false, false);
#undef DUNET_SKN
    LAUNCH_CHECK();
    TRY(prof_end(st));
    return 0;
  }
  // 8 blocks per SM in total (2 to 32 measured slower), each streaming a long contiguous range of one 8-channel plane (the
  // statistics prologue is paid once per block)
  const int per_plane = std::max(1, (148 * 8 + planes - 1) / planes);
  // one bf16 read + one bf16 write per element (+ read of the residual, + 1/8 write of the pooled tensor); launches that move
  // less than 64 MB are launch-latency bound and are reported as their own family so that the HBM roofline of the large
  // ones stays readable
  const double nbytes = (prec ? 2.0 : 1.0) * B * c.coutp * (double)p->V[lvl] * (4.0 + (add.hi ? 2.0 : 0.0) + (pooled.hi ? 0.25 : 0.0));
  const int ptag = nbytes >= 64e6 ? PROF_NORM : PROF_NORM_SMALL;
  if (PROF_ON) prof_of(p)->bytes[ptag] += nbytes;
  TRY(prof_begin(ptag, st));
  const int mode = prec ? MODE_FP32X3 : (is_fp16(p) ? MODE_FP16 : MODE_BF16);
  if (prec && add.hi && !add.lo) return fail(DUNET_E_STATE, "fp32x3 normalise needs a hi + lo residual");
  if (!prec && add.lo) return fail(DUNET_E_STATE, "16-bit normalise cannot take a hi + lo residual");
  a.out_single_h = (prec && !out.lo) ? 1 : 0;  // split-precision producer, fp16 consumer (encoder feature maps in fp16 mode)
  if (a.out_single_h && !is_fp16(p)) return fail(DUNET_E_STATE, "single-tensor output of a split-precision pass exists in fp16 mode only");
#define DUNET_NORM(KERN, GRID)                                                                     \
  do {                                                                                             \
    if (mode == MODE_FP32X3) {                                                                     \
      if (add.hi) launch_k(KERN<true, MODE_FP32X3>, GRID, dim3(NORM_THREADS), 0, st, a);           \
      else launch_k(KERN<false, MODE_FP32X3>, GRID, dim3(NORM_THREADS), 0, st, a);                 \
    } else if (mode == MODE_FP16) {                                                                \
      if (add.hi) launch_k(KERN<true, MODE_FP16>, GRID, dim3(NORM_THREADS), 0, st, a);             \
      else launch_k(KERN<false, MODE_FP16>, GRID, dim3(NORM_THREADS), 0, st, a);                   \
    } else {                                                                                       \
      if (add.hi) launch_k(KERN<true, MODE_BF16>, GRID, dim3(NORM_THREADS), 0, st, a);             \
      else launch_k(KERN<false, MODE_BF16>, GRID, dim3(NORM_THREADS), 0, st, a);                   \
    }                                                                                              \
  } while (0)
  if (pooled.hi) {
    const dim3 grid(grid_for(p->V[lvl] / 4, NORM_THREADS, per_plane), planes);
    DUNET_NORM(norm_act_pool_kernel, grid);
  } else {
    const dim3 grid(grid_for(p->V[lvl], NORM_THREADS * (prec ? 2 : 4), per_plane), planes);
    DUNET_NORM(norm_act_kernel, grid);
  }
#undef DUNET_NORM
  LAUNCH_CHECK();
  TRY(prof_end(st));
  return 0;
}

// conv -> IN -> LReLU (+temb bias) -> conv -> IN -> LReLU (+add, +pool).  With `defer_last_norm` the second normalise
// pass is left to the consumer (the final 1x1 conv kernel applies it on the fly): the raw output stays in ws.raw and
// *nseg_out describes its statistics rows in ws.partial.
static int run_twoconv(const dunet_plan* p, const TwoConvW& t, Act src0, Act src1, BiasRef temb_bias, Act add, Act out,
                       Act pooled, int lvl, int B, uint8_t* ws, const WsLayout& L, cudaStream_t st,
                       bool defer_last_norm = false, int* nseg_out = nullptr, Act* raw_out = nullptr) {
  const bool tp = t.a.split;  // this block runs in split precision (hi + lo tensors)
  const Act raw_a = ws_act_x(p, ws, L.raw, t.a.coutp, lvl, B, tp), mid = ws_act_x(p, ws, L.mid, t.a.coutp, lvl, B, tp);
  const Act raw_b = ws_act_x(p, ws, L.raw, t.b.coutp, lvl, B, tp);
  float* partial = reinterpret_cast<float*>(ws + L.partial);
  float* splitk = reinterpret_cast<float*>(ws + L.splitk);
  int nseg = 0, ps_a = 0;
  const ConvPlan pa = conv_plan(p, t.a, lvl, /*may_split=*/true), pb = conv_plan(p, t.b, lvl, /*may_split=*/true);
  TRY(run_conv(p, t.a, pa, src0, src1, raw_a, partial, splitk, &nseg, lvl, B, st, nullptr, pb.fuse_input ? nullptr : &ps_a));
  if (pb.fuse_input) {
    // conv_1 normalises conv_0's raw output on load: only the affine map is materialised.  conv_1 writes its own raw
    // output to ws.mid (ws.raw is still being read) -- callers get the buffer through *raw_out.
    float* affine = reinterpret_cast<float*>(ws + L.affine);
    const int planes = B * (t.a.coutp / 8);
    TRY(prof_begin(PROF_OTHER, st));
    launch_k(in_affine_kernel, dim3(planes), dim3(256), 0, st, (const float*)partial, nseg, (const float*)t.a.gamma,
             (const float*)t.a.beta, t.a.coutp / 8, (double)p->V[lvl], 1e-5f, affine);
    LAUNCH_CHECK();
    TRY(prof_end(st));
    FuseIn f;
    f.affine = affine; f.bias = temb_bias;
    const Act raw_b2 = ws_act_x(p, ws, L.mid, t.b.coutp, lvl, B, tp);
    TRY(run_conv(p, t.b, pb, raw_a, Act(), raw_b2, partial, splitk, &nseg, lvl, B, st, &f));
    if (raw_out) *raw_out = raw_b2;
    if (defer_last_norm) {
      *nseg_out = nseg;
      return 0;
    }
    TRY(run_norm(p, t.b, raw_b2, partial, nseg, BiasRef(), add, out, pooled, lvl, B, st));
    return 0;
  }
  if (raw_out) *raw_out = raw_b;
  int ps = 0;  // K-split partial tiles left for the normalise pass (deep levels, see run_conv)
  TRY(run_norm(p, t.a, raw_a, partial, nseg, temb_bias, Act(), mid, Act(), lvl, B, st, ps_a, splitk));
  TRY(run_conv(p, t.b, pb, mid, Act(), raw_b, partial, splitk, &nseg, lvl, B, st, nullptr, (defer_last_norm || raw_out) ? nullptr : &ps));
  if (defer_last_norm) {
    *nseg_out = nseg;
    return 0;
  }
  TRY(run_norm(p, t.b, raw_b, partial, nseg, BiasRef(), add, out, pooled, lvl, B, st, ps, splitk));
  return 0;
}

static int run_deconv(const dunet_plan* p, const DeconvW& d, Act in, Act out, int lvl_in, int B, cudaStream_t st) {
  const bool prec = d.parts == 3;
  const DeconvPlan dp = deconv_plan(p, d, lvl_in);
  if (dp.kernel == DECONV_REF) {  // CUDA-core debug kernel
    if (prec) return fail(DUNET_E_UNSUPPORTED, "DUNET_FLAG_REF_CONV and DUNET_FLAG_FP32X3 are mutually exclusive");
    const long long total = (long long)B * (d.coutp / 8) * 8 * p->V[lvl_in];
    DUNET_FMT(fmt_h(p, prec), deconv2_kernel<HF><<<grid_for(total, 256, 148 * 32), 256, 0, st>>>(in.hi, d.cinp, d.packed, d.bias, out.hi, d.coutp,
                                                                                         p->D[lvl_in], p->H[lvl_in], p->W[lvl_in], B));
    LAUNCH_CHECK();
    return 0;
  }
  if (prec && (!in.lo || !out.lo)) return fail(DUNET_E_STATE, "fp32x3 transposed conv needs hi + lo tensors");
  const int D = p->D[lvl_in], H = p->H[lvl_in], W = p->W[lvl_in];
  // like the normalise launches: below 64 MB a launch is latency bound and is reported as its own family
  const double dbytes = (prec ? 2.0 : 1.0) * B * (double)p->V[lvl_in] * 2.0 * (d.cinp + 8.0 * d.coutp);
  const int dtag = dbytes >= 64e6 ? PROF_DECONV : PROF_DECONV_SMALL;
  if (PROF_ON) prof_of(p)->bytes[dtag] += dbytes;
  CUtensorMap t[4];
  switch (dp.kernel) {
    case DECONV_TC: {
      TRY(make_act_tmap(&t[0], in.hi, B * (d.cinp / 8), D, H, W, 8, 0));
      DeconvTcArgs b;
      memset(&b, 0, sizeof b);
      b.w = d.packed_tc; b.out = out.hi; b.bias = d.bias; b.chunks_in = d.cinp / 8; b.cout = d.coutp; b.D = D; b.H = H; b.W = W;
      b.tiles_x = (W + CONV_TX - 1) / CONV_TX; b.tiles_y = (H + CONV_TY - 1) / CONV_TY; b.tiles_z = (D + 1) / 2;
      b.n_tiles = 8 * d.coutp / 128; b.batch = B; b.dbg = getenv("DUNET_DBG_DECONV") ? g_conv_dbg : nullptr;
      const long long tiles = (long long)b.tiles_x * b.tiles_y * b.tiles_z * B;
      const unsigned grid = (unsigned)std::min<long long>(tiles, p->num_sms);
      TRY(prof_begin(dtag, st));
      if (d.cinp == 64) DUNET_FMT(is_fp16(p), launch_k(deconv2_tc_kernel<1, 2, HF>, dim3(grid), dim3(DeconvTc<1, 2>::THREADS), DeconvTc<1, 2>::SMEM_BYTES, st, t[0], b));
      else DUNET_FMT(is_fp16(p), launch_k(deconv2_tc_kernel<2, 2, HF>, dim3(grid), dim3(DeconvTc<2, 2>::THREADS), DeconvTc<2, 2>::SMEM_BYTES, st, t[0], b));
      LAUNCH_CHECK();
      TRY(prof_end(st));
      return 0;
    }
    case DECONV_FLAT: {
      TRY(make_flat_tmap(&t[0], in.hi, B * (d.cinp / 8), D, H, W, dp.flat.hx, dp.flat.ty, 0));
      t[1] = t[2] = t[3] = t[0];
      ConvFlatArgs f;
      memset(&f, 0, sizeof f);
      f.w = d.packed_tc; f.out = out.hi; f.bias = d.bias; f.deconv = 1;
      f.segs = make_segs(d.cinp / 64, d.cinp / 8, 0, 0, false);
      f.cout = d.coutp; f.D = D; f.H = H; f.W = W; f.n_tiles = 8 * d.coutp / 128; f.batch = B; f.ksplit = 1; f.ksub = 1;
      return launch_flat(p, t, f, dp.flat, is_fp16(p), dtag, st);
    }
    default: {  // DECONV_GENERIC
      TRY(make_act_tmap(&t[0], in.hi, B * (d.cinp / 8), D, H, W, 8, 0));
      t[1] = t[2] = t[3] = t[0];
      if (prec) TRY(make_act_tmap(&t[1], in.lo, B * (d.cinp / 8), D, H, W, 8, 0));
      ConvTcArgs a;
      memset(&a, 0, sizeof a);
      a.w = d.packed_tc; a.out = out.hi; a.out_lo = out.lo; a.bias = d.bias;
      // fp32x3: [in.hi | in.lo | in.hi] x [W.hi | W.hi | W.lo]
      a.segs = make_segs(d.cinp / 64, d.cinp / 8, 0, 0, false);
      if (prec) {
        a.segs.n = 3; a.segs.ncb = 3 * (d.cinp / 64);
        a.segs.s[1] = a.segs.s[0]; a.segs.s[1].tmap = 1;
        a.segs.s[2] = a.segs.s[0];
      }
      a.cout = d.coutp; a.D = D; a.H = H; a.W = W;
      a.tiles_x = (W + CONV_TX - 1) / CONV_TX; a.tiles_y = (H + CONV_TY - 1) / CONV_TY; a.tiles_z = (D + 1) / 2;
      a.n_tiles = 8 * d.coutp / 128; a.ksplit = 1; a.batch = B; a.dbg = nullptr;
      int rc = 0;
      DUNET_FMT(fmt_h(p, prec), rc = launch_conv_tc<64, 128, 2, MODE_DECONV2, HF>(p, t, a, st, dtag));
      return rc;
    }
  }
}

// Sub-batches of a batch of B windows.  With DUNET_FLAG_DUAL_STREAM a batch of >= 4 windows (2-3 measured within noise)
// runs as two half batches of B0 = ceil(B / 2) windows on the plan's internal streams.  Half h holds windows
// [h * B0, h * B0 + nb) and the workspace part at h * ws_stride, which is laid out for nb windows (ws_layout(p, nb) of a
// shorter last half fits in the B0-window part).  Otherwise there is one part: the whole batch and workspace.
struct SubBatches {
  int n, B0;
  size_t ws_stride;
};
static SubBatches sub_batches(const dunet_plan* p, int B, bool dual) {
  SubBatches s;
  s.n = dual ? 2 : 1;
  s.B0 = (B + s.n - 1) / s.n;
  s.ws_stride = ws_layout(p, s.B0).total;
  return s;
}
static bool dual_batch(const dunet_plan* p, int B) { return B >= 4 && (p->cfg.flags & DUNET_FLAG_DUAL_STREAM); }
// Does this call run as two sub-batches?  Not while the profiler is on (kernel times would overlap).  A call that skips
// the encoder must read the embeddings back through the partition they were written with.
static bool use_dual(dunet_plan* p, int B, int run_encoder) {
  const bool dual = run_encoder ? (dual_batch(p, B) && !PROF_ON) : (p->emb_dual && p->emb_B == B);
  if (run_encoder) { p->emb_B = B; p->emb_dual = dual; }
  return dual;
}
// body(b0, nb, ws_h, stream_h) for every sub-batch: one part runs on the caller's stream; two parts are forked from the
// caller's stream onto half_stream[h] and joined back into it with events (device-side waits, no host synchronisation)
template <typename Body>
static int run_sub_batches(dunet_plan* p, const SubBatches& s, int B, uint8_t* ws, cudaStream_t st, Body&& body) {
  if (s.n == 1) return body(0, B, ws, st);
  CUDA_TRY(cudaEventRecord(p->ev_fork, st));
  for (int h = 0; h < s.n; ++h) {
    CUDA_TRY(cudaStreamWaitEvent(p->half_stream[h], p->ev_fork, 0));
    TRY(body(h * s.B0, std::min(s.B0, B - h * s.B0), ws + h * s.ws_stride, p->half_stream[h]));
    CUDA_TRY(cudaEventRecord(p->ev_join[h], p->half_stream[h]));
  }
  for (int h = 0; h < s.n; ++h) CUDA_TRY(cudaStreamWaitEvent(st, p->ev_join[h], 0));
  return 0;
}

static int check_call(const dunet_plan* p, int B, const void* ws) {
  if (!p) return fail(DUNET_E_INVALID, "plan is NULL");
  if (!p->committed) return fail(DUNET_E_STATE, "plan not committed (dunet_plan_commit)");
  if (B < 1 || B > p->cfg.batch_max) return fail(DUNET_E_INVALID, "batch %d outside [1, %d]", B, p->cfg.batch_max);
  if (!ws || (reinterpret_cast<uintptr_t>(ws) & 255u)) return fail(DUNET_E_INVALID, "workspace must be non-NULL and 256-byte aligned");
  return 0;
}

static int launch_pack(const dunet_plan* p, const float* src0, int c0, const float* src1, int c1, Act dst, int c_pad,
                       long long vox, int B, cudaStream_t st, bool triple = false) {
  DUNET_FMT(fmt_h(p, dst.lo != nullptr || triple), launch_k(pack_c8_kernel<HF>, dim3(grid_for((long long)B * (c_pad / 8) * vox, 256)), dim3(256), 0, st,
                                 src0, c0, src1, c1, dst.hi, dst.lo, c_pad, vox, B, triple ? 1 : 0));
  LAUNCH_CHECK();
  return 0;
}

static int encode_impl(dunet_plan* p, const float* image, int B, uint8_t* ws, const WsLayout& L, cudaStream_t st) {
  const bool ep = enc_prec(p), triple = p->enc[0].a.triple;
  const Act in_pack = ws_act_x(p, ws, L.in_pack, p->in_pad, 0, B, ep && !triple);
  TRY(launch_pack(p, image, p->cfg.in_channels, nullptr, 0, in_pack, p->in_pad, p->V[0], B, st, triple));
  for (int l = 0; l < 5; ++l) {
    const Act src = l ? ws_act_x(p, ws, L.epool[l], p->fp[l - 1], l, B, ep) : in_pack;
    const Act pooled = l < 4 ? ws_act_x(p, ws, L.epool[l + 1], p->fp[l], l + 1, B, ep) : Act();
    // feature maps: hi + lo pairs in fp32x3 mode; ONE fp16 tensor in fp16 mode (rounded once from the split-precision result)
    TRY(run_twoconv(p, p->enc[l], src, Act(), BiasRef(), Act(), ws_act(p, ws, L.emb[l], p->fp[l], l, B), pooled, l, B, ws, L, st));
  }
  return 0;
}

// U-Net body given in_pack = cat([image, x_t]); leaves the RAW output of upcat_1.conv_1 in ws.raw
static int unet_body(dunet_plan* p, BiasRef temb_row, int B, uint8_t* ws, const WsLayout& L, cudaStream_t st,
                     int* last_nseg, Act* last_raw) {
  const Act in_pack = ws_act(p, ws, L.in_pack, p->in_pad, 0, B);
  for (int l = 0; l < 5; ++l) {
    const Act src = l ? ws_act(p, ws, L.dpool[l], p->fp[l - 1], l, B) : in_pack;
    const Act pooled = l < 4 ? ws_act(p, ws, L.dpool[l + 1], p->fp[l], l + 1, B) : Act();
    TRY(run_twoconv(p, p->den[l], src, Act(), temb_row.at(p->temb_off[l]), ws_act(p, ws, L.emb[l], p->fp[l], l, B),
                    ws_act(p, ws, L.x[l], p->fp[l], l, B), pooled, l, B, ws, L, st));
  }
  Act prev = ws_act(p, ws, L.x[4], p->fp[4], 4, B);
  for (int l = 4; l >= 1; --l) {
    const Act up = ws_act(p, ws, L.up[l], p->upp[l], l - 1, B);
    TRY(run_deconv(p, p->dec[l], prev, up, l, B, st));
    const Act u = ws_act(p, ws, L.u[l], p->uoutp[l], l - 1, B);
    TRY(run_twoconv(p, p->upc[l], ws_act(p, ws, L.x[l - 1], p->fp[l - 1], l - 1, B), up, temb_row.at(p->temb_off[5 + (4 - l)]),
                    Act(), u, Act(), l - 1, B, ws, L, st, /*defer_last_norm=*/l == 1, last_nseg, l == 1 ? last_raw : nullptr));
    prev = u;
  }
  return 0;
}

static int launch_temb(dunet_plan* p, const int* d_t, int rows, float* table, cudaStream_t st) {
  TembArgs a;
  a.w0 = p->dense[0]; a.b0 = p->dense[1]; a.w1 = p->dense[2]; a.b1 = p->dense[3];
  const TwoConvW* blocks[9] = {&p->den[0], &p->den[1], &p->den[2], &p->den[3], &p->den[4],
                               &p->upc[4], &p->upc[3], &p->upc[2], &p->upc[1]};
  for (int i = 0; i < 9; ++i) {
    a.pw[i] = blocks[i]->tp_w; a.pb[i] = blocks[i]->tp_b; a.pc[i] = blocks[i]->a.coutr; a.poff[i] = p->temb_off[i];
  }
  a.row = p->temb_row; a.tmap = d_t; a.table = table;
  temb_table_kernel<<<rows, 512, 0, st>>>(a);
  LAUNCH_CHECK();
  return 0;
}

// fills the part of FinalDdimArgs that folds upcat_1.conv_1's InstanceNorm + LeakyReLU into the final 1x1 conv
static void final_args_common(dunet_plan* p, FinalDdimArgs& a, uint8_t* ws, const WsLayout& L, int nseg, int B, Act feat) {
  (void)ws; (void)L;
  memset(&a, 0, sizeof a);
  a.feat = feat.hi; a.feat_lo = feat.lo; a.F = p->fp[5]; a.w = p->final_w; a.b = p->final_b; a.C = p->C;
  a.partial = reinterpret_cast<float*>(ws + L.partial); a.nseg = nseg; a.gamma = p->upc[1].b.gamma; a.beta = p->upc[1].b.beta;
  a.eps = 1e-5f; a.slope = 0.1f; a.in_pad = p->in_pad; a.vox = p->V[0]; a.batch = B; a.in_ch = p->cfg.in_channels;
}

static int launch_final(dunet_plan* p, const FinalDdimArgs& a, cudaStream_t st) {
  // 3 blocks per SM in total (2 to 32 measured slower)
  const dim3 grid(grid_for((a.vox + 15) / 16 * 32, FINAL_THREADS, std::max(1, 148 * 3 / a.batch)), a.batch);
  if (a.F != 64 && a.F != 128) return fail(DUNET_E_UNSUPPORTED, "final conv: padded features[5] must be 64 or 128");
  const bool prec = a.feat_lo != nullptr;
#define DUNET_FINAL_MC(NT, MC)                                                                     \
  do {                                                                                             \
    if (prec) {                                                                                    \
      if (a.F == 64) launch_k(final_ddim_kernel<NT, 4, MODE_FP32X3, MC>, grid, dim3(FINAL_THREADS), 0, st, a); \
      else launch_k(final_ddim_kernel<NT, 8, MODE_FP32X3, MC>, grid, dim3(FINAL_THREADS), 0, st, a);           \
    } else if (is_fp16(p)) {                                                                       \
      if (a.F == 64) launch_k(final_ddim_kernel<NT, 4, MODE_FP16, MC>, grid, dim3(FINAL_THREADS), 0, st, a);   \
      else launch_k(final_ddim_kernel<NT, 8, MODE_FP16, MC>, grid, dim3(FINAL_THREADS), 0, st, a);             \
    } else {                                                                                       \
      if (a.F == 64) launch_k(final_ddim_kernel<NT, 4, MODE_BF16, MC>, grid, dim3(FINAL_THREADS), 0, st, a);   \
      else launch_k(final_ddim_kernel<NT, 8, MODE_BF16, MC>, grid, dim3(FINAL_THREADS), 0, st, a);             \
    }                                                                                              \
  } while (0)
#define DUNET_FINAL(NT)                         \
  do {                                          \
    if (a.in_ch > 1) DUNET_FINAL_MC(NT, true);  \
    else DUNET_FINAL_MC(NT, false);             \
  } while (0)
  if (PROF_ON)  // feature map read once (bf16) + fp32 state x_t and sum(x0) read+written + bf16 re-pack of the next input
    prof_of(p)->bytes[PROF_FINAL] += (double)a.batch * (double)a.vox * ((prec ? 4.0 : 2.0) * a.F + (a.x_t ? 16.0 * a.C : 0.0) + (a.logits_out ? 4.0 * a.C : 0.0) + (a.next_in ? 2.0 * a.C : 0.0));
  TRY(prof_begin(PROF_FINAL, st));
  if (a.C <= 8) DUNET_FINAL(1);
  else if (a.C <= 16) DUNET_FINAL(2);
  else DUNET_FINAL(4);
#undef DUNET_FINAL
#undef DUNET_FINAL_MC
  LAUNCH_CHECK();
  TRY(prof_end(st));
  return 0;
}

// ------------------------------------------------------------------------------------------------ HD95
// HD95 workspace: per-class state, then per voxel an int16 D-offset, an int16 envelope stack, an (int16, int16)
// (D, H)-offset, and room for d_AB ++ d_BA (at most two fp64 per voxel).  Reused by every class.
struct Hd95Layout {
  size_t meta, off1, stack, off2, keys, total;
};
static Hd95Layout hd95_layout(const int32_t dims[3]) {
  const size_t V = (size_t)dims[0] * dims[1] * dims[2];
  Hd95Layout L;
  size_t o = 0;
  auto take = [&](size_t bytes) { const size_t at = o; o += (bytes + 255) / 256 * 256; return at; };
  L.meta = take(sizeof(Hd95Meta));
  L.off1 = take(V * sizeof(int16_t));
  L.stack = take(V * sizeof(int16_t));
  L.off2 = take(V * sizeof(int32_t));
  L.keys = take(2 * V * sizeof(unsigned long long));
  L.total = o;
  return L;
}
static int hd95_check_dims(int32_t channels, const int32_t dims[3]) {
  if (!dims || channels < 1) return fail(DUNET_E_INVALID, "bad argument");
  for (int d = 0; d < 3; ++d) {
    if (dims[d] < 1) return fail(DUNET_E_INVALID, "dims[%d] = %d must be >= 1", d, dims[d]);
    if (dims[d] > HD_MAX_DIM) return fail(DUNET_E_UNSUPPORTED, "dims[%d] = %d exceeds %d", d, dims[d], HD_MAX_DIM);
  }
  return 0;
}

template <typename LabelT>
static int hd95_class(const uint8_t* pred, const LabelT* label, const HdGeom& g, char* ws, const Hd95Layout& L, double* out,
                      cudaStream_t st) {
  Hd95Meta* m = reinterpret_cast<Hd95Meta*>(ws + L.meta);
  int16_t* off1 = reinterpret_cast<int16_t*>(ws + L.off1);
  int16_t* stack = reinterpret_cast<int16_t*>(ws + L.stack);
  int32_t* off2 = reinterpret_cast<int32_t*>(ws + L.off2);
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(ws + L.keys);
  const long long V = (long long)g.D * g.H * g.W;
  auto lines = [](long long n) { return (unsigned)((n + HD_LINE_THREADS - 1) / HD_LINE_THREADS); };
  hd95_init_kernel<<<1, 256, 0, st>>>(m);
  LAUNCH_CHECK();
  hd95_box_kernel<LabelT><<<grid_for(V, 256, 148 * 8), 256, 0, st>>>(pred, label, g, m);
  LAUNCH_CHECK();
  // d_AB: queries border(pred), sites border(label); then d_BA
  hd95_pass_d_kernel<LabelT><<<lines((long long)g.H * g.W), HD_LINE_THREADS, 0, st>>>(label, g, m, off1);
  LAUNCH_CHECK();
  hd95_pass_h_kernel<<<lines((long long)g.D * g.W), HD_LINE_THREADS, 0, st>>>(g, m, off1, stack, off2);
  LAUNCH_CHECK();
  hd95_pass_w_kernel<uint8_t><<<lines((long long)g.D * g.H), HD_LINE_THREADS, 0, st>>>(pred, g, m, off2, stack, keys);
  LAUNCH_CHECK();
  hd95_pass_d_kernel<uint8_t><<<lines((long long)g.H * g.W), HD_LINE_THREADS, 0, st>>>(pred, g, m, off1);
  LAUNCH_CHECK();
  hd95_pass_h_kernel<<<lines((long long)g.D * g.W), HD_LINE_THREADS, 0, st>>>(g, m, off1, stack, off2);
  LAUNCH_CHECK();
  hd95_pass_w_kernel<LabelT><<<lines((long long)g.D * g.H), HD_LINE_THREADS, 0, st>>>(label, g, m, off2, stack, keys);
  LAUNCH_CHECK();
  const int sel_grid = grid_for(2 * V, 256, 148 * 8);
  for (int pass = 0; pass < HD_RADIX_PASSES; ++pass) {
    hd95_select_kernel<<<sel_grid, 256, 0, st>>>(m, keys, 56 - 8 * pass);
    LAUNCH_CHECK();
  }
  hd95_finish_kernel<<<sel_grid, 256, 0, st>>>(m, keys, out);
  LAUNCH_CHECK();
  return 0;
}

// ================================================================================================== C ABI
extern "C" {

int dunet_version(void) { return DUNET_VERSION; }
const char* dunet_last_error(void) { return g_err.c_str(); }
uint64_t dunet_launch_count(void) { return g_launches.load(); }

int dunet_profile_enable(dunet_plan* p, int32_t on) {
  if (!p) return fail(DUNET_E_INVALID, "plan is NULL");
  Prof* pr = prof_of(p);
  pr->used = 0;
  pr->flops = 0.0;
  for (double& b : pr->bytes) b = 0.0;
  pr->on = on != 0;
  return 0;
}

int dunet_profile_read(dunet_plan* p, double* conv_ms, uint64_t* conv_launches, double* conv_flops) {
  if (!p || !conv_ms || !conv_launches || !conv_flops) return fail(DUNET_E_INVALID, "NULL argument");
  Prof* pr = prof_of(p);
  double total = 0.0;
  uint64_t n = 0;
  for (size_t i = 0; i < pr->used; ++i) {
    if (pr->recs[i].tag != PROF_CONV) continue;
    CUDA_TRY(cudaEventSynchronize(pr->recs[i].b));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, pr->recs[i].a, pr->recs[i].b));
    total += ms;
    ++n;
  }
  *conv_ms = total; *conv_launches = n; *conv_flops = pr->flops;
  return 0;
}

int dunet_profile_read_all(dunet_plan* p, double* ms_by_tag, uint64_t* launches_by_tag, double* bytes_by_tag) {
  if (!p || !ms_by_tag || !launches_by_tag) return fail(DUNET_E_INVALID, "NULL argument");
  Prof* pr = prof_of(p);
  for (int i = 0; i < PROF_TAGS; ++i) { ms_by_tag[i] = 0.0; launches_by_tag[i] = 0; if (bytes_by_tag) bytes_by_tag[i] = pr->bytes[i]; }
  for (size_t i = 0; i < pr->used; ++i) {
    CUDA_TRY(cudaEventSynchronize(pr->recs[i].b));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, pr->recs[i].a, pr->recs[i].b));
    ms_by_tag[pr->recs[i].tag] += ms;
    launches_by_tag[pr->recs[i].tag] += 1;
  }
  return 0;
}

int dunet_profile_dump(dunet_plan* p, double* ms, int32_t* tags, int32_t capacity, int32_t* count) {
  if (!p || !ms || !tags || !count) return fail(DUNET_E_INVALID, "NULL argument");
  Prof* pr = prof_of(p);
  int n = 0;
  for (size_t i = 0; i < pr->used && n < capacity; ++i, ++n) {
    CUDA_TRY(cudaEventSynchronize(pr->recs[i].b));
    float t = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&t, pr->recs[i].a, pr->recs[i].b));
    ms[n] = t; tags[n] = pr->recs[i].tag;
  }
  *count = n;
  return 0;
}

int dunet_debug_barrier_timeouts(uint32_t* out_flag) {
  if (!out_flag) return fail(DUNET_E_INVALID, "out_flag is NULL");
  CUDA_TRY(cudaMemcpyFromSymbol(out_flag, g_barrier_timeout_flag, sizeof(uint32_t)));
  return 0;
}

int dunet_plan_create(dunet_plan** out, const dunet_cfg* cfg) {
  if (!out || !cfg) return fail(DUNET_E_INVALID, "NULL argument");
  int ndev = 0;
  CUDA_TRY(cudaGetDeviceCount(&ndev));
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) return fail(DUNET_E_UNSUPPORTED, "libdunet_b200 needs an sm_100a device (found sm_%d%d); there is no fallback path", prop.major, prop.minor);
  // the encoder's first conv packs [A.hi | A.lo | A.hi] of the image into ONE 32-channel block: 3 * in_channels <= 32
  if (cfg->in_channels < 1 || cfg->in_channels > DUNET_MAX_IN_CHANNELS)
    return fail(DUNET_E_UNSUPPORTED, "in_channels = %d outside [1, %d]", cfg->in_channels, DUNET_MAX_IN_CHANNELS);
  // the denoiser input [x_0 .. x_{C-1}, image ..] is packed into in_pad = 32 channels
  if (cfg->num_classes < 1 || cfg->num_classes > FINAL_MAX_C)
    return fail(DUNET_E_UNSUPPORTED, "num_classes must be in [1, 31]");
  if (cfg->num_classes + cfg->in_channels > 32)
    return fail(DUNET_E_UNSUPPORTED, "num_classes + in_channels = %d exceeds 32", cfg->num_classes + cfg->in_channels);
  for (int d = 0; d < 3; ++d)
    if (cfg->patch[d] < 32 || cfg->patch[d] % 16) return fail(DUNET_E_INVALID, "patch edge %d must be a multiple of 16 and >= 32", cfg->patch[d]);
  for (int i = 0; i < 6; ++i)
    if (cfg->features[i] < 1 || cfg->features[i] > 2048) return fail(DUNET_E_INVALID, "features[%d] = %d out of range", i, cfg->features[i]);
  if (cfg->features[4] % 2 || cfg->features[3] % 2 || cfg->features[2] % 2)
    return fail(DUNET_E_INVALID, "features[2..4] must be even (UpCat halves the channels)");
  if (cfg->batch_max < 1 || cfg->num_steps < 1 || cfg->num_steps > 1000) return fail(DUNET_E_INVALID, "bad batch_max / num_steps");
  if (pad_to(cfg->features[5], 64) > FINAL_MAX_F) return fail(DUNET_E_UNSUPPORTED, "features[5] > %d not implemented", FINAL_MAX_F);

  if ((cfg->flags & DUNET_FLAG_FP32X3) && (cfg->flags & DUNET_FLAG_REF_CONV))
    return fail(DUNET_E_UNSUPPORTED, "DUNET_FLAG_REF_CONV and DUNET_FLAG_FP32X3 are mutually exclusive");
  if ((cfg->flags & DUNET_FLAG_FP32X3) && (cfg->flags & DUNET_FLAG_FP16))
    return fail(DUNET_E_UNSUPPORTED, "DUNET_FLAG_FP16 and DUNET_FLAG_FP32X3 are mutually exclusive (the hi/lo split is bf16)");
  int sms = 0;
  TRY(dev_prepare(&sms));  // per-device kernel attributes (shared-memory opt-in), once per device
  dunet_plan* p = new dunet_plan();
  p->cfg = *cfg;
  p->num_sms = sms;
  const int parts = (cfg->flags & DUNET_FLAG_FP32X3) ? 3 : 1;
  const int parts_enc = enc_prec(p) ? 3 : 1;
  const int cb64 = (cfg->flags & DUNET_FLAG_TC64_CB64) ? 64 : 32;
  p->C = cfg->num_classes;
  for (int l = 0; l < 5; ++l) {
    p->D[l] = cfg->patch[0] >> l; p->H[l] = cfg->patch[1] >> l; p->W[l] = cfg->patch[2] >> l;
    p->V[l] = (long long)p->D[l] * p->H[l] * p->W[l];
  }
  for (int i = 0; i < 6; ++i) { p->fr[i] = cfg->features[i]; p->fp[i] = pad_to(cfg->features[i], 64); }
  // UpCat(in=f[l], cat=f[l-1], out, halves): denoiser.py:276-280
  for (int l = 4; l >= 1; --l) {
    p->upr[l] = (l == 1) ? p->fr[1] : p->fr[l] / 2;
    p->upp[l] = pad_to(p->upr[l], 64);
    p->uoutr[l] = (l == 1) ? p->fr[5] : p->fr[l - 1];
    p->uoutp[l] = pad_to(p->uoutr[l], 64);
  }
  // encoder (no temb), pretrained/basic_unet.py:491-494
  for (int l = 0; l < 5; ++l) {
    TwoConvW& e = p->enc[l];
    if (l == 0) {
      e.a.shape(cfg->in_channels, p->in_pad, 0, 0, p->fr[0], parts_enc, cb64);
      if (e.a.split && 3 * cfg->in_channels <= 32 && !(cfg->flags & DUNET_FLAG_REF_CONV)) {  // hi, lo, hi of the image in ONE block
        e.a.shape(cfg->in_channels, p->in_pad, 0, 0, p->fr[0], 1, cb64);
        e.a.split = true; e.a.triple = true;
      }
    } else e.a.shape(p->fr[l - 1], p->fp[l - 1], 0, 0, p->fr[l], parts_enc, cb64);
    e.b.shape(p->fr[l], p->fp[l], 0, 0, p->fr[l], parts_enc, cb64);
    TwoConvW& d = p->den[l];
    d.has_temb = true;
    if (l == 0) { d.a.shape(cfg->in_channels + p->C, p->in_pad, 0, 0, p->fr[0], parts, cb64); d.a.rot = cfg->in_channels; }
    else d.a.shape(p->fr[l - 1], p->fp[l - 1], 0, 0, p->fr[l], parts, cb64);
    d.b.shape(p->fr[l], p->fp[l], 0, 0, p->fr[l], parts, cb64);
  }
  for (int l = 4; l >= 1; --l) {
    TwoConvW& u = p->upc[l];
    u.has_temb = true;
    u.a.shape(p->fr[l - 1], p->fp[l - 1], p->upr[l], p->upp[l], p->uoutr[l], parts, cb64);  // cat([skip, up]) denoiser.py:190
    u.b.shape(p->uoutr[l], p->uoutp[l], 0, 0, p->uoutr[l], parts, cb64);
    DeconvW& d = p->dec[l];
    d.cinr = p->fr[l]; d.cinp = p->fp[l]; d.coutr = p->upr[l]; d.coutp = p->upp[l]; d.parts = parts;
  }
  // checkpoint keys (SURVEY Appendix F)
  add_twoconv_slots(p, "embed_model.conv_0", &p->enc[0]);
  for (int l = 1; l < 5; ++l) add_twoconv_slots(p, "embed_model.down." + std::to_string(l - 1) + ".convs", &p->enc[l]);
  add_slot(p, "model.temb.dense.0.weight", K_DENSE, p, {512, 128}, 0);
  add_slot(p, "model.temb.dense.0.bias", K_DENSE, p, {512}, 1);
  add_slot(p, "model.temb.dense.1.weight", K_DENSE, p, {512, 512}, 2);
  add_slot(p, "model.temb.dense.1.bias", K_DENSE, p, {512}, 3);
  add_twoconv_slots(p, "model.conv_0", &p->den[0]);
  for (int l = 1; l < 5; ++l) add_twoconv_slots(p, "model.down_" + std::to_string(l) + ".convs", &p->den[l]);
  for (int l = 4; l >= 1; --l) {
    const std::string pre = "model.upcat_" + std::to_string(l);
    add_slot(p, pre + ".upsample.deconv.weight", K_DECONV_W, &p->dec[l], {p->dec[l].cinr, p->dec[l].coutr, 2, 2, 2});
    add_slot(p, pre + ".upsample.deconv.bias", K_DECONV_B, &p->dec[l], {p->dec[l].coutr});
    add_twoconv_slots(p, pre + ".convs", &p->upc[l]);
  }
  add_slot(p, "model.final_conv.weight", K_FINAL_W, p, {p->C, p->fr[5], 1, 1, 1});
  add_slot(p, "model.final_conv.bias", K_FINAL_B, p, {p->C});
  // temb bias table geometry: 9 TwoConv blocks in forward order
  {
    const TwoConvW* blocks[9] = {&p->den[0], &p->den[1], &p->den[2], &p->den[3], &p->den[4],
                                 &p->upc[4], &p->upc[3], &p->upc[2], &p->upc[1]};
    int off = 0;
    for (int i = 0; i < 9; ++i) { p->temb_off[i] = off; off += blocks[i]->a.coutp; }
    p->temb_row = off;
  }
  *out = p;
  return 0;
}

void dunet_plan_destroy(dunet_plan* p) {
  if (!p) return;
  // sub-batch work may still be running on the internal streams: it reads the plan's weights and tables
  for (cudaStream_t s : p->half_stream)
    if (s) cudaStreamSynchronize(s);
  for (void* q : p->owned) cudaFree(q);
  if (p->h_t) cudaFreeHost(p->h_t);
  for (cudaEvent_t e : p->t_ev) if (e) cudaEventDestroy(e);
  for (ProfRec& r : p->prof.recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  for (int i = 0; i < 2; ++i) {
    if (p->half_stream[i]) cudaStreamDestroy(p->half_stream[i]);
    if (p->ev_join[i]) cudaEventDestroy(p->ev_join[i]);
  }
  if (p->ev_fork) cudaEventDestroy(p->ev_fork);
  delete p;
}

int dunet_plan_set_weight(dunet_plan* p, const char* key, const float* src, const int64_t* shape, int32_t ndim, void* stream) {
  if (!p || !key || !src || !shape) return fail(DUNET_E_INVALID, "NULL argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  auto it = p->slots.find(key);
  if (it == p->slots.end()) return fail(DUNET_E_INVALID, "unexpected checkpoint key '%s'", key);
  Slot& s = it->second;
  if ((int)s.shape.size() != ndim) return fail(DUNET_E_INVALID, "key '%s': expected %zu dims, got %d", key, s.shape.size(), ndim);
  for (int i = 0; i < ndim; ++i)
    if (s.shape[i] != shape[i]) return fail(DUNET_E_INVALID, "key '%s': dim %d is %lld, expected %lld", key, i, (long long)shape[i], (long long)s.shape[i]);
  if (!aligned16(src)) return fail(DUNET_E_INVALID, "key '%s': pointer not 16-byte aligned", key);
  p->committed = false;
  switch (s.kind) {
    case K_CONV_W: {
      ConvW* c = static_cast<ConvW*>(s.obj);
      if (!c->packed) TRY(dev_alloc(p, (void**)&c->packed, c->packed_elems() * sizeof(bf16)));
      const int cinr = c->c0r + c->c1r;
      pack_conv_w_kernel<<<grid_for((long long)c->packed_elems(), 256), 256, 0, st>>>(
          src, c->packed, c->coutr, cinr, c->c0r, c->c0p, c->c1r, c->cb_ch, c->n_tile, c->ncb(), c->n_tiles, c->rot, c->parts, fmt_h(p, c->split) ? 1 : 0, c->triple ? 1 : 0);
      LAUNCH_CHECK();
      if (c->coutp == 64) {
        const size_t n64 = c->packed64_elems();
        if (!c->packed64) TRY(dev_alloc(p, (void**)&c->packed64, n64 * sizeof(bf16)));
        pack_conv_w64_kernel<<<grid_for((long long)n64, 256), 256, 0, st>>>(src, c->packed64, c->coutr, cinr, c->c0r, c->c0p,
                                                                             c->c1r, c->cb64, c->ncb64(), c->rot, c->parts, fmt_h(p, c->split) ? 1 : 0, c->triple ? 1 : 0);
        LAUNCH_CHECK();
      }
      if (p->cfg.flags & DUNET_FLAG_KEEP_FP32_WEIGHTS) {
        const size_t bytes = (size_t)c->coutr * cinr * 27 * sizeof(float);
        if (!c->w32) TRY(dev_alloc(p, (void**)&c->w32, bytes));
        CUDA_TRY(cudaMemcpyAsync(c->w32, src, bytes, cudaMemcpyDeviceToDevice, st));
      }
      c->have_w = true;
      break;
    }
    case K_CONV_B:  // a per-channel constant before InstanceNorm is removed by the mean subtraction (SURVEY App. F)
      static_cast<ConvW*>(s.obj)->have_cb = true;
      break;
    case K_IN_G:
    case K_IN_B: {
      ConvW* c = static_cast<ConvW*>(s.obj);
      float** dst = s.kind == K_IN_G ? &c->gamma : &c->beta;
      if (!*dst) TRY(dev_alloc(p, (void**)dst, c->coutp * sizeof(float)));
      copy_pad_rows_kernel<<<1, 256, 0, st>>>(src, *dst, 1, c->coutr, 1, c->coutp);  // padded channels: gamma = beta = 0
      LAUNCH_CHECK();
      (s.kind == K_IN_G ? c->have_g : c->have_b) = true;
      break;
    }
    case K_TP_W:
    case K_TP_B: {
      TwoConvW* t = static_cast<TwoConvW*>(s.obj);
      const size_t n = s.kind == K_TP_W ? (size_t)t->a.coutr * 512 : (size_t)t->a.coutr;
      float** dst = s.kind == K_TP_W ? &t->tp_w : &t->tp_b;
      if (!*dst) TRY(dev_alloc(p, (void**)dst, n * sizeof(float)));
      CUDA_TRY(cudaMemcpyAsync(*dst, src, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
      (s.kind == K_TP_W ? t->have_tpw : t->have_tpb) = true;
      break;
    }
    case K_DENSE: {
      size_t n = 1;
      for (auto d : s.shape) n *= (size_t)d;
      if (!p->dense[s.idx]) TRY(dev_alloc(p, (void**)&p->dense[s.idx], n * sizeof(float)));
      CUDA_TRY(cudaMemcpyAsync(p->dense[s.idx], src, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
      break;
    }
    case K_DECONV_W: {
      DeconvW* d = static_cast<DeconvW*>(s.obj);
      const size_t n = 8ull * d->cinp * d->coutp;
      if (!d->packed) TRY(dev_alloc(p, (void**)&d->packed, n * sizeof(bf16)));
      pack_deconv_w_kernel<<<grid_for((long long)n, 256), 256, 0, st>>>(src, d->packed, d->cinr, d->coutr, d->cinp, d->coutp, is_fp16(p) ? 1 : 0);
      LAUNCH_CHECK();
      if (!d->packed_tc) TRY(dev_alloc(p, (void**)&d->packed_tc, n * d->parts * sizeof(bf16)));
      pack_deconv_tc_w_kernel<<<grid_for((long long)n * d->parts, 256), 256, 0, st>>>(src, d->packed_tc, d->cinr, d->coutr, d->cinp,
                                                                                      d->coutp, d->parts, is_fp16(p) ? 1 : 0);
      LAUNCH_CHECK();
      d->have_w = true;
      break;
    }
    case K_DECONV_B: {
      DeconvW* d = static_cast<DeconvW*>(s.obj);
      if (!d->bias) TRY(dev_alloc(p, (void**)&d->bias, d->coutp * sizeof(float)));
      copy_pad_rows_kernel<<<1, 256, 0, st>>>(src, d->bias, 1, d->coutr, 1, d->coutp);
      LAUNCH_CHECK();
      d->have_b = true;
      break;
    }
    case K_FINAL_W: {
      if (!p->final_w) TRY(dev_alloc(p, (void**)&p->final_w, (size_t)p->C * p->fp[5] * sizeof(float)));
      copy_pad_rows_kernel<<<grid_for((long long)p->C * p->fp[5], 256), 256, 0, st>>>(src, p->final_w, p->C, p->fr[5], p->C, p->fp[5]);
      LAUNCH_CHECK();
      break;
    }
    case K_FINAL_B: {
      if (!p->final_b) TRY(dev_alloc(p, (void**)&p->final_b, p->C * sizeof(float)));
      CUDA_TRY(cudaMemcpyAsync(p->final_b, src, p->C * sizeof(float), cudaMemcpyDeviceToDevice, st));
      break;
    }
  }
  s.seen = true;
  return 0;
}

int dunet_plan_set_schedule(dunet_plan* p, int32_t n, const int32_t* tmap, const float* sr, const float* srm1, const float* acp) {
  if (!p || !tmap || !sr || !srm1 || !acp) return fail(DUNET_E_INVALID, "NULL argument");
  if (n != p->cfg.num_steps) return fail(DUNET_E_INVALID, "schedule has %d steps, plan was created for %d", n, p->cfg.num_steps);
  p->n_steps = n;
  p->tmap.assign(tmap, tmap + n);
  p->sr.assign(sr, sr + n); p->srm1.assign(srm1, srm1 + n); p->acp.assign(acp, acp + n);
  for (int i = 0; i < n; ++i)
    if (!(srm1[i] > 0.f) || tmap[i] < 0) return fail(DUNET_E_INVALID, "schedule entry %d invalid", i);
  p->committed = false;
  return 0;
}

int dunet_plan_commit(dunet_plan* p, void* stream) {
  if (!p) return fail(DUNET_E_INVALID, "plan is NULL");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  for (auto& kv : p->slots)
    if (!kv.second.seen) return fail(DUNET_E_STATE, "checkpoint key '%s' was never set (%zu keys expected)", kv.first.c_str(), p->slots.size());
  if (p->n_steps == 0) return fail(DUNET_E_STATE, "schedule not set (dunet_plan_set_schedule)");
  if (!p->d_tmap) TRY(dev_alloc(p, (void**)&p->d_tmap, (p->n_steps + 1) * sizeof(int)));
  if (!p->temb_table) TRY(dev_alloc(p, (void**)&p->temb_table, (size_t)(p->n_steps + 1) * p->temb_row * sizeof(float)));
  CUDA_TRY(cudaMemsetAsync(p->temb_table, 0, (size_t)(p->n_steps + 1) * p->temb_row * sizeof(float), st));
  CUDA_TRY(cudaMemcpyAsync(p->d_tmap, p->tmap.data(), p->n_steps * sizeof(int), cudaMemcpyHostToDevice, st));
  TRY(launch_temb(p, p->d_tmap, p->n_steps, p->temb_table, st));
  // everything the per-step entry points need later is created here: "no hidden allocation after commit"
  if (!p->d_t) {
    TRY(dev_alloc(p, (void**)&p->d_t, (size_t)p->cfg.batch_max * sizeof(int)));
    TRY(dev_alloc(p, (void**)&p->temb_scratch, (size_t)p->cfg.batch_max * p->temb_row * sizeof(float)));
    CUDA_TRY(cudaMallocHost((void**)&p->h_t, (size_t)dunet_plan::T_RING * p->cfg.batch_max * sizeof(int)));
    for (int i = 0; i < dunet_plan::T_RING; ++i) CUDA_TRY(cudaEventCreateWithFlags(&p->t_ev[i], cudaEventDisableTiming));
  }
  if (!p->half_stream[0]) {
    for (int i = 0; i < 2; ++i) {
      CUDA_TRY(cudaStreamCreateWithFlags(&p->half_stream[i], cudaStreamNonBlocking));
      CUDA_TRY(cudaEventCreateWithFlags(&p->ev_join[i], cudaEventDisableTiming));
    }
    CUDA_TRY(cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming));
  }
  CUDA_TRY(cudaStreamSynchronize(st));  // host vector above must outlive the copy; commit is a setup-time call
  p->committed = true;
  return 0;
}

int dunet_workspace_bytes(const dunet_plan* p, int32_t batch, size_t* out) {
  if (!p || !out) return fail(DUNET_E_INVALID, "NULL argument");
  if (batch < 1 || batch > p->cfg.batch_max) return fail(DUNET_E_INVALID, "batch %d outside [1, %d]", batch, p->cfg.batch_max);
  const SubBatches s = sub_batches(p, batch, dual_batch(p, batch));
  *out = std::max(ws_layout(p, batch).total, s.n * s.ws_stride);
  return 0;
}

int dunet_encode(dunet_plan* p, const float* image, int32_t B, void* workspace, void* stream) {
  TRY(check_call(p, B, workspace));
  if (!image || !aligned16(image)) return fail(DUNET_E_INVALID, "image must be a 16-byte aligned device pointer");
  p->emb_B = B; p->emb_dual = false;
  return encode_impl(p, image, B, static_cast<uint8_t*>(workspace), ws_layout(p, B), static_cast<cudaStream_t>(stream));
}

int dunet_get_embedding(dunet_plan* p, int32_t level, float* out, int32_t B, void* workspace, void* stream) {
  TRY(check_call(p, B, workspace));
  if (level < 0 || level > 4 || !out) return fail(DUNET_E_INVALID, "bad level / NULL out");
  const WsLayout L = ws_layout(p, B);
  const Act e = ws_act(p, static_cast<uint8_t*>(workspace), L.emb[level], p->fp[level], level, B);
  DUNET_FMT(fmt_h(p, e.lo != nullptr), unpack_c8_kernel<HF><<<grid_for((long long)B * (p->fp[level] / 8) * p->V[level], 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      e.hi, e.lo, p->fp[level], out, p->fr[level], p->V[level], B));
  LAUNCH_CHECK();
  return 0;
}

int dunet_set_embedding(dunet_plan* p, int32_t level, const float* in, int32_t B, void* workspace, void* stream) {
  TRY(check_call(p, B, workspace));
  if (level < 0 || level > 4 || !in) return fail(DUNET_E_INVALID, "bad level / NULL in");
  p->emb_B = B; p->emb_dual = false;
  const WsLayout L = ws_layout(p, B);
  return launch_pack(p, in, p->fr[level], nullptr, 0, ws_act(p, static_cast<uint8_t*>(workspace), L.emb[level], p->fp[level], level, B),
                     p->fp[level], p->V[level], B, static_cast<cudaStream_t>(stream));
}

int dunet_denoise_step(dunet_plan* p, const float* x_t, const float* image, const int32_t* t_original, float* logits_out,
                       int32_t B, void* workspace, void* stream) {
  TRY(check_call(p, B, workspace));
  if (!x_t || !image || !logits_out || !t_original) return fail(DUNET_E_INVALID, "NULL tensor argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  const WsLayout L = ws_layout(p, B);
  // one timestep shared by the batch and present in the respaced schedule (the inference call): its precomputed row
  int row = -1;
  bool shared = true;
  for (int n = 0; n < B; ++n) {
    if (t_original[n] < 0) return fail(DUNET_E_INVALID, "timestep %d of sample %d is negative", (int)t_original[n], n);
    shared = shared && t_original[n] == t_original[0];
  }
  if (shared)
    for (int i = 0; i < p->n_steps; ++i)
      if (p->tmap[i] == t_original[0]) row = i;
  BiasRef temb;
  if (row >= 0) {
    temb.p = p->temb_table + (size_t)row * p->temb_row;
  } else {
    // training-style call (models/diffusion/diffusion.py:71-84: `step` is a per-sample tensor of arbitrary timesteps):
    // build one bias row per sample.  The timesteps travel through a pinned ring slot owned by the plan.
    const int slot = p->t_slot;
    p->t_slot = (slot + 1) % dunet_plan::T_RING;
    CUDA_TRY(cudaEventSynchronize(p->t_ev[slot]));  // the copy that last used this slot has been consumed
    int* h = p->h_t + (size_t)slot * p->cfg.batch_max;
    for (int n = 0; n < B; ++n) h[n] = t_original[n];
    CUDA_TRY(cudaMemcpyAsync(p->d_t, h, (size_t)B * sizeof(int), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaEventRecord(p->t_ev[slot], st));
    TRY(launch_temb(p, p->d_t, B, p->temb_scratch, st));
    temb.p = p->temb_scratch;
    temb.n_stride = p->temb_row;
  }
  TRY(launch_pack(p, x_t, p->C, image, p->cfg.in_channels, ws_act(p, ws, L.in_pack, p->in_pad, 0, B), p->in_pad, p->V[0], B, st));
  int nseg = 0;
  Act feat;
  TRY(unet_body(p, temb, B, ws, L, st, &nseg, &feat));
  FinalDdimArgs a;
  final_args_common(p, a, ws, L, nseg, B, feat);
  a.image = image; a.logits_out = logits_out;
  a.r = 1.f; a.m = 1.f; a.abp = 1.f;
  return launch_final(p, a, st);
}

// where the initial x_T of a batch comes from: the caller's tensor, or the library's counter-based generator
struct NoiseSrc {
  const float* given = nullptr;      // [B][C][vox] fp32 or nullptr
  unsigned long long seed = 0;
  const int64_t* ids = nullptr;      // host [B]: noise stream id per window (generator only)
  int draw = 0;                      // ensemble draw index, folded into the stream id
};

// One batch (or half batch) of windows on one stream, workspace laid out for exactly B windows: encoder (optional), noise
// initialisation, the N DDIM steps.  Leaves sum_k clamp(x0_k) in ws.acc and the last sample in ws.x_t, both voxel-major.
// per_step_stride = elements between consecutive steps in per_step_logits (the FULL batch size when halves are used).
static int ddim_core(dunet_plan* p, const float* image, const NoiseSrc& nz, int id0, float* per_step_logits, size_t per_step_stride,
                     int B, int run_encoder, int zero_acc, uint8_t* ws, cudaStream_t st) {
  const WsLayout L = ws_layout(p, B);
  const int CP = p->C <= 8 ? 8 : (p->C <= 16 ? 16 : 32);
  float* x_t = reinterpret_cast<float*>(ws + L.x_t);   // voxel-major [B][vox][CP]
  float* acc = reinterpret_cast<float*>(ws + L.acc);
  if (run_encoder) TRY(encode_impl(p, image, B, ws, L, st));
  const Act in_pack = ws_act(p, ws, L.in_pack, p->in_pad, 0, B);
  for (int b0 = 0; b0 < B; b0 += INIT_MAX_B) {  // x_t = noise, acc = 0, first conv input = [noise, image] in one pass
    const int nb = std::min(INIT_MAX_B, B - b0);
    DdimInitArgs ia;
    memset(&ia, 0, sizeof ia);
    ia.noise = nz.given ? nz.given + (size_t)b0 * p->C * p->V[0] : nullptr;
    ia.image = image + (size_t)b0 * p->cfg.in_channels * p->V[0];
    ia.x_t = x_t + (size_t)b0 * p->V[0] * CP; ia.acc = acc + (size_t)b0 * p->V[0] * CP;
    ia.next_in = in_pack.hi + (size_t)b0 * p->in_pad * p->V[0];
    ia.next_in_lo = in_pack.lo ? in_pack.lo + (size_t)b0 * p->in_pad * p->V[0] : nullptr;
    ia.C = p->C; ia.CP = CP; ia.in_pad = p->in_pad; ia.batch = nb; ia.zero_acc = zero_acc; ia.vox = p->V[0]; ia.seed = nz.seed;
    ia.in_ch = p->cfg.in_channels;
    for (int j = 0; j < nb; ++j) ia.ids[j] = nz.ids ? (long long)(((unsigned long long)nz.ids[id0 + b0 + j] & 0xFFFFFFFFFFull) | ((unsigned long long)nz.draw << 40)) : 0;
    const int nch = std::max(CP, p->in_pad) / 8;
    if (PROF_ON) prof_of(p)->bytes[PROF_GLUE] += (double)nb * p->V[0] * (CP * 8.0 + p->in_pad * 2.0 + 4.0 * p->cfg.in_channels + (nz.given ? 4.0 * p->C : 0.0));
    TRY(prof_begin(PROF_GLUE, st));
    DUNET_FMT(fmt_h(p, in_pack.lo != nullptr), launch_k(ddim_init_kernel<HF>, dim3(grid_for((long long)nb * p->V[0] * nch, 256, 148 * 8)), dim3(256), 0, st, ia));
    LAUNCH_CHECK();
    TRY(prof_end(st));
  }
  for (int i = p->n_steps - 1, k = 0; i >= 0; --i, ++k) {  // gaussian_diffusion.py:694 indices high -> low
    int nseg = 0;
    Act feat;
    BiasRef temb;
    temb.p = p->temb_table + (size_t)i * p->temb_row;
    TRY(unet_body(p, temb, B, ws, L, st, &nseg, &feat));
    FinalDdimArgs a;
    final_args_common(p, a, ws, L, nseg, B, feat);
    a.image = image; a.x_t = x_t; a.acc = acc;
    a.logits_out = per_step_logits ? per_step_logits + (size_t)k * per_step_stride : nullptr;
    a.next_in = i > 0 ? in_pack.hi : nullptr;
    a.next_in_lo = i > 0 ? in_pack.lo : nullptr;
    a.r = p->sr[i]; a.m = p->srm1[i]; a.abp = p->acp[i];
    TRY(launch_final(p, a, st));
  }
  return 0;
}

// ddim_core + conversion of the voxel-major results to the reference's planar fp32 tensors
static int ddim_sample_impl(dunet_plan* p, const float* image, const float* noise, float* acc_out, float* per_step_logits,
                            size_t per_step_stride, float* final_x, int B, int run_encoder, float out_scale, int out_accumulate,
                            uint8_t* ws, cudaStream_t st) {
  NoiseSrc nz;
  nz.given = noise;
  TRY(ddim_core(p, image, nz, 0, per_step_logits, per_step_stride, B, run_encoder, 1, ws, st));
  const WsLayout L = ws_layout(p, B);
  const int CP = p->C <= 8 ? 8 : (p->C <= 16 ? 16 : 32);
  const int sgrid = grid_for((long long)B * p->V[0] * (CP / 4), 256, 148 * 8);
  TRY(prof_begin(PROF_GLUE, st));
  launch_k(state_from_vm_kernel, dim3(sgrid), dim3(256), 0, st, (const float*)(ws + L.acc), acc_out, p->C, CP, (long long)p->V[0], B, out_scale,
           out_accumulate);
  LAUNCH_CHECK();
  TRY(prof_end(st));
  if (final_x) {
    launch_k(state_from_vm_kernel, dim3(sgrid), dim3(256), 0, st, (const float*)(ws + L.x_t), final_x, p->C, CP, (long long)p->V[0], B, 1.f, 0);
    LAUNCH_CHECK();
  }
  return 0;
}

int dunet_ddim_sample(dunet_plan* p, const float* image, const float* noise, float* acc_out, float* per_step_logits,
                      float* final_x, int32_t B, int32_t run_encoder, float out_scale, int32_t out_accumulate, void* workspace,
                      void* stream) {
  TRY(check_call(p, B, workspace));
  if (!image || !noise || !acc_out) return fail(DUNET_E_INVALID, "NULL tensor argument");
  if (!aligned16(image) || !aligned16(noise) || !aligned16(acc_out)) return fail(DUNET_E_INVALID, "tensors must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  const size_t per_step_stride = (size_t)B * p->C * p->V[0];
  const SubBatches s = sub_batches(p, B, use_dual(p, B, run_encoder));
  return run_sub_batches(p, s, B, ws, st, [&](int b0, int nb, uint8_t* ws_h, cudaStream_t sh) -> int {
    const size_t img_off = (size_t)b0 * p->cfg.in_channels * p->V[0], st_off = (size_t)b0 * p->C * p->V[0];
    return ddim_sample_impl(p, image + img_off, noise + st_off, acc_out + st_off, per_step_logits ? per_step_logits + st_off : nullptr,
                            per_step_stride, final_x ? final_x + st_off : nullptr, nb, run_encoder, out_scale, out_accumulate, ws_h, sh);
  });
}

static int check_box(const int32_t v[3], const int32_t pd[3], const int32_t s[3]) {
  for (int d = 0; d < 3; ++d)
    if (pd[d] < 1 || v[d] < 1 || s[d] < 0 || s[d] + pd[d] > v[d])
      return fail(DUNET_E_INVALID, "window [%d, %d) outside volume extent %d on axis %d", s[d], s[d] + pd[d], v[d], d);
  return 0;
}

int dunet_crop_window(const float* volume, const int32_t v[3], float* patch, const int32_t pd[3], const int32_t s[3], void* stream) {
  if (!volume || !patch || !v || !pd || !s) return fail(DUNET_E_INVALID, "NULL argument");
  TRY(check_box(v, pd, s));
  crop_window_kernel<<<grid_for((long long)pd[0] * pd[1] * pd[2], 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      volume, patch, v[0], v[1], v[2], pd[0], pd[1], pd[2], s[0], s[1], s[2]);
  LAUNCH_CHECK();
  return 0;
}

// volume [nc][v], patches [B][nc][pd]
static int crop_batch(const dunet_plan* p, const float* volume, const int32_t v[3], int nc, float* patches, const int32_t pd[3],
                      const int32_t* starts, int B, cudaStream_t st) {
  const long long pe = (long long)pd[0] * pd[1] * pd[2] * nc;  // elements per window
  for (int b0 = 0; b0 < B; b0 += INIT_MAX_B) {
    const int nb = std::min(INIT_MAX_B, B - b0);
    CropArgs c;
    memset(&c, 0, sizeof c);
    c.vol = volume; c.patches = patches + (size_t)b0 * pe;
    c.VD = v[0]; c.VH = v[1]; c.VW = v[2]; c.PD = pd[0]; c.PH = pd[1]; c.PW = pd[2]; c.batch = nb; c.nc = nc;
    for (int j = 0; j < nb; ++j) {
      TRY(check_box(v, pd, starts + 3 * (b0 + j)));
      for (int d = 0; d < 3; ++d) c.start[j][d] = starts[3 * (b0 + j) + d];
    }
    if (p) {
      if (PROF_ON) prof_of(p)->bytes[PROF_GLUE] += 8.0 * nb * pe;
      TRY(prof_begin(PROF_GLUE, st));
    }
    launch_k(crop_windows_kernel, dim3(grid_for(pe * nb, 256)), dim3(256), 0, st, c);
    LAUNCH_CHECK();
    if (p) TRY(prof_end(st));
  }
  return 0;
}

int dunet_crop_windows(const float* volume, const int32_t v[3], float* patches, const int32_t pd[3], const int32_t* starts,
                       int32_t B, void* stream) {
  if (!volume || !patches || !v || !pd || !starts || B < 1) return fail(DUNET_E_INVALID, "bad argument");
  return crop_batch(nullptr, volume, v, 1, patches, pd, starts, B, static_cast<cudaStream_t>(stream));
}

int dunet_infer_windows(dunet_plan* p, const float* volume, const int32_t v[3], const int32_t* starts, int32_t B,
                        const float* noise, uint64_t seed, const int64_t* noise_ids, int32_t ensemble, float* out_volume,
                        float* count_volume, const float* weights, void* workspace, void* stream) {
  TRY(check_call(p, B, workspace));
  if (!volume || !v || !starts || !out_volume) return fail(DUNET_E_INVALID, "NULL argument");
  if (!noise && !noise_ids) return fail(DUNET_E_INVALID, "either noise or noise_ids must be given");
  if (ensemble < 1) return fail(DUNET_E_INVALID, "ensemble must be >= 1");
  if ((weights == nullptr) != (count_volume == nullptr)) return fail(DUNET_E_INVALID, "weights and count_volume go together (gaussian blend)");
  if (!aligned16(volume) || !aligned16(out_volume) || (noise && !aligned16(noise))) return fail(DUNET_E_INVALID, "tensors must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  const int32_t pd[3] = {p->D[0], p->H[0], p->W[0]};
  const int CP = p->C <= 8 ? 8 : (p->C <= 16 ? 16 : 32);
  const SubBatches sb = sub_batches(p, B, use_dual(p, B, 1));
  TRY(run_sub_batches(p, sb, B, ws, st, [&](int b0, int nb, uint8_t* ws_h, cudaStream_t sh) -> int {
    float* image = reinterpret_cast<float*>(ws_h + ws_layout(p, nb).image);
    TRY(crop_batch(p, volume, v, p->cfg.in_channels, image, pd, starts + 3 * b0, nb, sh));  // window crop: one launch per sub-batch
    for (int r = 0; r < ensemble; ++r) {  // BASELINE config 4: R independent noise draws, summed; the encoder runs once
      NoiseSrc nz;
      nz.given = noise ? noise + ((size_t)r * B + b0) * p->C * p->V[0] : nullptr;
      nz.seed = seed; nz.ids = noise_ids; nz.draw = r;
      TRY(ddim_core(p, image, nz, b0, nullptr, 0, nb, r == 0, r == 0, ws_h, sh));
    }
    return 0;
  }));
  // MONAI's window order on the caller's stream (fp32 sums in the oracle's order): window b is row b % B0 of the
  // accumulator of sub-batch b / B0
  const float scale = 1.f / (float)ensemble;
  for (int b = 0; b < B; ++b) {
    const int h = b / sb.B0, nb = std::min(sb.B0, B - h * sb.B0);
    const float* acc = reinterpret_cast<const float*>(ws + h * sb.ws_stride + ws_layout(p, nb).acc) + (size_t)(b % sb.B0) * p->V[0] * CP;
    const int32_t* s = starts + 3 * b;
    if (PROF_ON) prof_of(p)->bytes[PROF_GLUE] += (double)p->V[0] * (4.0 * CP + 8.0 * p->C);
    TRY(prof_begin(PROF_GLUE, st));
    launch_k(stitch_from_vm_kernel, dim3(grid_for(p->V[0], 256, 148 * 8)), dim3(256), 0, st, out_volume, count_volume, acc, weights, p->C, CP,
             v[0], v[1], v[2], pd[0], pd[1], pd[2], s[0], s[1], s[2], scale);
    LAUNCH_CHECK();
    TRY(prof_end(st));
  }
  return 0;
}

int dunet_zero(void* ptr, size_t bytes, void* stream) {
  if (!ptr) return fail(DUNET_E_INVALID, "NULL argument");
  CUDA_TRY(cudaMemsetAsync(ptr, 0, bytes, static_cast<cudaStream_t>(stream)));
  return 0;
}

int dunet_stitch_add(float* out_volume, const int32_t v[3], int32_t channels, const float* patch, const int32_t pd[3],
                     const int32_t s[3], void* stream) {
  if (!out_volume || !patch || !v || !pd || !s || channels < 1) return fail(DUNET_E_INVALID, "bad argument");
  TRY(check_box(v, pd, s));
  stitch_add_kernel<<<grid_for((long long)channels * pd[0] * pd[1] * pd[2], 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      out_volume, patch, channels, v[0], v[1], v[2], pd[0], pd[1], pd[2], s[0], s[1], s[2]);
  LAUNCH_CHECK();
  return 0;
}

int dunet_finalize(float* out_volume, const int32_t v[3], int32_t channels, const int32_t* cd, const int32_t* ch,
                   const int32_t* cw, uint8_t* binary, uint8_t* argmax_labels, void* stream) {
  if (!out_volume || !v || !cd || !ch || !cw || channels < 1) return fail(DUNET_E_INVALID, "bad argument");
  finalize_kernel<<<grid_for((long long)v[0] * v[1] * v[2], 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      out_volume, cd, ch, cw, binary, argmax_labels, channels, v[0], v[1], v[2]);
  LAUNCH_CHECK();
  return 0;
}

int dunet_stitch_add_weighted(float* out_volume, float* count_volume, const int32_t v[3], int32_t channels, const float* patch,
                              const float* weights, const int32_t pd[3], const int32_t s[3], void* stream) {
  if (!out_volume || !count_volume || !patch || !weights || !v || !pd || !s || channels < 1) return fail(DUNET_E_INVALID, "bad argument");
  TRY(check_box(v, pd, s));
  stitch_add_weighted_kernel<<<grid_for((long long)channels * pd[0] * pd[1] * pd[2], 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      out_volume, count_volume, patch, weights, channels, v[0], v[1], v[2], pd[0], pd[1], pd[2], s[0], s[1], s[2]);
  LAUNCH_CHECK();
  return 0;
}

int dunet_finalize_weighted(float* out_volume, const float* count_volume, const int32_t v[3], int32_t channels, uint8_t* binary,
                            uint8_t* argmax_labels, void* stream) {
  if (!out_volume || !count_volume || !v || channels < 1) return fail(DUNET_E_INVALID, "bad argument");
  const long long vv = (long long)v[0] * v[1] * v[2];
  finalize_weighted_kernel<<<grid_for(vv, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(out_volume, count_volume, binary,
                                                                                            argmax_labels, channels, vv);
  LAUNCH_CHECK();
  return 0;
}

int dunet_scale_intensity(const float* in, float* out, int64_t n, float a_min, float a_max, float b_min, float b_max, int32_t clip,
                          void* stream) {
  if (!in || !out || n < 1) return fail(DUNET_E_INVALID, "bad argument");
  if (!(a_max > a_min)) return fail(DUNET_E_INVALID, "a_max must exceed a_min");
  scale_intensity_kernel<<<grid_for(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(in, out, (long long)n, a_min, a_max, b_min,
                                                                                       b_max, clip);
  LAUNCH_CHECK();
  return 0;
}

int dunet_foreground_bbox(const float* image, int32_t channels, const int32_t dims[3], int32_t* bbox_dev, void* stream) {
  if (!image || !dims || !bbox_dev || channels < 1) return fail(DUNET_E_INVALID, "bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  bbox_init_kernel<<<1, 32, 0, st>>>(bbox_dev, dims[0], dims[1], dims[2]);
  LAUNCH_CHECK();
  foreground_bbox_kernel<<<grid_for((long long)channels * dims[0] * dims[1] * dims[2], 256, 148 * 8), 256, 0, st>>>(
      image, channels, dims[0], dims[1], dims[2], bbox_dev);
  LAUNCH_CHECK();
  return 0;
}

int dunet_crop_box(const float* in, int32_t channels, const int32_t dims[3], float* out, const int32_t out_dims[3],
                   const int32_t start[3], void* stream) {
  if (!in || !out || !dims || !out_dims || !start || channels < 1) return fail(DUNET_E_INVALID, "bad argument");
  TRY(check_box(dims, out_dims, start));
  crop_box_kernel<<<grid_for((long long)channels * out_dims[0] * out_dims[1] * out_dims[2], 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      in, out, channels, dims[0], dims[1], dims[2], out_dims[0], out_dims[1], out_dims[2], start[0], start[1], start[2]);
  LAUNCH_CHECK();
  return 0;
}

int dunet_resample_spacing(const float* in, int32_t channels, const int32_t dims[3], float* out, const int32_t out_dims[3],
                           const double ratio[3], int32_t mode, void* stream) {
  if (!in || !out || !dims || !out_dims || !ratio || channels < 1) return fail(DUNET_E_INVALID, "bad argument");
  if (mode != 0 && mode != 1) return fail(DUNET_E_INVALID, "mode must be 0 (trilinear) or 1 (nearest)");
  for (int d = 0; d < 3; ++d)
    if (dims[d] < 1 || out_dims[d] < 1 || !(ratio[d] > 0.0)) return fail(DUNET_E_INVALID, "bad dims / ratio on axis %d", d);
  resample_spacing_kernel<<<grid_for((long long)channels * out_dims[0] * out_dims[1] * out_dims[2], 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      in, out, channels, dims[0], dims[1], dims[2], out_dims[0], out_dims[1], out_dims[2], ratio[0], ratio[1], ratio[2], mode);
  LAUNCH_CHECK();
  return 0;
}

int dunet_invert_labels(const float* blended, int32_t channels, const int32_t vol_dims[3], const int32_t offset[3],
                        const int32_t res_dims[3], const double ratio[3], const int32_t box_start[3], const int32_t box_dims[3],
                        const int32_t out_dims[3], int32_t mode, uint8_t* binary, uint8_t* argmax, void* stream) {
  if (!blended || !vol_dims || !offset || !res_dims || !ratio || !box_start || !box_dims || !out_dims)
    return fail(DUNET_E_INVALID, "NULL argument");
  if (!binary && !argmax) return fail(DUNET_E_INVALID, "binary and argmax are both NULL: nothing to write");
  if (channels < 1) return fail(DUNET_E_INVALID, "channels = %d must be >= 1", channels);
  if (argmax && channels > 256) return fail(DUNET_E_INVALID, "argmax labels are uint8: channels = %d must be <= 256", channels);
  if (mode != 0 && mode != 1) return fail(DUNET_E_INVALID, "mode must be 0 (nearest) or 1 (trilinear)");
  for (int d = 0; d < 3; ++d)
    if (!(ratio[d] > 0.0) || !std::isfinite(ratio[d])) return fail(DUNET_E_INVALID, "ratio[%d] = %g must be finite and > 0", d, ratio[d]);
  TRY(check_box(vol_dims, res_dims, offset));     // the resampled volume inside the driver volume
  TRY(check_box(out_dims, box_dims, box_start));  // the foreground box inside the output grid
  InvertLabelsArgs a;
  a.blended = blended;
  a.C = channels;
  a.VH = vol_dims[1];
  a.VW = vol_dims[2];
  a.vol_vox = (long long)vol_dims[0] * vol_dims[1] * vol_dims[2];
  for (int d = 0; d < 3; ++d) {
    a.off[d] = offset[d]; a.res[d] = res_dims[d]; a.box_start[d] = box_start[d]; a.box_dims[d] = box_dims[d];
    a.out[d] = out_dims[d]; a.ratio[d] = ratio[d];
  }
  a.nearest = mode == 0;
  a.binary = binary;
  a.argmax = argmax;
  invert_labels_kernel<<<grid_for((long long)out_dims[0] * out_dims[1] * out_dims[2], 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
  LAUNCH_CHECK();
  return 0;
}

int dunet_uncertainty_fuse(const float* per_step, int32_t runs, int32_t n_steps, int64_t n, float* out, void* stream) {
  if (!per_step || !out || runs < 1 || n_steps < 1 || n < 1) return fail(DUNET_E_INVALID, "bad argument");
  uncertainty_fuse_kernel<<<grid_for(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(per_step, out, runs, n_steps, (long long)n);
  LAUNCH_CHECK();
  return 0;
}

// ---- CUDA IPC helpers for the peer-memory exchange (one process per GPU: a rank maps the other ranks' partial-sum
// buffers into its own address space; NVLink peer access is enabled by the open call)
int dunet_ipc_alloc(void** ptr, size_t bytes, uint8_t handle_out[64]) {
  if (!ptr || !handle_out || bytes == 0) return fail(DUNET_E_INVALID, "bad argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  CUDA_TRY(cudaMalloc(ptr, bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, *ptr);
  if (e != cudaSuccess) {
    cudaFree(*ptr);
    *ptr = nullptr;
    return fail(DUNET_E_CUDA, "cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
  }
  memcpy(handle_out, &h, 64);
  return 0;
}
int dunet_ipc_open(const uint8_t handle[64], void** ptr) {
  if (!handle || !ptr) return fail(DUNET_E_INVALID, "NULL argument");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  CUDA_TRY(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return 0;
}
int dunet_ipc_close(void* ptr) {
  if (ptr) CUDA_TRY(cudaIpcCloseMemHandle(ptr));
  return 0;
}
int dunet_ipc_free(void* ptr) {
  if (ptr) CUDA_TRY(cudaFree(ptr));
  return 0;
}

int dunet_finalize_peers(const float* const* partial_ptrs, const int32_t* slab_lo, const int32_t* slab_hi, int32_t n_src,
                         const int32_t v[3], int32_t channel_lo, int32_t channel_hi, const int32_t* cd, const int32_t* ch,
                         const int32_t* cw, uint8_t* binary, float* blended, void* stream) {
  if (!partial_ptrs || !slab_lo || !slab_hi || !v || !cd || !ch || !cw || !binary) return fail(DUNET_E_INVALID, "NULL argument");
  if (n_src < 1 || n_src > PEER_MAX_SRC) return fail(DUNET_E_INVALID, "n_src must be in [1, %d]", PEER_MAX_SRC);
  if (channel_lo < 0 || channel_hi <= channel_lo) return fail(DUNET_E_INVALID, "bad channel range");
  if (v[2] % 4) return fail(DUNET_E_UNSUPPORTED, "dunet_finalize_peers needs a volume width that is a multiple of 4");
  FinalizePeersArgs a;
  memset(&a, 0, sizeof a);
  for (int k = 0; k < n_src; ++k) {
    if (!partial_ptrs[k] || !aligned16(partial_ptrs[k])) return fail(DUNET_E_INVALID, "source %d is NULL or not 16-byte aligned", k);
    a.src[k] = partial_ptrs[k]; a.lo[k] = slab_lo[k]; a.hi[k] = slab_hi[k];
  }
  a.n_src = n_src; a.cd = cd; a.ch = ch; a.cw = cw; a.binary = binary; a.blended = blended;
  a.c_lo = channel_lo; a.c_hi = channel_hi; a.D = v[0]; a.H = v[1]; a.W = v[2];
  const long long total = (long long)v[0] * v[1] * v[2] / 4 * (channel_hi - channel_lo);
  finalize_peers_kernel<<<grid_for(total, 256, 148 * 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
  LAUNCH_CHECK();
  return 0;
}

int dunet_q_sample(const float* x_start, const float* noise_in, float* noise_out, const int64_t* t_dev, const float* sqrt_ac,
                   const float* sqrt_1mac, float* out, int32_t batch, int64_t per_sample, uint64_t seed, int64_t id0, void* stream) {
  if (!x_start || !t_dev || !sqrt_ac || !sqrt_1mac || !out || batch < 1 || per_sample < 1) return fail(DUNET_E_INVALID, "bad argument");
  if (!noise_in && !noise_out) return fail(DUNET_E_INVALID, "generated noise needs noise_out (the reference returns it)");
  q_sample_kernel<<<grid_for((per_sample + 3) / 4 * batch, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      x_start, noise_in, noise_out, reinterpret_cast<const long long*>(t_dev), sqrt_ac, sqrt_1mac, out, (long long)per_sample, batch,
      (unsigned long long)seed, (long long)id0);
  LAUNCH_CHECK();
  return 0;
}

int dunet_dice_counts(const uint8_t* pred, const void* label, int32_t label_is_float, int32_t channels, int64_t voxels,
                      uint64_t* counts, void* stream) {
  if (!pred || !label || !counts || channels < 1 || voxels < 1) return fail(DUNET_E_INVALID, "bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  CUDA_TRY(cudaMemsetAsync(counts, 0, (size_t)channels * 3 * sizeof(uint64_t), st));
  const dim3 grid(grid_for(voxels, 256, 148 * 8 / std::max(1, std::min(channels, 8))), channels);
  if (label_is_float)
    dice_counts_kernel<float><<<grid, 256, 0, st>>>(pred, static_cast<const float*>(label), (long long)voxels,
                                                    reinterpret_cast<unsigned long long*>(counts));
  else
    dice_counts_kernel<uint8_t><<<grid, 256, 0, st>>>(pred, static_cast<const uint8_t*>(label), (long long)voxels,
                                                      reinterpret_cast<unsigned long long*>(counts));
  LAUNCH_CHECK();
  return 0;
}

int dunet_hd95_workspace_bytes(int32_t channels, const int32_t dims[3], size_t* out_bytes) {
  TRY(hd95_check_dims(channels, dims));
  if (!out_bytes) return fail(DUNET_E_INVALID, "out_bytes is NULL");
  *out_bytes = hd95_layout(dims).total;
  return 0;
}

int dunet_hd95(const uint8_t* pred, const void* label, int32_t label_is_float, int32_t channels, const int32_t dims[3],
               const double spacing[3], double* hd95_out, void* workspace, size_t workspace_bytes, void* stream) {
  TRY(hd95_check_dims(channels, dims));
  if (!pred || !label || !spacing || !hd95_out || !workspace) return fail(DUNET_E_INVALID, "NULL argument");
  if ((label_is_float && (reinterpret_cast<uintptr_t>(label) & 3u)) || (reinterpret_cast<uintptr_t>(hd95_out) & 7u))
    return fail(DUNET_E_INVALID, "label (fp32) must be 4-byte and hd95_out 8-byte aligned");
  if (reinterpret_cast<uintptr_t>(workspace) & 255u) return fail(DUNET_E_INVALID, "workspace must be 256-byte aligned");
  for (int d = 0; d < 3; ++d)
    if (!std::isfinite(spacing[d]) || !(spacing[d] > 0.0)) return fail(DUNET_E_INVALID, "spacing[%d] must be finite and > 0", d);
  const Hd95Layout L = hd95_layout(dims);
  if (workspace_bytes < L.total) return fail(DUNET_E_INVALID, "workspace of %zu bytes, %zu needed", workspace_bytes, L.total);
  const HdGeom g{dims[0], dims[1], dims[2], spacing[0], spacing[1], spacing[2]};
  const size_t V = (size_t)dims[0] * dims[1] * dims[2];
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  for (int c = 0; c < channels; ++c) {
    if (label_is_float)
      TRY(hd95_class(pred + c * V, static_cast<const float*>(label) + c * V, g, ws, L, hd95_out + c, st));
    else
      TRY(hd95_class(pred + c * V, static_cast<const uint8_t*>(label) + c * V, g, ws, L, hd95_out + c, st));
  }
  return 0;
}

int dunet_op_conv3x3x3(const float* src0, int32_t c0, const float* src1, int32_t c1, const float* weight, int32_t cout,
                       float* out, int32_t B, const int32_t dims[3], int32_t use_ref, void* stream) {
  if (!src0 || !weight || !out || !dims || c0 < 1 || cout < 1 || B < 1) return fail(DUNET_E_INVALID, "bad argument");
  if (c1 > 0 && !src1) return fail(DUNET_E_INVALID, "src1 is NULL but c1 > 0");
  if (use_ref < 0 || use_ref > 6) return fail(DUNET_E_INVALID, "use_ref_kernel must be 0..6");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool prec = use_ref == 3 || use_ref == 4, fp16 = use_ref >= 5;
  const bool generic_only = use_ref == 2 || use_ref == 4 || use_ref == 6;
  dunet_plan tmp;  // only geometry fields are used by run_conv
  memset(&tmp.cfg, 0, sizeof tmp.cfg);
  TRY(dev_prepare(&tmp.num_sms));
  tmp.cfg.flags = use_ref == 1 ? (DUNET_FLAG_REF_CONV | DUNET_FLAG_KEEP_FP32_WEIGHTS) : (prec ? DUNET_FLAG_FP32X3 : (fp16 ? DUNET_FLAG_FP16 : 0));
  if (generic_only) tmp.cfg.flags |= DUNET_FLAG_GENERIC_CONV;  // voxel-as-M generic kernel only (no Cout = 64 / flattened-plane kernels)
  tmp.D[0] = dims[0]; tmp.H[0] = dims[1]; tmp.W[0] = dims[2];
  tmp.V[0] = (long long)dims[0] * dims[1] * dims[2];
  ConvW c;
  const bool small = (c1 == 0 && c0 <= 32);
  c.shape(c0, small ? 32 : pad_to(c0, 64), c1, c1 > 0 ? pad_to(c1, 64) : 0, cout, prec ? 3 : 1);
  if (c1 > 0 && (c0 % 8)) return fail(DUNET_E_UNSUPPORTED, "concat needs c0 %% 8 == 0");
  const long long vox = tmp.V[0];
  const size_t pm = prec ? 2 : 1;
  Act a0, a1, raw;
  CUDA_TRY(cudaMallocAsync((void**)&a0.hi, pm * B * c.c0p * vox * sizeof(bf16), st));
  CUDA_TRY(cudaMallocAsync((void**)&raw.hi, pm * B * c.coutp * vox * sizeof(bf16), st));
  if (prec) { a0.lo = a0.hi + (size_t)B * c.c0p * vox; raw.lo = raw.hi + (size_t)B * c.coutp * vox; }
  TRY(launch_pack(&tmp, src0, c0, nullptr, 0, a0, c.c0p, vox, B, st));
  if (c1 > 0) {
    CUDA_TRY(cudaMallocAsync((void**)&a1.hi, pm * B * c.c1p * vox * sizeof(bf16), st));
    if (prec) a1.lo = a1.hi + (size_t)B * c.c1p * vox;
    TRY(launch_pack(&tmp, src1, c1, nullptr, 0, a1, c.c1p, vox, B, st));
  }
  int rc = 0;
  if (use_ref == 1) {
    c.w32 = const_cast<float*>(weight);
  } else {
    CUDA_TRY(cudaMallocAsync((void**)&c.packed, c.packed_elems() * sizeof(bf16), st));
    pack_conv_w_kernel<<<grid_for((long long)c.packed_elems(), 256), 256, 0, st>>>(
        weight, c.packed, c.coutr, c0 + c1, c.c0r, c.c0p, c.c1r, c.cb_ch, c.n_tile, c.ncb(), c.n_tiles, 0, c.parts, fp16 ? 1 : 0, 0);
    LAUNCH_CHECK();
    if (c.coutp == 64 && !generic_only) {
      const size_t n64 = c.packed64_elems();
      CUDA_TRY(cudaMallocAsync((void**)&c.packed64, n64 * sizeof(bf16), st));
      pack_conv_w64_kernel<<<grid_for((long long)n64, 256), 256, 0, st>>>(weight, c.packed64, c.coutr, c0 + c1, c.c0r, c.c0p,
                                                                           c.c1r, c.cb64, c.ncb64(), 0, c.parts, fp16 ? 1 : 0, 0);
      LAUNCH_CHECK();
    }
  }
  int nseg_unused = 0;
  rc = run_conv(&tmp, c, conv_plan(&tmp, c, 0, /*may_split=*/false), a0, a1, raw, nullptr, nullptr, &nseg_unused, 0, B, st);
  if (rc == 0) {
    DUNET_FMT(fp16, unpack_c8_kernel<HF><<<grid_for((long long)B * (c.coutp / 8) * vox, 256), 256, 0, st>>>(raw.hi, raw.lo, c.coutp, out, cout, vox, B));
    g_launches.fetch_add(1);
    if (cudaGetLastError() != cudaSuccess) rc = fail(DUNET_E_CUDA, "unpack launch failed");
  }
  cudaFreeAsync(a0.hi, st);
  cudaFreeAsync(raw.hi, st);
  if (a1.hi) cudaFreeAsync(a1.hi, st);
  if (c.packed) cudaFreeAsync(c.packed, st);
  if (c.packed64) cudaFreeAsync(c.packed64, st);
  return rc;
}

int dunet_op_deconv2x2x2(const float* src, int32_t cin, const float* weight, const float* bias, int32_t cout, float* out,
                         int32_t B, const int32_t dims[3], int32_t use_ref, void* stream) {
  if (!src || !weight || !bias || !out || !dims || cin < 1 || cout < 1 || B < 1) return fail(DUNET_E_INVALID, "bad argument");
  if (use_ref < 0 || use_ref > 6) return fail(DUNET_E_INVALID, "use_ref_kernel must be 0..6");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool prec = use_ref == 3 || use_ref == 4, fp16 = use_ref >= 5;
  dunet_plan tmp;
  memset(&tmp.cfg, 0, sizeof tmp.cfg);
  TRY(dev_prepare(&tmp.num_sms));
  tmp.cfg.flags = use_ref == 1 ? DUNET_FLAG_REF_CONV : ((use_ref == 2 || use_ref == 4 || use_ref == 6) ? DUNET_FLAG_GENERIC_CONV : 0);
  if (prec) tmp.cfg.flags |= DUNET_FLAG_FP32X3;
  if (fp16) tmp.cfg.flags |= DUNET_FLAG_FP16;
  tmp.D[0] = dims[0]; tmp.H[0] = dims[1]; tmp.W[0] = dims[2];
  tmp.V[0] = (long long)dims[0] * dims[1] * dims[2];
  DeconvW d;
  d.cinr = cin; d.cinp = pad_to(cin, 64); d.coutr = cout; d.coutp = pad_to(cout, 64); d.parts = prec ? 3 : 1;
  const long long vox = tmp.V[0];
  const size_t nw = 8ull * d.cinp * d.coutp;
  const size_t pm = prec ? 2 : 1;
  Act a0, o;
  CUDA_TRY(cudaMallocAsync((void**)&a0.hi, pm * B * d.cinp * vox * sizeof(bf16), st));
  CUDA_TRY(cudaMallocAsync((void**)&o.hi, pm * B * d.coutp * vox * 8 * sizeof(bf16), st));
  if (prec) { a0.lo = a0.hi + (size_t)B * d.cinp * vox; o.lo = o.hi + (size_t)B * d.coutp * vox * 8; }
  CUDA_TRY(cudaMallocAsync((void**)&d.packed, nw * sizeof(bf16), st));
  CUDA_TRY(cudaMallocAsync((void**)&d.packed_tc, nw * d.parts * sizeof(bf16), st));
  CUDA_TRY(cudaMallocAsync((void**)&d.bias, d.coutp * sizeof(float), st));
  TRY(launch_pack(&tmp, src, cin, nullptr, 0, a0, d.cinp, vox, B, st));
  pack_deconv_w_kernel<<<grid_for((long long)nw, 256), 256, 0, st>>>(weight, d.packed, cin, cout, d.cinp, d.coutp, fp16 ? 1 : 0);
  LAUNCH_CHECK();
  pack_deconv_tc_w_kernel<<<grid_for((long long)nw * d.parts, 256), 256, 0, st>>>(weight, d.packed_tc, cin, cout, d.cinp, d.coutp, d.parts, fp16 ? 1 : 0);
  LAUNCH_CHECK();
  copy_pad_rows_kernel<<<1, 256, 0, st>>>(bias, d.bias, 1, cout, 1, d.coutp);
  LAUNCH_CHECK();
  int rc = run_deconv(&tmp, d, a0, o, 0, B, st);
  if (rc == 0) {
    DUNET_FMT(fp16, unpack_c8_kernel<HF><<<grid_for((long long)B * (d.coutp / 8) * vox * 8, 256), 256, 0, st>>>(o.hi, o.lo, d.coutp, out, cout, vox * 8, B));
    g_launches.fetch_add(1);
    if (cudaGetLastError() != cudaSuccess) rc = fail(DUNET_E_CUDA, "unpack launch failed");
  }
  cudaFreeAsync(a0.hi, st); cudaFreeAsync(o.hi, st); cudaFreeAsync(d.packed, st); cudaFreeAsync(d.packed_tc, st); cudaFreeAsync(d.bias, st);
  return rc;
}

int dunet_debug_conv_geometry(const int32_t dims[3], int32_t cin, int32_t cout, uint32_t flags, int32_t out[16]) {
  if (!dims || !out || cin < 1 || cout < 1 || dims[0] < 1 || dims[1] < 1 || dims[2] < 1) return fail(DUNET_E_INVALID, "bad argument");
  dunet_plan tmp;  // geometry fields only; no CUDA call is made
  memset(&tmp.cfg, 0, sizeof tmp.cfg);
  tmp.cfg.flags = flags;
  tmp.D[0] = dims[0]; tmp.H[0] = dims[1]; tmp.W[0] = dims[2];
  tmp.V[0] = (long long)dims[0] * dims[1] * dims[2];
  ConvW c;
  c.shape(cin, cin <= 32 ? 32 : pad_to(cin, 64), 0, 0, cout, (flags & DUNET_FLAG_FP32X3) ? 3 : 1);
  const ConvPlan g = conv_plan(&tmp, c, 0, /*may_split=*/true);  // as a layer of a plan runs it
  out[0] = g.kernel == CONV_TC64 ? 0 : (g.kernel == CONV_FLAT ? 2 : 1);  // the reference kernel reports 1
  out[1] = g.zt; out[2] = g.tiles_x; out[3] = g.tiles_y; out[4] = g.tiles_z; out[5] = g.ksplit; out[6] = g.ksub;
  out[7] = g.flat.hx; out[8] = g.flat.ty; out[9] = g.flat.npos; out[10] = g.flat.a_slots; out[11] = g.flat.w_slots; out[12] = g.flat.smem;
  out[13] = g.tiles * c.n_tiles; out[14] = c.n_tiles; out[15] = c.ncb();
  return 0;
}

int dunet_debug_set_conv_timeline(int64_t* dev_buffer) {
  g_conv_dbg = reinterpret_cast<long long*>(dev_buffer);
  g_conv_dbg_count = 0;
  return 0;
}

}  // extern "C"
