// HD95 surface distance per class (medpy hd95 with connectivity 1, the metric Diff-UNet results are reported with
// beside Dice).  One class at a time, for A = prediction and B = label:
//
//   border(M)  = M minus its 6-connected erosion, with the outside of the volume counted as background;
//   d_AB       = for every border voxel of A, the distance to the nearest border voxel of B (spacing-weighted);
//   HD95       = numpy.percentile(d_AB ++ d_BA, 95), linear interpolation.
//
// Every site and every query lies in the bounding box of A ∪ B, so the distance transform restricted to that box is
// exact.  hd95_box_kernel finds the box and the two border counts; the three separable passes then run over the box
// only, with grids sized for the whole volume whose surplus threads exit at once (the box lives in device memory: no
// host synchronisation).  Pass D (axis 0) finds the nearest site on each D-line; passes H and W take the lower envelope
// of parabolas (Felzenszwalb & Huttenlocher) and carry the integer offset to the nearest site, so pass W, which runs
// only at the query voxels, forms each distance exactly as scipy's distance_transform_edt does:
// sqrt(((s0 d0)^2 + (s1 d1)^2) + (s2 d2)^2) in fp64.  The two order statistics of the percentile come from a radix
// select on the fp64 bit patterns (non-negative doubles order as uint64).
#pragma once
#include <climits>
#include <cooperative_groups.h>
#include <cstdint>
#include <cuda_runtime.h>

namespace dunet {

constexpr int16_t HD_NONE = INT16_MIN;  // no site on the line; offsets need |d| <= 32766, hence dims <= 32767
constexpr int HD_MAX_DIM = 32767;
constexpr int HD_LINE_THREADS = 128;
constexpr int HD_RADIX_PASSES = 8;      // 8-bit digits of a 64-bit key

struct HdGeom {
  int D, H, W;
  double s0, s1, s2;  // spacing per array axis
};

// Per-class state, re-initialised by hd95_init_kernel before every class.
struct Hd95Meta {
  int lo[3], hi[3];               // bounding box of A ∪ B, inclusive
  unsigned long long n[2];        // |border(A)|, |border(B)|: the lengths of d_AB and d_BA
  unsigned long long fill;        // distances appended so far
  unsigned long long prefix;      // radix select: the digits of x[lo] found so far (all of them after the last pass)
  unsigned long long rank;        // rank of x[lo] among the keys that share `prefix`
  unsigned long long eq;          // after the last pass: how many keys equal x[lo]
  unsigned long long above;       // smallest key greater than x[lo]
  unsigned int done;              // blocks finished in the current select / finish launch
  unsigned long long hist[256];   // digit histogram of the current select pass
};

template <typename T>
__device__ __forceinline__ bool hd_fg(const T* __restrict__ m, long long v) { return m[v] != T(0); }

template <typename T>
__device__ __forceinline__ bool hd_border(const T* __restrict__ m, int z, int y, int x, const HdGeom& g) {
  const long long W = g.W, HW = (long long)g.H * g.W, v = z * HW + y * W + x;
  if (!hd_fg(m, v)) return false;
  if (z == 0 || z == g.D - 1 || y == 0 || y == g.H - 1 || x == 0 || x == g.W - 1) return true;
  return !hd_fg(m, v - HW) || !hd_fg(m, v + HW) || !hd_fg(m, v - W) || !hd_fg(m, v + W) || !hd_fg(m, v - 1) ||
         !hd_fg(m, v + 1);
}

__device__ __forceinline__ bool hd_empty(const Hd95Meta* m) { return m->n[0] == 0 || m->n[1] == 0; }

// numpy.percentile(x, 95) on n sorted values, default 'linear' method: virtual index h = (n - 1) * 0.95.
__device__ __forceinline__ void hd_percentile_index(unsigned long long n, unsigned long long& lo, unsigned long long& hi,
                                                    double& gamma) {
  const double h = __dmul_rn((double)(n - 1), 0.95), f = floor(h);
  lo = (unsigned long long)f;
  hi = lo + 1 < n ? lo + 1 : n - 1;
  gamma = __dsub_rn(h, f);
}

__global__ void hd95_init_kernel(Hd95Meta* m) {
  const int t = threadIdx.x;  // 256 threads
  m->hist[t] = 0;
  if (t < 3) { m->lo[t] = INT_MAX; m->hi[t] = -1; }
  if (t == 0) {
    m->n[0] = m->n[1] = 0;
    m->fill = m->prefix = m->rank = m->eq = 0;
    m->above = ~0ull;
    m->done = 0;
  }
}

// Bounding box of A ∪ B and the border counts of A and B.  Grid-stride over the whole volume.
template <typename LabelT>
__global__ void __launch_bounds__(256) hd95_box_kernel(const uint8_t* __restrict__ pred, const LabelT* __restrict__ label,
                                                       HdGeom g, Hd95Meta* m) {
  const long long V = (long long)g.D * g.H * g.W;
  int lo0 = INT_MAX, lo1 = INT_MAX, lo2 = INT_MAX, hi0 = -1, hi1 = -1, hi2 = -1;
  unsigned int na = 0, nb = 0;
  for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v < V; v += (long long)gridDim.x * blockDim.x) {
    const bool a = pred[v] != 0, b = label[v] != LabelT(0);
    if (!a && !b) continue;
    const int x = (int)(v % g.W), y = (int)(v / g.W % g.H), z = (int)(v / ((long long)g.W * g.H));
    lo0 = min(lo0, z); lo1 = min(lo1, y); lo2 = min(lo2, x);
    hi0 = max(hi0, z); hi1 = max(hi1, y); hi2 = max(hi2, x);
    na += (a && hd_border(pred, z, y, x, g)) ? 1u : 0u;
    nb += (b && hd_border(label, z, y, x, g)) ? 1u : 0u;
  }
  lo0 = __reduce_min_sync(0xffffffffu, lo0); lo1 = __reduce_min_sync(0xffffffffu, lo1); lo2 = __reduce_min_sync(0xffffffffu, lo2);
  hi0 = __reduce_max_sync(0xffffffffu, hi0); hi1 = __reduce_max_sync(0xffffffffu, hi1); hi2 = __reduce_max_sync(0xffffffffu, hi2);
  na = __reduce_add_sync(0xffffffffu, na);
  nb = __reduce_add_sync(0xffffffffu, nb);
  if ((threadIdx.x & 31) == 0) {
    if (hi0 >= 0) {
      atomicMin(&m->lo[0], lo0); atomicMin(&m->lo[1], lo1); atomicMin(&m->lo[2], lo2);
      atomicMax(&m->hi[0], hi0); atomicMax(&m->hi[1], hi1); atomicMax(&m->hi[2], hi2);
    }
    if (na) atomicAdd(&m->n[0], (unsigned long long)na);
    if (nb) atomicAdd(&m->n[1], (unsigned long long)nb);
  }
}

// Pass D: one thread per D-line (y, x) of the box.  off[v] = z' - z for the nearest site z' on the line, HD_NONE if
// the line has none (ties: the lower z').
template <typename SiteT>
__global__ void __launch_bounds__(HD_LINE_THREADS) hd95_pass_d_kernel(const SiteT* __restrict__ site, HdGeom g,
                                                                      const Hd95Meta* __restrict__ m, int16_t* __restrict__ off) {
  if (hd_empty(m)) return;
  const int bw = m->hi[2] - m->lo[2] + 1;
  const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (t >= (long long)(m->hi[1] - m->lo[1] + 1) * bw) return;
  const int y = m->lo[1] + (int)(t / bw), x = m->lo[2] + (int)(t % bw);
  const long long HW = (long long)g.H * g.W, base = (long long)y * g.W + x;
  int last = -1;
  for (int z = m->lo[0]; z <= m->hi[0]; ++z) {
    if (hd_border(site, z, y, x, g)) last = z;
    off[z * HW + base] = last < 0 ? HD_NONE : (int16_t)(last - z);
  }
  int next = -1;
  for (int z = m->hi[0]; z >= m->lo[0]; --z) {
    const long long v = z * HW + base;
    const int16_t o = off[v];
    if (o == 0) { next = z; continue; }
    if (next >= 0 && (o == HD_NONE || next - z < -o)) off[v] = (int16_t)(next - z);
  }
}

// Lower envelope of the parabolas f_q(p) = (s (p - q))^2 + F(q) over the sites q in [lo, hi] of one line
// (Felzenszwalb & Huttenlocher).  cost(q, F) returns false where q is no site.  The stack holds site positions at
// stack[k * stride]; F of a stacked site is read again through `cost`.  The test "the intersection of (b, q) is not
// right of the intersection of (a, b)" is cross-multiplied rather than divided, so it is exact whenever the squared
// terms are.  Returns the top index, -1 when the line has no site.
template <typename Cost>
__device__ __forceinline__ int hd_envelope(int lo, int hi, double s, const Cost& cost, int16_t* stack, long long stride) {
  const double w = s * s;
  int top = -1;
  for (int q = lo; q <= hi; ++q) {
    double Fq;
    if (!cost(q, Fq)) continue;
    while (top >= 1) {
      const int b = stack[top * stride], a = stack[(top - 1) * stride];
      double Fa, Fb;
      cost(a, Fa);
      cost(b, Fb);
      const double nbq = (Fq - Fb) + w * ((double)(q - b) * (double)(q + b));
      const double nab = (Fb - Fa) + w * ((double)(b - a) * (double)(b + a));
      if (nbq * (double)(b - a) <= nab * (double)(q - b)) --top;
      else break;
    }
    stack[++top * stride] = (int16_t)q;
  }
  return top;
}

// The envelope segment that holds position p: segments are ordered along the line, so k only moves forward.
template <typename Cost>
__device__ __forceinline__ int hd_envelope_at(int p, int k, int top, double s, const Cost& cost, const int16_t* stack,
                                              long long stride) {
  while (k < top) {
    const int a = stack[k * stride], b = stack[(k + 1) * stride];
    double Fa, Fb;
    cost(a, Fa);
    cost(b, Fb);
    const double ta = s * (double)(p - a), tb = s * (double)(p - b);
    if (tb * tb + Fb <= ta * ta + Fa) ++k;
    else break;
  }
  return k;
}

__device__ __forceinline__ int32_t hd_pack(int dz, int dy) { return (int32_t)((uint32_t)(uint16_t)dz | ((uint32_t)(uint16_t)dy << 16)); }
__device__ __forceinline__ int hd_dz(int32_t o) { return (int16_t)(o & 0xffff); }
__device__ __forceinline__ int hd_dy(int32_t o) { return (int16_t)(o >> 16); }

// Pass H: one thread per H-line (z, x) of the box.  off2[v] = (dz, dy) of the nearest site in the (z, x) plane slice
// that passes D and H have seen, dz = HD_NONE if there is none.
__global__ void __launch_bounds__(HD_LINE_THREADS) hd95_pass_h_kernel(HdGeom g, const Hd95Meta* __restrict__ m,
                                                                      const int16_t* __restrict__ off1, int16_t* __restrict__ stack,
                                                                      int32_t* __restrict__ off2) {
  if (hd_empty(m)) return;
  const int bw = m->hi[2] - m->lo[2] + 1, lo = m->lo[1], hi = m->hi[1];
  const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (t >= (long long)(m->hi[0] - m->lo[0] + 1) * bw) return;
  const int z = m->lo[0] + (int)(t / bw), x = m->lo[2] + (int)(t % bw);
  const long long W = g.W, row0 = (long long)z * g.H * g.W + x;
  const double s0 = g.s0;
  auto cost = [&](int y, double& F) {
    const int16_t o = off1[row0 + y * W];
    if (o == HD_NONE) return false;
    const double d = s0 * (double)o;
    F = d * d;
    return true;
  };
  int16_t* stk = stack + row0 + lo * W;
  const int top = hd_envelope(lo, hi, g.s1, cost, stk, W);
  int k = 0;
  for (int y = lo; y <= hi; ++y) {
    if (top < 0) { off2[row0 + y * W] = hd_pack(HD_NONE, 0); continue; }
    k = hd_envelope_at(y, k, top, g.s1, cost, stk, W);
    const int q = stk[k * W];
    off2[row0 + y * W] = hd_pack(off1[row0 + q * W], q - y);
  }
}

// Pass W: one thread per W-line (z, y) of the box; evaluated only at the query voxels, border(query).  Appends
// sqrt(((s0 dz)^2 + (s1 dy)^2) + (s2 dx)^2), rounded as scipy rounds it (no FMA), to keys[] as its fp64 bit pattern.
template <typename QueryT>
__global__ void __launch_bounds__(HD_LINE_THREADS) hd95_pass_w_kernel(const QueryT* __restrict__ query, HdGeom g, Hd95Meta* m,
                                                                      const int32_t* __restrict__ off2, int16_t* __restrict__ stack,
                                                                      unsigned long long* __restrict__ keys) {
  if (hd_empty(m)) return;
  const int bh = m->hi[1] - m->lo[1] + 1, lo = m->lo[2], hi = m->hi[2];
  const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (t >= (long long)(m->hi[0] - m->lo[0] + 1) * bh) return;
  const int z = m->lo[0] + (int)(t / bh), y = m->lo[1] + (int)(t % bh);
  const long long row0 = ((long long)z * g.H + y) * g.W;
  const double s0 = g.s0, s1 = g.s1;
  auto cost = [&](int x, double& F) {
    const int32_t o = off2[row0 + x];
    if (hd_dz(o) == HD_NONE) return false;
    const double a = s0 * (double)hd_dz(o), b = s1 * (double)hd_dy(o);
    F = __dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b));
    return true;
  };
  int16_t* stk = stack + row0 + lo;
  const int top = hd_envelope(lo, hi, g.s2, cost, stk, 1);
  if (top < 0) return;  // only when B has no border voxel, which hd_empty has excluded
  int k = 0;
  for (int x = lo; x <= hi; ++x) {
    if (!hd_border(query, z, y, x, g)) continue;
    k = hd_envelope_at(x, k, top, g.s2, cost, stk, 1);
    const int q = stk[k];
    const int32_t o = off2[row0 + q];
    const double a = __dmul_rn(s0, (double)hd_dz(o)), b = __dmul_rn(s1, (double)hd_dy(o)), c = __dmul_rn(g.s2, (double)(q - x));
    const double d = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b)), __dmul_rn(c, c)));
    cooperative_groups::coalesced_group grp = cooperative_groups::coalesced_threads();
    unsigned long long base = 0;
    if (grp.thread_rank() == 0) base = atomicAdd(&m->fill, (unsigned long long)grp.size());
    base = grp.shfl(base, 0);
    keys[base + grp.thread_rank()] = (unsigned long long)__double_as_longlong(d);
  }
}

// Last block of a grid-stride launch: true in every thread of the block that finishes last (its predecessors' global
// writes are visible to it).
__device__ __forceinline__ bool hd_last_block(unsigned int* done) {
  __shared__ bool last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(done, 1u) == gridDim.x - 1;
  __syncthreads();
  if (last) __threadfence();
  return last;
}

// One radix-select pass over the 8-bit digit at `shift` (56, 48, ..., 0) for the key of rank lo: histogram of the
// keys that match the digits found so far, then the last block picks the digit.  256 threads.
__global__ void __launch_bounds__(256) hd95_select_kernel(Hd95Meta* m, const unsigned long long* __restrict__ keys, int shift) {
  if (hd_empty(m)) return;
  __shared__ unsigned int h[256];
  __shared__ unsigned long long incl[256];
  const int tid = threadIdx.x;
  h[tid] = 0;
  __syncthreads();
  const unsigned long long n = m->n[0] + m->n[1], prefix = m->prefix;
  const unsigned long long mask = shift == 56 ? 0ull : ~0ull << (shift + 8);
  for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + tid; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
    const unsigned long long k = keys[i];
    if ((k & mask) == prefix) atomicAdd(&h[(k >> shift) & 255], 1u);
  }
  __syncthreads();
  if (h[tid]) atomicAdd(&m->hist[tid], (unsigned long long)h[tid]);
  if (!hd_last_block(&m->done)) return;
  unsigned long long rank = m->rank;
  if (shift == 56) {
    unsigned long long lo, hi;
    double gamma;
    hd_percentile_index(n, lo, hi, gamma);
    rank = lo;
  }
  const unsigned long long c = atomicExch(&m->hist[tid], 0ull);
  incl[tid] = c;
  __syncthreads();
  for (int o = 1; o < 256; o <<= 1) {
    const unsigned long long v = tid >= o ? incl[tid - o] : 0ull;
    __syncthreads();
    incl[tid] += v;
    __syncthreads();
  }
  const unsigned long long excl = incl[tid] - c;
  if (excl <= rank && rank < incl[tid]) {
    m->prefix = prefix | ((unsigned long long)tid << shift);
    m->rank = rank - excl;
    m->eq = c;
  }
  if (tid == 0) m->done = 0;
}

// x[hi] (the smallest key above x[lo] unless x[lo] repeats past rank lo) and the percentile's linear interpolation,
// numpy's _lerp without FMA.  Writes NaN when A or B is empty.  256 threads.
__global__ void __launch_bounds__(256) hd95_finish_kernel(Hd95Meta* m, const unsigned long long* __restrict__ keys, double* out) {
  if (hd_empty(m)) {
    if (blockIdx.x == 0 && threadIdx.x == 0) *out = __longlong_as_double(0x7ff8000000000000ll);
    return;
  }
  const unsigned long long n = m->n[0] + m->n[1], xlo = m->prefix;
  unsigned long long lo, hi;
  double gamma;
  hd_percentile_index(n, lo, hi, gamma);
  const bool next = hi > lo && m->rank + 1 >= m->eq;
  unsigned long long best = ~0ull;
  if (next)
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
      const unsigned long long k = keys[i];
      if (k > xlo && k < best) best = k;
    }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long v = __shfl_xor_sync(0xffffffffu, best, o);
    best = v < best ? v : best;
  }
  if ((threadIdx.x & 31) == 0 && best != ~0ull) atomicMin(&m->above, best);
  if (!hd_last_block(&m->done) || threadIdx.x != 0) return;
  const double a = __longlong_as_double((long long)xlo);
  const double b = next ? __longlong_as_double((long long)atomicAdd(&m->above, 0ull)) : a;
  const double diff = __dsub_rn(b, a);
  *out = gamma >= 0.5 ? __dsub_rn(b, __dmul_rn(diff, __dsub_rn(1.0, gamma))) : __dadd_rn(a, __dmul_rn(diff, gamma));
}

}  // namespace dunet
