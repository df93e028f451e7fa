// SURVEY.md 8f-4: MAE and S-measure of the reference's test path (twig/metric/MAE.py:18-36, Smeasure.py:18-36;
// arithmetic = pysodmetrics 1.3.1, restated in oracle/metrics_ref.py) as batched per-image reductions.
//
// HBM-bound integer/byte work: the wrappers quantise prediction and label to uint8 first, so every sum the two
// metrics need is an exact integer.  Pass 1 quantises (2 bytes per pixel kept) and reduces min / max / foreground
// count / foreground index sums per image; pass 2 accumulates, per centroid quadrant, the integer moments
// S(d), S(g), S(d^2), S(d g), S(d^2 g) of d = pred_u8 - min; a one-thread-per-image tail evaluates both metrics in
// float64 from the exact integers (variances as N*S2 - S1^2: no cancellation).  No atomics, no floating-point
// reduction: results are bit-stable and independent of the launch geometry.  The weighted F-measure (below
// metric_curves_kernel) reuses the quantise and info passes and adds an exact Euclidean distance transform.
#include <math_constants.h>

#include "common.cuh"

namespace dgtd {

constexpr int MROWS = 8;     // image rows per CTA
constexpr int NS1 = 5;       // min, max, count, sum(row), sum(col)
constexpr int NS2 = 20;      // 4 quadrants x {S(d), S(g), S(d^2), S(d g), S(d^2 g)}

struct MetricWs {
  unsigned char* pu8;
  unsigned char* gu8;
  long long* part1;   // [B][chunks][NS1]
  int* info;          // [B][4] = dmin, R, x, y
  unsigned long long* part2;  // [B][chunks][NS2]
  unsigned int* part3;        // [B][chunks][512]: 256-bin histograms of the re-quantised prediction, fg | bg
};

static inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

static MetricWs carve(void* ws, int B, int H, int W, size_t* total) {
  const size_t hw = (size_t)H * W, chunks = (size_t)cdiv(H, MROWS);
  size_t off = 0;
  MetricWs m;
  char* base = (char*)ws;
  m.pu8 = (unsigned char*)(base + off); off = align256(off + B * hw);
  m.gu8 = (unsigned char*)(base + off); off = align256(off + B * hw);
  m.part1 = (long long*)(base + off); off = align256(off + B * chunks * NS1 * sizeof(long long));
  m.info = (int*)(base + off); off = align256(off + (size_t)B * 4 * sizeof(int));
  m.part2 = (unsigned long long*)(base + off); off = align256(off + B * chunks * NS2 * sizeof(unsigned long long));
  m.part3 = (unsigned int*)(base + off); off = align256(off + B * chunks * 512 * sizeof(unsigned int));
  if (total) *total = off;
  return m;
}

// Per-image geometry.  Every image owns an H x W slot (row pitch W) of the batch tensors and of the workspace.
// `Dense`: the image fills its slot.  `Sized`: image b is the top-left sizes[b] = (H_b, W_b) of its slot and the rest
// of the slot is never read; a size outside [2, H] x [2, W] reads as 0 x 0, so the image does no work and its outputs
// are NaN.  Chunks, rows and tiles of the slot outside the image write identity partials, so an image's values equal
// a Dense call on its crop alone, bit for bit.
struct Dims { int h, w; };

struct Dense {
  static constexpr bool sized = false;
  int H, W;
  __device__ __forceinline__ Dims dims(int) const { return {H, W}; }
  // slot offset of pixel i (row-major index within an image of width w)
  __device__ __forceinline__ int64_t at(int i, int) const { return i; }
};

struct Sized {
  static constexpr bool sized = true;
  const int* sizes;   // [B][2] = (H_b, W_b)
  int H, W;
  __device__ __forceinline__ Dims dims(int b) const {
    const int h = sizes[2 * b], w = sizes[2 * b + 1];
    return (h >= 2 && h <= H && w >= 2 && w <= W) ? Dims{h, w} : Dims{0, 0};
  }
  __device__ __forceinline__ int64_t at(int i, int w) const {
    const int r = i / w;
    return (int64_t)r * W + (i - r * w);
  }
};

__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// pass 1: `(x * 255).astype(np.uint8)` (Smeasure.py:25-26), gt > 128, per-band statistics
template <class G>
__global__ void __launch_bounds__(256) metric_quantise_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                                                              MetricWs m, G geo) {
  __shared__ long long red[8][NS1];
  const int b = blockIdx.y, chunk = blockIdx.x, nchunks = gridDim.x;
  const Dims d = geo.dims(b);
  const int H = d.h, W = d.w;
  const int r0 = chunk * MROWS, r1 = min(H, r0 + MROWS);
  const int64_t img = (int64_t)b * geo.H * geo.W;
  int vmin = 255, vmax = 0;
  long long cnt = 0, srow = 0, scol = 0;
  for (int i = r0 * W + threadIdx.x; i < r1 * W; i += 256) {
    const int64_t o = img + geo.at(i, W);
    const float p = pred[o], g = gt[o];
    const int pu = (int)(unsigned char)(int)(__fmul_rn(p, 255.0f));     // truncation toward zero, like astype
    const int gu = (int)(unsigned char)(int)(__fmul_rn(g, 255.0f));
    const int fg = gu > 128;
    m.pu8[o] = (unsigned char)pu;
    m.gu8[o] = (unsigned char)fg;
    vmin = min(vmin, pu);
    vmax = max(vmax, pu);
    if (fg) {
      const int r = i / W;
      cnt += 1;
      srow += r;
      scol += i - r * W;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    vmin = min(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
    vmax = max(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
  }
  cnt = warp_sum_ll(cnt);
  srow = warp_sum_ll(srow);
  scol = warp_sum_ll(scol);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    red[warp][0] = vmin; red[warp][1] = vmax; red[warp][2] = cnt; red[warp][3] = srow; red[warp][4] = scol;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    long long a = red[0][0], c = red[0][1], n = red[0][2], sr = red[0][3], sc = red[0][4];
    for (int w = 1; w < 8; ++w) {
      a = min(a, red[w][0]); c = max(c, red[w][1]); n += red[w][2]; sr += red[w][3]; sc += red[w][4];
    }
    long long* o = m.part1 + ((int64_t)b * nchunks + chunk) * NS1;
    o[0] = a; o[1] = c; o[2] = n; o[3] = sr; o[4] = sc;
  }
}

// per image: min-max normalisation constants (`_prepare_data`) and the centroid split (`Smeasure.centroid`)
template <class G>
__global__ void metric_info_kernel(MetricWs m, int nchunks, int B, G geo) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const Dims d = geo.dims(b);
  const long long* p = m.part1 + (int64_t)b * nchunks * NS1;
  long long a = 255, c = 0, n = 0, sr = 0, sc = 0;
  for (int k = 0; k < nchunks; ++k) {
    a = min(a, p[k * NS1 + 0]); c = max(c, p[k * NS1 + 1]); n += p[k * NS1 + 2]; sr += p[k * NS1 + 3]; sc += p[k * NS1 + 4];
  }
  int dmin = (int)a, R = (int)(c - a);
  if (R == 0) { dmin = 0; R = 255; }          // constant prediction: pred / 255 is left un-normalised
  double x, y;
  if (n == 0) {
    x = rint((double)d.w / 2.0); y = rint((double)d.h / 2.0);     // np.round = half to even
  } else {
    y = rint((double)sr / (double)n); x = rint((double)sc / (double)n);
  }
  int* o = m.info + b * 4;
  o[0] = dmin; o[1] = R; o[2] = (int)x + 1; o[3] = (int)y + 1;
}

// pass 2: integer moments per centroid quadrant
template <class G>
__global__ void __launch_bounds__(256) metric_moments_kernel(MetricWs m, G geo) {
  __shared__ unsigned long long red[8][NS2];
  const int b = blockIdx.y, chunk = blockIdx.x, nchunks = gridDim.x;
  const Dims dm = geo.dims(b);
  const int H = dm.h, W = dm.w;
  const int r0 = chunk * MROWS, r1 = min(H, r0 + MROWS);
  const int64_t img = (int64_t)b * geo.H * geo.W;
  const int dmin = m.info[b * 4 + 0], cx = m.info[b * 4 + 2], cy = m.info[b * 4 + 3];
  unsigned int s[NS2];
#pragma unroll
  for (int k = 0; k < NS2; ++k) s[k] = 0u;
  for (int i = r0 * W + threadIdx.x; i < r1 * W; i += 256) {
    const int64_t o = img + geo.at(i, W);
    const unsigned int d = (unsigned int)((int)m.pu8[o] - dmin), g = m.gu8[o];
    const int r = i / W, c = i - r * W;
    const int q = (r >= cy ? 2 : 0) + (c >= cx ? 1 : 0);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const unsigned int sel = (q == k) ? 1u : 0u;
      s[k * 5 + 0] += sel * d;
      s[k * 5 + 1] += sel * g;
      s[k * 5 + 2] += sel * d * d;
      s[k * 5 + 3] += sel * d * g;
      s[k * 5 + 4] += sel * d * d * g;
    }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < NS2; ++k) {
    unsigned long long v = s[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < NS2) {
    unsigned long long v = 0;
    for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x];
    m.part2[((int64_t)b * nchunks + chunk) * NS2 + threadIdx.x] = v;
  }
}

__device__ double ssim_from_moments(double N, double Sd, double Sg, double Sd2, double Sdg, double R) {
  // pysodmetrics Smeasure.ssim with x = pred = d / R, y = gt; unbiased (N - 1) moments from exact integers
  const double x = Sd / (R * N), y = Sg / N;
  const double den = N * (N - 1.0);
  const double sx = (N * Sd2 - Sd * Sd) / (den * R * R);
  const double sy = (N * Sg - Sg * Sg) / den;
  const double sxy = (N * Sdg - Sd * Sg) / (den * R);
  const double alpha = 4.0 * x * y * sxy;
  const double beta = (x * x + y * y) * (sx + sy);
  if (alpha != 0.0) return alpha / (beta + 2.220446049250313e-16);
  return beta == 0.0 ? 1.0 : 0.0;
}

__device__ double s_object_from_moments(double n, double S1, double S2, double R) {
  // values v = e / R with integer e: mean and std(ddof = 1)
  const double x = S1 / (R * n);
  const double var = (n * S2 - S1 * S1) / (n * (n - 1.0) * R * R);
  const double sigma = sqrt(var > 0.0 ? var : 0.0);
  return 2.0 * x / (x * x + 1.0 + sigma + 2.220446049250313e-16);
}

// out[b][0] = MAE, out[b][1] = S-measure; OS doubles per image
template <class G, int OS>
__global__ void metric_final_kernel(MetricWs m, int nchunks, int B, G geo, double* __restrict__ out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const Dims d = geo.dims(b);
  const int H = d.h, W = d.w;
  if (G::sized && H == 0) { out[b * OS + 0] = out[b * OS + 1] = CUDART_NAN; return; }
  double S[NS2];
  for (int k = 0; k < NS2; ++k) {
    unsigned long long v = 0;
    for (int c = 0; c < nchunks; ++c) v += m.part2[((int64_t)b * nchunks + c) * NS2 + k];
    S[k] = (double)v;      // < 2^53 for any image up to 16k x 16k
  }
  const double R = (double)m.info[b * 4 + 1];
  const int cx = m.info[b * 4 + 2], cy = m.info[b * 4 + 3];
  const double n = (double)H * (double)W;
  double Sd = 0, Sg = 0, Sd2 = 0, Sdg = 0, Sd2g = 0;
  for (int q = 0; q < 4; ++q) {
    Sd += S[q * 5 + 0]; Sg += S[q * 5 + 1]; Sd2 += S[q * 5 + 2]; Sdg += S[q * 5 + 3]; Sd2g += S[q * 5 + 4];
  }
  const double n_fg = Sg, n_bg = n - Sg;
  // MAE.step: mean |pred - gt| = (sum_bg d + sum_fg (R - d)) / (R n)
  out[b * OS + 0] = ((Sd - Sdg) + (n_fg * R - Sdg)) / (R * n);
  double sm;
  if (n_fg == 0.0) {
    sm = 1.0 - Sd / (R * n);
  } else if (n_bg == 0.0) {
    sm = Sd / (R * n);
  } else {
    const double Nq[4] = {(double)cy * cx, (double)cy * (W - cx), (double)(H - cy) * cx, (double)(H - cy) * (W - cx)};
    const double w1 = Nq[0] / n, w2 = Nq[1] / n, w3 = Nq[2] / n, w4 = 1.0 - w1 - w2 - w3;
    const double wq[4] = {w1, w2, w3, w4};
    bool degenerate = (n_fg < 2.0) || (n_bg < 2.0);     // the library's NaN cases: max(0, nan) == 0
    double region = 0.0;
    for (int q = 0; q < 4; ++q) {
      if (Nq[q] < 2.0) { degenerate = true; continue; }
      region += wq[q] * ssim_from_moments(Nq[q], S[q * 5 + 0], S[q * 5 + 1], S[q * 5 + 2], S[q * 5 + 3], R);
    }
    if (degenerate) {
      sm = 0.0;
    } else {
      // Smeasure.object: fg values pred[gt], bg values (1 - pred)[~gt] = (R - d) / R
      const double bd = Sd - Sdg, bd2 = Sd2 - Sd2g;
      const double e1 = n_bg * R - bd, e2 = n_bg * R * R - 2.0 * R * bd + bd2;
      const double u = n_fg / n;
      const double object = u * s_object_from_moments(n_fg, Sdg, Sd2g, R) + (1.0 - u) * s_object_from_moments(n_bg, e1, e2, R);
      sm = 0.5 * object + 0.5 * region;
      sm = sm > 0.0 ? sm : 0.0;
    }
  }
  out[b * OS + 1] = sm;
}

// p(u): the min-max normalised prediction of u8 value u, (u/255 - min/255) / (max/255 - min/255), in the library's
// IEEE order (explicit round-to-nearest intrinsics: no contraction).  dmin = 0, R = 255 is both the constant-prediction
// convention of metric_info_kernel (no normalisation) and the full-range case, where (p0 - 0) / (1 - 0) == p0 exactly.
__device__ __forceinline__ double norm_pred(int u, int dmin, int R) {
  const double p0 = __ddiv_rn((double)u, 255.0);
  const double mn = __ddiv_rn((double)dmin, 255.0), mx = __ddiv_rn((double)(dmin + R), 255.0);
  return (dmin == 0 && R == 255) ? p0 : __ddiv_rn(__dsub_rn(p0, mn), __dsub_rn(mx, mn));
}

// F- / E-measure (pysodmetrics `Fmeasure.cal_pr`, `Emeasure.cal_em_with_cumsumhistogram`): both are functions of the
// foreground / background histograms of the min-max normalised prediction re-quantised to uint8.  The library
// does that re-quantisation in float64 -- p(u) * 255, truncated -- and a value that lands on an integer can fall
// either side of it, so the 256-entry map is evaluated with the same IEEE operations in the same order.
template <class G>
__global__ void __launch_bounds__(256) metric_hist_kernel(MetricWs m, G geo) {
  __shared__ unsigned int hist[512];
  __shared__ unsigned char lut[256];
  const int b = blockIdx.y, chunk = blockIdx.x, nchunks = gridDim.x;
  const int dmin = m.info[b * 4 + 0], R = m.info[b * 4 + 1];
  {
    const int u = threadIdx.x;
    const double p = norm_pred(u, dmin, R);
    const int q = (u >= dmin && u <= dmin + R) ? (int)__dmul_rn(p, 255.0) : 0;
    lut[u] = (unsigned char)q;
    hist[u] = 0u;
    hist[256 + u] = 0u;
  }
  __syncthreads();
  const Dims d = geo.dims(b);
  const int H = d.h, W = d.w;
  const int r0 = chunk * MROWS, r1 = min(H, r0 + MROWS);
  const int64_t img = (int64_t)b * geo.H * geo.W;
  for (int i = r0 * W + threadIdx.x; i < r1 * W; i += 256) {
    const int64_t o = img + geo.at(i, W);
    atomicAdd(&hist[(m.gu8[o] ? 0 : 256) + lut[m.pu8[o]]], 1u);   // integer: exact in any order
  }
  __syncthreads();
  unsigned int* o = m.part3 + ((int64_t)b * nchunks + chunk) * 512;
  o[threadIdx.x] = hist[threadIdx.x];
  o[256 + threadIdx.x] = hist[256 + threadIdx.x];
}

// ---- adaptive threshold: numpy's `p.mean()` --------------------------------------------------------------------------
// pysodmetrics binarises at min(2 * p.mean(), 1), and a threshold one ulp off changes the binary map whenever 2 * mean
// lands on a prediction level, so the mean is summed in numpy's order: `pairwise_sum` over the flattened image, where a
// block of n <= 128 elements is a leaf (eight accumulators r[k] += a[i + k] for i = 8, 16, ... < n - n % 8, combined as
// ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7)), then the n % 8 rest in order; below 8 elements, in order from 0)
// and a larger block splits at n / 2 - (n / 2) % 8.  The tree depends on N = H_b W_b only.  A node is addressed by the
// bits of a path from its subtree's root (1 = right child); a node that stops splitting before the path ends is
// summed once, by the path whose remaining bits are 0, and its value is kept at that position.  The mean kernel sums
// one "tile" (a node whose leaves are at most PW_CTA_LEVELS splits down) per CTA, 8 lanes per leaf, and combines its
// leaves in shared memory; the curves tail combines the tiles.  No atomics: the result depends on N and the pixels
// only, not on how the tree is cut into tiles.
constexpr int PW_LEAF = 128;
constexpr int PW_CTA_LEVELS = 7;     // 2^7 leaf positions per CTA, 4 per group of 8 lanes

__host__ __device__ __forceinline__ int pw_left(int n) { return (n >> 1) & ~7; }

// splits from a node of n elements down to its deepest leaf, counted up to `cap`: the right child is never the smaller
// one, so the deepest leaf is on the right spine
__host__ __device__ __forceinline__ int pw_depth(int n, int cap) {
  int d = 0;
  for (; n > PW_LEAF && d < cap; ++d) n -= pw_left(n);
  return d;
}

__device__ __forceinline__ bool pw_is_leaf(int n) { return n <= PW_LEAF; }
__device__ __forceinline__ bool pw_is_tile(int n) { return pw_depth(n, PW_CTA_LEVELS + 1) <= PW_CTA_LEVELS; }

struct PwNode { int off, n, level; };

// follow the `levels` high bits of `path` down from a root of n elements, stopping early at a node where stop(n)
template <class Stop>
__device__ __forceinline__ PwNode pw_descend(int n, int path, int levels, Stop stop) {
  int off = 0, l = 0;
  for (; l < levels && !stop(n); ++l) {
    const int left = pw_left(n);
    if ((path >> (levels - 1 - l)) & 1) { off += left; n -= left; } else { n = left; }
  }
  return {off, n, l};
}

// tiles per image: 2^(top levels) for any image of at most n pixels (right child <= ceil(n / 2) + 7)
static int pw_slots(int64_t n) {
  int d = 0;
  for (; n > PW_LEAF; ++d) n = (n + 1) / 2 + 7;
  return 1 << (d > PW_CTA_LEVELS ? d - PW_CTA_LEVELS : 0);
}

// msum[b][p] = pairwise sum of tile p of image b (p = the tile's path from the root), read through the u8 prediction
// and the p(u) table
template <class G>
__global__ void __launch_bounds__(256) metric_mean_kernel(MetricWs m, G geo, double* __restrict__ msum, int slots) {
  __shared__ double tab[256];
  __shared__ double val[1 << PW_CTA_LEVELS];
  const int b = blockIdx.y, p = blockIdx.x;
  const Dims d = geo.dims(b);
  const int N = d.h * d.w, W = d.w;
  const int top = max(0, pw_depth(N, 32) - PW_CTA_LEVELS);
  if (N == 0 || p >= (1 << top)) return;
  const PwNode tile = pw_descend(N, p, top, pw_is_tile);
  if (p & ((1 << (top - tile.level)) - 1)) return;          // the tile is summed by a lower path
  tab[threadIdx.x] = norm_pred(threadIdx.x, m.info[b * 4 + 0], m.info[b * 4 + 1]);
  __syncthreads();
  const unsigned char* pu = m.pu8 + (int64_t)b * geo.H * geo.W;
  const int k = threadIdx.x & 7;
  for (int pos = threadIdx.x >> 3; pos < (1 << PW_CTA_LEVELS); pos += 32) {     // warp-uniform trip count
    const PwNode leaf = pw_descend(tile.n, pos, PW_CTA_LEVELS, pw_is_leaf);
    const bool mine = (pos & ((1 << (PW_CTA_LEVELS - leaf.level)) - 1)) == 0;
    const int off = tile.off + leaf.off, n = leaf.n, nfull = n - n % 8;
    double s = 0.0;
    if (mine && n >= 8) {
      s = tab[pu[geo.at(off + k, W)]];
      for (int i = 8 + k; i < nfull; i += 8) s += tab[pu[geo.at(off + i, W)]];
    }
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    if (mine && k == 0) {
      for (int i = nfull; i < n; ++i) s += tab[pu[geo.at(off + i, W)]];     // n < 8: s = 0, then every element
      val[pos] = s;
    }
  }
  __syncthreads();
  for (int L = PW_CTA_LEVELS - 1; L >= 0; --L) {
    for (int q = threadIdx.x; q < (1 << L); q += 256) {
      const PwNode c = pw_descend(tile.n, q, L, pw_is_leaf);
      if (c.level == L && !pw_is_leaf(c.n))
        val[q << (PW_CTA_LEVELS - L)] += val[(2 * q + 1) << (PW_CTA_LEVELS - 1 - L)];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) msum[(int64_t)b * slots + p] = val[0];
}

// Emeasure.cal_em_with_cumsumhistogram at one threshold (and cal_em_with_threshold: the same arithmetic and order)
__device__ __forceinline__ double emeasure(double fg_fg, double fg_bg, double gt_fg, double size) {
  const double eps = 2.220446049250313e-16;
  const double pred_fg = fg_fg + fg_bg, pred_bg = size - pred_fg;
  double total;
  if (gt_fg == 0.0) {
    total = pred_bg;
  } else if (gt_fg == size) {
    total = pred_fg;
  } else {
    const double bg_fg = gt_fg - fg_fg, bg_bg = pred_bg - bg_fg;
    const double mp = pred_fg / size, mg = gt_fg / size;
    const double a[2] = {1.0 - mp, 0.0 - mp}, c[2] = {1.0 - mg, 0.0 - mg};
    const double numel[4] = {fg_fg, fg_bg, bg_fg, bg_bg};
    total = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const double x = a[i >> 1], y = c[i & 1];
      const double align = 2.0 * (x * y) / (x * x + y * y + eps);
      total += (align + 1.0) * (align + 1.0) / 4.0 * numel[i];
    }
  }
  return total / (size - 1.0 + eps);
}

// curves[b][0][i] = changeable F-measure, curves[b][1][i] = E-measure at threshold 255 - i (the library's order).
// FULL: also curves[b][2][i] = precision, curves[b][3][i] = recall, and vals[b][2] = adaptive F-measure, vals[b][3] =
// adaptive E-measure from the tiles' sums msum[b][.] of metric_mean_kernel (combined here, in place).
template <class G, bool FULL>
__global__ void __launch_bounds__(256) metric_curves_kernel(MetricWs m, int nchunks, G geo, double* __restrict__ curves,
                                                            double* msum, int slots, double* __restrict__ vals) {
  constexpr int NC = FULL ? 4 : 2;
  __shared__ double cf[256], cb[256];
  __shared__ int ustar;
  const int b = blockIdx.x, t = threadIdx.x;
  const Dims d = geo.dims(b);
  if (G::sized && d.h == 0) {
#pragma unroll
    for (int k = 0; k < NC; ++k) curves[((int64_t)b * NC + k) * 256 + t] = CUDART_NAN;
    if (FULL && t == 0) vals[b * 4 + 2] = vals[b * 4 + 3] = CUDART_NAN;
    return;
  }
  if (FULL) {
    // the levels above the tiles, bottom up, then p(u) >= min(2 * mean, 1) for u >= u* only (p is increasing)
    const int N = d.h * d.w, top = max(0, pw_depth(N, 32) - PW_CTA_LEVELS);
    double* ms = msum + (int64_t)b * slots;
    for (int L = top - 1; L >= 0; --L) {
      for (int q = t; q < (1 << L); q += 256) {
        const PwNode c = pw_descend(N, q, L, pw_is_tile);
        if (c.level == L && !pw_is_tile(c.n)) ms[q << (top - L)] += ms[(2 * q + 1) << (top - 1 - L)];
      }
      __syncthreads();
    }
    const double thr = fmin(__dmul_rn(2.0, __ddiv_rn(ms[0], (double)N)), 1.0);
    const int dmin = m.info[b * 4 + 0], R = m.info[b * 4 + 1];
    if (t == 0) ustar = 256;
    __syncthreads();
    if (t >= dmin && t <= dmin + R && norm_pred(t, dmin, R) >= thr) atomicMin(&ustar, t);
  }
  unsigned long long f = 0, g = 0;
  for (int c = 0; c < nchunks; ++c) {
    const unsigned int* o = m.part3 + ((int64_t)b * nchunks + c) * 512;
    f += o[255 - t];          // flipped: entry t holds bin 255 - t
    g += o[256 + 255 - t];
  }
  cf[t] = (double)f;
  cb[t] = (double)g;
  __syncthreads();
  if (t == 0) {               // cumulative sums (exact: integers below 2^53)
    for (int i = 1; i < 256; ++i) { cf[i] += cf[i - 1]; cb[i] += cb[i - 1]; }
  }
  __syncthreads();
  const double size = (double)d.h * (double)d.w, gt_fg = cf[255];
  const double fg_fg = cf[t], fg_bg = cb[t];
  // Fmeasure.cal_pr, beta^2 = 0.3
  {
    double ps = fg_fg + fg_bg;
    if (ps == 0.0) ps = 1.0;
    const double T = gt_fg > 1.0 ? gt_fg : 1.0;
    const double prec = fg_fg / ps, rec = fg_fg / T;
    const double num = 1.3 * prec * rec;
    const double den = num == 0.0 ? 1.0 : 0.3 * prec + rec;
    curves[((int64_t)b * NC + 0) * 256 + t] = num / den;
    if (FULL) {
      curves[((int64_t)b * NC + 2) * 256 + t] = prec;
      curves[((int64_t)b * NC + 3) * 256 + t] = rec;
    }
  }
  curves[((int64_t)b * NC + 1) * 256 + t] = emeasure(fg_fg, fg_bg, gt_fg, size);
  if (FULL && t == 0) {
    // the pixels with p >= threshold are those with lut >= lut[u*]: entry 255 - lut[u*] of the cumulative counts
    const int dmin = m.info[b * 4 + 0], R = m.info[b * 4 + 1], u = ustar;
    double i_fg = 0.0, i_bg = 0.0;
    if (u < 256) {
      const int k = 255 - (int)__dmul_rn(norm_pred(u, dmin, R), 255.0);
      i_fg = cf[k];
      i_bg = cb[k];
    }
    // Fmeasure.cal_adaptive_fm: its own formula, not the curve's
    double fm = 0.0;
    if (i_fg != 0.0) {
      const double pre = __ddiv_rn(i_fg, __dadd_rn(i_fg, i_bg)), rec = __ddiv_rn(i_fg, gt_fg);
      fm = __ddiv_rn(__dmul_rn(__dmul_rn(1.3, pre), rec), __dadd_rn(__dmul_rn(0.3, pre), rec));
    }
    vals[b * 4 + 2] = fm;
    vals[b * 4 + 3] = emeasure(i_fg, i_bg, gt_fg, size);
  }
}

// ---- weighted F-measure (pysodmetrics `WeightedFmeasure.cal_wfm`, beta = 1) -----------------------------------------
// After the quantise and info passes above: (1) a table pass evaluates E = |p(u) - g| for both labels; (2) a column
// pass finds, per pixel, the nearest foreground row in its column (the lower row on a tie); (3) a row pass takes the
// lower envelope of the parabolas (x - j)^2 + dy_j^2 (Meijster et al. 2000, exact integer separators; the lower
// column on a tie), writes the u8 prediction of the nearest foreground pixel (Et, transposed) and sums the
// distance-weighted background errors of the row; (4) a tile pass applies the 7x7 Gaussian to Et at the foreground
// pixels and sums min(E, EA) per tile; (5) a per-image tail.  The two-pass tie rules make the nearest pixel the one
// with the least (squared distance, column, row): SciPy's `distance_transform_edt(return_indices=True)`.
// Row / column indices are int32 and squared distances int64 (H * W < 2^28).  No floating-point atomics: every
// sum has a fixed order that depends on H and W only.
constexpr int WCOLS = 32;    // columns per CTA of the column pass (one per lane)
constexpr int WTILE = 32;    // square output tile of the Gaussian pass
constexpr int WROWS = 64;    // image rows (one per thread) per CTA of the row pass

__device__ __forceinline__ int cdiv_d(int a, int b) { return (a + b - 1) / b; }

struct WfmWs {
  int* near;          // [B][H][W] nearest foreground row in the pixel's column, -1 if the column has none
  int* stk_s;         // [B][H][W] per-row envelope stack: parabola (column) ...
  int* stk_t;         // [B][H][W] ... and the first x it owns
  unsigned char* etT; // [B][W][H] u8 prediction at the nearest foreground pixel, transposed
  double* tab;        // [B][2][256] E for a background (0) / foreground (1) pixel of u8 value u
  double* rowbg;      // [B][H] sum over the row's background pixels of E * (2 - 0.5^(D / 5))
  double* tilefg;     // [B][tiles] sum over the tile's foreground pixels of min(E, EA)
};

static MetricWs carve_wfm(void* ws, int B, int H, int W, WfmWs* w, size_t* total) {
  const size_t hw = (size_t)H * W, chunks = (size_t)cdiv(H, MROWS);
  const size_t tiles = (size_t)cdiv(H, WTILE) * cdiv(W, WTILE);
  size_t off = 0;
  MetricWs m = {};
  char* base = (char*)ws;
  m.pu8 = (unsigned char*)(base + off); off = align256(off + B * hw);
  m.gu8 = (unsigned char*)(base + off); off = align256(off + B * hw);
  m.part1 = (long long*)(base + off); off = align256(off + B * chunks * NS1 * sizeof(long long));
  m.info = (int*)(base + off); off = align256(off + (size_t)B * 4 * sizeof(int));
  w->near = (int*)(base + off); off = align256(off + B * hw * sizeof(int));
  w->stk_s = (int*)(base + off); off = align256(off + B * hw * sizeof(int));
  w->stk_t = (int*)(base + off); off = align256(off + B * hw * sizeof(int));
  w->etT = (unsigned char*)(base + off); off = align256(off + B * hw);
  w->tab = (double*)(base + off); off = align256(off + (size_t)B * 512 * sizeof(double));
  w->rowbg = (double*)(base + off); off = align256(off + (size_t)B * H * sizeof(double));
  w->tilefg = (double*)(base + off); off = align256(off + B * tiles * sizeof(double));
  if (total) *total = off;
  return m;
}

// tab[b][g][u] = |p(u) - g|
__global__ void __launch_bounds__(256) wfm_table_kernel(MetricWs m, WfmWs w) {
  const int b = blockIdx.x, u = threadIdx.x;
  const double p = norm_pred(u, m.info[b * 4 + 0], m.info[b * 4 + 1]);
  w.tab[b * 512 + u] = fabs(p);
  w.tab[b * 512 + 256 + u] = fabs(__dsub_rn(p, 1.0));
}

// one lane per column, one warp per band of rows: band ends first, then each band scans down and up
template <class G>
__global__ void __launch_bounds__(256) wfm_column_kernel(MetricWs m, WfmWs w, G geo) {
  __shared__ int first[8][WCOLS], last[8][WCOLS];
  const int b = blockIdx.y, lane = threadIdx.x & 31, band = threadIdx.x >> 5;
  const int x = blockIdx.x * WCOLS + lane;
  const Dims d = geo.dims(b);
  const int H = d.h, W = d.w, P = geo.W;
  const int len = (H + 7) / 8, r0 = min(H, band * len), r1 = min(H, r0 + len);
  const int64_t img = (int64_t)b * geo.H * geo.W;
  const unsigned char* g = m.gu8 + img + x;
  int* nr = w.near + img + x;
  int f = -1, l = -1;
  if (x < W)
    for (int y = r0; y < r1; ++y)
      if (g[(int64_t)y * P]) { if (f < 0) f = y; l = y; }
  first[band][lane] = f;
  last[band][lane] = l;
  __syncthreads();
  if (x >= W) return;
  int up = -1, dn = -1;                      // nearest foreground row above the band / below it
  for (int k = 0; k < band; ++k) if (last[k][lane] >= 0) up = last[k][lane];
  for (int k = 7; k > band; --k) if (first[k][lane] >= 0) dn = first[k][lane];
  for (int y = r1 - 1; y >= r0; --y) {       // nearest at or below y, parked in the output
    if (g[(int64_t)y * P]) dn = y;
    nr[(int64_t)y * P] = dn;
  }
  for (int y = r0; y < r1; ++y) {            // nearest at or above y; a tie goes to the lower row
    if (g[(int64_t)y * P]) up = y;
    const int d = nr[(int64_t)y * P];
    nr[(int64_t)y * P] = (up >= 0 && (d < 0 || y - up <= d - y)) ? up : d;
  }
}

// one thread per image row: lower envelope of f_j(x) = (x - j)^2 + (near_j - y)^2 over the columns j that have a
// foreground pixel.  Parabola j gives way to u > j from x = sep(j, u) + 1 on, sep = floor((u^2 - j^2 + dy_u^2 -
// dy_j^2) / (2 (u - j))): an x where both are equal stays with the lower column.
template <class G>
__global__ void __launch_bounds__(WROWS) wfm_row_kernel(MetricWs m, WfmWs w, int B, G geo) {
  const int64_t row = (int64_t)blockIdx.x * WROWS + threadIdx.x;
  if (row >= (int64_t)B * geo.H) return;
  const int b = (int)(row / geo.H), y = (int)(row - (int64_t)b * geo.H);
  const Dims d = geo.dims(b);
  const int H = d.h, W = d.w, P = geo.W, PT = geo.H;
  if (G::sized && y >= H) return;            // below the image: the tail does not read rowbg[y]
  const int64_t img = (int64_t)b * geo.H * geo.W;
  const int* nr = w.near + row * P;
  int* S = w.stk_s + row * P;
  int* T = w.stk_t + row * P;
  int q = -1, sq = 0, tq = 0;
  long long dq2 = 0;                          // dy^2 of the top parabola
  for (int u = 0; u < W; ++u) {
    const int r = nr[u];
    if (r < 0) continue;
    const long long du2 = (long long)(r - y) * (r - y);
    // pop while u is strictly below the top parabola where that one starts
    while (q >= 0) {
      const long long a = (long long)(tq - sq) * (tq - sq) + dq2, c = (long long)(tq - u) * (tq - u) + du2;
      if (a <= c) break;
      if (--q >= 0) {
        sq = S[q]; tq = T[q];
        const long long d = nr[sq] - y;
        dq2 = d * d;
      }
    }
    if (q < 0) {
      q = 0; sq = u; tq = 0; dq2 = du2;
      S[0] = u; T[0] = 0;
    } else {
      const long long num = (long long)u * u - (long long)sq * sq + du2 - dq2;     // >= 0 after the pops
      const long long t = 1 + num / (2ll * (u - sq));
      if (t < W) {
        ++q; sq = u; tq = (int)t; dq2 = du2;
        S[q] = u; T[q] = tq;
      }
    }
  }
  const unsigned char* pu = m.pu8 + img + (int64_t)y * P;
  const unsigned char* gu = m.gu8 + img + (int64_t)y * P;
  unsigned char* et = w.etT + img + y;
  const double* tab0 = w.tab + b * 512;
  constexpr double kLogHalfOver5 = -0.6931471805599453 / 5.0;    // np.log(0.5) / 5
  double bg = 0.0;
  if (q >= 0) {
    int rq = nr[sq];
    for (int x = W - 1; x >= 0; --x) {
      et[(int64_t)x * PT] = m.pu8[img + (int64_t)rq * P + sq];
      if (!gu[x]) {
        const long long dx = x - sq, dy = rq - y;
        const double dist = sqrt((double)(dx * dx + dy * dy));
        bg += __dmul_rn(tab0[pu[x]], __dsub_rn(2.0, exp(__dmul_rn(kLogHalfOver5, dist))));
      }
      if (x == tq && --q >= 0) { sq = S[q]; tq = T[q]; rq = nr[sq]; }
    }
  } else {                                    // no foreground in the image: the tail returns 0
    for (int x = 0; x < W; ++x) et[(int64_t)x * PT] = 0;
  }
  w.rowbg[row] = bg;
}

// matlab_style_gauss2D((7, 7), sigma = 5) as pysodmetrics evaluates it, indexed by (|dy|, |dx|)
__constant__ double c_gauss7[4][4] = {
    {0.023835778808354184, 0.023363798765182044, 0.022003197046847913, 0.019909316004406315},
    {0.023363798765182044, 0.022901164553037447, 0.02156750455382744, 0.019515085133964022},
    {0.022003197046847913, 0.02156750455382744, 0.02031151086671146, 0.018378615049044533},
    {0.019909316004406315, 0.019515085133964022, 0.018378615049044533, 0.016629658588054284}};

// EA = Et (*) K with zero padding at the foreground pixels of a 32 x 32 tile; sum of min(E, EA) over them
template <class G>
__global__ void __launch_bounds__(256) wfm_gauss_kernel(MetricWs m, WfmWs w, G geo) {
  constexpr int S = WTILE + 6;
  __shared__ double et[S][S + 1];
  __shared__ double red[256];
  const int tiles_x = (geo.W + WTILE - 1) / WTILE;
  const int b = blockIdx.y, y0 = (blockIdx.x / tiles_x) * WTILE, x0 = (blockIdx.x % tiles_x) * WTILE;
  const Dims d = geo.dims(b);
  const int H = d.h, W = d.w, P = geo.W, PT = geo.H;
  if (G::sized && (y0 >= H || x0 >= W)) {                // outside the image: the tail does not read it
    if (threadIdx.x == 0) w.tilefg[(int64_t)b * gridDim.x + blockIdx.x] = 0.0;
    return;
  }
  const int64_t img = (int64_t)b * geo.H * geo.W;
  const double* tab1 = w.tab + b * 512 + 256;
  for (int i = threadIdx.x; i < S * S; i += 256) {      // lanes run along y: Et is stored transposed
    const int yy = i % S, xx = i / S, y = y0 - 3 + yy, x = x0 - 3 + xx;
    et[yy][xx] = (y >= 0 && y < H && x >= 0 && x < W) ? tab1[w.etT[img + (int64_t)x * PT + y]] : 0.0;
  }
  __syncthreads();
  const int tx = threadIdx.x & 31;
  double s = 0.0;
  for (int ty = threadIdx.x >> 5; ty < WTILE; ty += 8) {
    const int y = y0 + ty, x = x0 + tx;
    if (y >= H || x >= W || !m.gu8[img + (int64_t)y * P + x]) continue;
    double ea = 0.0;
#pragma unroll
    for (int i = 0; i < 7; ++i)
#pragma unroll
      for (int j = 0; j < 7; ++j) ea = fma(c_gauss7[abs(i - 3)][abs(j - 3)], et[ty + i][tx + j], ea);
    const double e = tab1[m.pu8[img + (int64_t)y * P + x]];
    s += ea < e ? ea : e;
  }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) w.tilefg[(int64_t)b * gridDim.x + blockIdx.x] = red[0];
}

// The image's own rows and its own cdiv(H_b, 32) x cdiv(W_b, 32) tiles, in row-major order: the float64 sums of a
// Sized call run in the order of a Dense call on the crop.
template <class G>
__global__ void wfm_final_kernel(MetricWs m, WfmWs w, int nchunks, int ntiles, int B, G geo, double* __restrict__ out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const Dims d = geo.dims(b);
  if (G::sized && d.h == 0) { out[b] = CUDART_NAN; return; }
  long long n = 0;
  for (int k = 0; k < nchunks; ++k) n += m.part1[((int64_t)b * nchunks + k) * NS1 + 2];
  if (n == 0) { out[b] = 0.0; return; }
  double fg = 0.0, bg = 0.0;
  const int tiles_x = cdiv_d(geo.W, WTILE), ty1 = cdiv_d(d.h, WTILE), tx1 = cdiv_d(d.w, WTILE);
  for (int ty = 0; ty < ty1; ++ty)
    for (int tx = 0; tx < tx1; ++tx) fg += w.tilefg[(int64_t)b * ntiles + ty * tiles_x + tx];
  for (int k = 0; k < d.h; ++k) bg += w.rowbg[(int64_t)b * geo.H + k];
  const double eps = 2.220446049250313e-16;
  const double tpw = (double)n - fg;
  const double R = 1.0 - fg / (double)n;
  const double P = tpw / (tpw + bg + eps);
  out[b] = 2.0 * R * P / (R + P + eps);
}

// The full table's workspace: carve()'s, then the tiles' sums of the mean pass
static size_t carve_full(int B, int H, int W, int* slots) {
  size_t off = 0;
  carve(nullptr, B, H, W, &off);
  *slots = pw_slots((int64_t)H * W);
  return off;
}

// FULL: out (B, 4) = MAE, S, adaptive F, adaptive E and curves (B, 4, 256) = F, E, precision, recall
template <bool FULL, class G>
static int launch_sod_metrics(const float* pred, const float* gt, void* ws, double* out, double* curves, int B, G geo,
                              cudaStream_t s) {
  MetricWs m = carve(ws, B, geo.H, geo.W, nullptr);
  const int nchunks = cdiv(geo.H, MROWS);
  metric_quantise_kernel<<<dim3(nchunks, B), 256, 0, s>>>(pred, gt, m, geo);
  DGTD_LAUNCH_CHECK("sod_metrics(quantise)");
  metric_info_kernel<<<cdiv(B, 32), 32, 0, s>>>(m, nchunks, B, geo);
  DGTD_LAUNCH_CHECK("sod_metrics(info)");
  metric_moments_kernel<<<dim3(nchunks, B), 256, 0, s>>>(m, geo);
  DGTD_LAUNCH_CHECK("sod_metrics(moments)");
  metric_final_kernel<G, FULL ? 4 : 2><<<cdiv(B, 32), 32, 0, s>>>(m, nchunks, B, geo, out);
  DGTD_LAUNCH_CHECK("sod_metrics(final)");
  if (curves) {
    metric_hist_kernel<<<dim3(nchunks, B), 256, 0, s>>>(m, geo);
    DGTD_LAUNCH_CHECK("sod_metrics(hist)");
    double* msum = nullptr;
    int slots = 0;
    if (FULL) {
      msum = (double*)((char*)ws + carve_full(B, geo.H, geo.W, &slots));
      metric_mean_kernel<<<dim3(slots, B), 256, 0, s>>>(m, geo, msum, slots);
      DGTD_LAUNCH_CHECK("sod_metrics_full(mean)");
    }
    metric_curves_kernel<G, FULL><<<B, 256, 0, s>>>(m, nchunks, geo, curves, msum, slots, out);
    DGTD_LAUNCH_CHECK("sod_metrics(curves)");
  }
  return 0;
}

template <class G>
static int launch_sod_wfm(const float* pred, const float* gt, void* ws, double* out, int B, G geo, cudaStream_t s) {
  const int H = geo.H, W = geo.W;
  WfmWs w;
  MetricWs m = carve_wfm(ws, B, H, W, &w, nullptr);
  const int nchunks = cdiv(H, MROWS), ntiles = cdiv(H, WTILE) * cdiv(W, WTILE);
  metric_quantise_kernel<<<dim3(nchunks, B), 256, 0, s>>>(pred, gt, m, geo);
  DGTD_LAUNCH_CHECK("sod_wfm(quantise)");
  metric_info_kernel<<<cdiv(B, 32), 32, 0, s>>>(m, nchunks, B, geo);
  DGTD_LAUNCH_CHECK("sod_wfm(info)");
  wfm_table_kernel<<<B, 256, 0, s>>>(m, w);
  DGTD_LAUNCH_CHECK("sod_wfm(table)");
  wfm_column_kernel<<<dim3(cdiv(W, WCOLS), B), 256, 0, s>>>(m, w, geo);
  DGTD_LAUNCH_CHECK("sod_wfm(column)");
  wfm_row_kernel<<<cdiv((int64_t)B * H, WROWS), WROWS, 0, s>>>(m, w, B, geo);
  DGTD_LAUNCH_CHECK("sod_wfm(row)");
  wfm_gauss_kernel<<<dim3(ntiles, B), 256, 0, s>>>(m, w, geo);
  DGTD_LAUNCH_CHECK("sod_wfm(gauss)");
  wfm_final_kernel<<<cdiv(B, 32), 32, 0, s>>>(m, w, nchunks, ntiles, B, geo, out);
  DGTD_LAUNCH_CHECK("sod_wfm(final)");
  return 0;
}

}  // namespace dgtd
using namespace dgtd;

extern "C" {

int64_t dgtd_sod_metrics_ws_bytes(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return 0;
  size_t total = 0;
  carve(nullptr, B, H, W, &total);
  return (int64_t)total;
}

int dgtd_sod_metrics_fwd(const float* pred, const float* gt, void* ws, double* out, double* curves, int B, int H,
                         int W, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(pred && gt && ws && out, "sod_metrics: null pointer");
  DGTD_CHECK_ARG(B > 0 && H > 1 && W > 1 && (int64_t)H * W < (1ll << 28), "sod_metrics: bad shape");
  DGTD_CHECK_ARG(((uintptr_t)ws & 255) == 0, "sod_metrics: workspace must be 256-byte aligned");
  return launch_sod_metrics<false>(pred, gt, ws, out, curves, B, Dense{H, W}, (cudaStream_t)stream);
}

int dgtd_sod_metrics_sized_fwd(const float* pred, const float* gt, const int32_t* sizes, void* ws, double* out,
                               double* curves, int B, int Hmax, int Wmax, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(pred && gt && sizes && ws && out, "sod_metrics: null pointer");
  DGTD_CHECK_ARG(B > 0 && Hmax > 1 && Wmax > 1 && (int64_t)Hmax * Wmax < (1ll << 28), "sod_metrics: bad shape");
  DGTD_CHECK_ARG(((uintptr_t)ws & 255) == 0, "sod_metrics: workspace must be 256-byte aligned");
  return launch_sod_metrics<false>(pred, gt, ws, out, curves, B, Sized{sizes, Hmax, Wmax}, (cudaStream_t)stream);
}

int64_t dgtd_sod_metrics_full_ws_bytes(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return 0;
  int slots = 0;
  const size_t off = carve_full(B, H, W, &slots);
  return (int64_t)align256(off + (size_t)B * slots * sizeof(double));
}

int dgtd_sod_metrics_full_fwd(const float* pred, const float* gt, void* ws, double* vals, double* curves, int B, int H,
                              int W, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(pred && gt && ws && vals && curves, "sod_metrics_full: null pointer");
  DGTD_CHECK_ARG(B > 0 && H > 1 && W > 1 && (int64_t)H * W < (1ll << 28), "sod_metrics_full: bad shape");
  DGTD_CHECK_ARG(((uintptr_t)ws & 255) == 0, "sod_metrics_full: workspace must be 256-byte aligned");
  return launch_sod_metrics<true>(pred, gt, ws, vals, curves, B, Dense{H, W}, (cudaStream_t)stream);
}

int dgtd_sod_metrics_full_sized_fwd(const float* pred, const float* gt, const int32_t* sizes, void* ws, double* vals,
                                    double* curves, int B, int Hmax, int Wmax, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(pred && gt && sizes && ws && vals && curves, "sod_metrics_full: null pointer");
  DGTD_CHECK_ARG(B > 0 && Hmax > 1 && Wmax > 1 && (int64_t)Hmax * Wmax < (1ll << 28), "sod_metrics_full: bad shape");
  DGTD_CHECK_ARG(((uintptr_t)ws & 255) == 0, "sod_metrics_full: workspace must be 256-byte aligned");
  return launch_sod_metrics<true>(pred, gt, ws, vals, curves, B, Sized{sizes, Hmax, Wmax}, (cudaStream_t)stream);
}

int64_t dgtd_sod_wfm_ws_bytes(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return 0;
  size_t total = 0;
  WfmWs w;
  carve_wfm(nullptr, B, H, W, &w, &total);
  return (int64_t)total;
}

int dgtd_sod_wfm_fwd(const float* pred, const float* gt, void* ws, double* out, int B, int H, int W,
                     dgtd_stream_t stream) {
  DGTD_CHECK_ARG(pred && gt && ws && out, "sod_wfm: null pointer");
  DGTD_CHECK_ARG(B > 0 && H > 1 && W > 1 && (int64_t)H * W < (1ll << 28), "sod_wfm: bad shape");
  DGTD_CHECK_ARG(((uintptr_t)ws & 255) == 0, "sod_wfm: workspace must be 256-byte aligned");
  return launch_sod_wfm(pred, gt, ws, out, B, Dense{H, W}, (cudaStream_t)stream);
}

int dgtd_sod_wfm_sized_fwd(const float* pred, const float* gt, const int32_t* sizes, void* ws, double* out, int B,
                           int Hmax, int Wmax, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(pred && gt && sizes && ws && out, "sod_wfm: null pointer");
  DGTD_CHECK_ARG(B > 0 && Hmax > 1 && Wmax > 1 && (int64_t)Hmax * Wmax < (1ll << 28), "sod_wfm: bad shape");
  DGTD_CHECK_ARG(((uintptr_t)ws & 255) == 0, "sod_wfm: workspace must be 256-byte aligned");
  return launch_sod_wfm(pred, gt, ws, out, B, Sized{sizes, Hmax, Wmax}, (cudaStream_t)stream);
}

}  // extern "C"
