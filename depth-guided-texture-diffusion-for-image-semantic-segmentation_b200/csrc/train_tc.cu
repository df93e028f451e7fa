// bf16 / tensor-core training path of the trunk: operand preparation for the tcgen05 gradient GEMMs.
//   dgrad  dX[M,K] = dY[M,N] . W[N,K]      -> tc_gemm2 with A = dY (bf16), B = W^T (cached)
//   wgrad  dW^T[K,N] = X^T[K,M] . dY^T[N,M] -> tc_gemm2 with both operands transposed (K-major over
//                                             the M rows) and split-K over M + fixed-order reduce
// The transposes are fused with the element-wise work that is needed anyway (DropPath / layer-scale
// factors, GELU and its derivative, bf16 down-cast), one pass over each tensor.
#include "tc_common.cuh"

namespace dgtd {

__device__ __forceinline__ float gelu_grad_f(float x) {
  const float phi = 0.3989422804014327f * expf(-0.5f * x * x);
  return 0.5f * (1.0f + erff(x * 0.70710678118654752440f)) + x * phi;
}

// gelu'(x) = Phi(x) + x phi(x) for two values at once on the bf16 training path: Phi from the packed polynomial of the
// forward epilogue (tc_common.cuh gelu_fast2: 0.5 + x Q(x^2) on |x| <= 4.5, abs error 3e-5), phi from one ex2.approx.
// ~11 issue slots per element instead of the erff + expf pair (~35); abs error <= 1e-4, far inside the bf16 rounding
// of the pre-activation it is evaluated at.
__device__ __forceinline__ void gelu_grad_fast2(float x0, float x1, float& d0, float& d1) {
  const float c0 = fminf(fmaxf(x0, -4.5f), 4.5f), c1 = fminf(fmaxf(x1, -4.5f), 4.5f);
  const uint64_t xc = pk2(c0, c1);
  const uint64_t t = mul2(xc, xc);
  uint64_t q = pk2(-1.400070736e-12f, -1.400070736e-12f);
  q = fma2(q, t, pk2(1.697307069e-10f, 1.697307069e-10f));
  q = fma2(q, t, pk2(-9.193762573e-09f, -9.193762573e-09f));
  q = fma2(q, t, pk2(2.958901695e-07f, 2.958901695e-07f));
  q = fma2(q, t, pk2(-6.365260363e-06f, -6.365260363e-06f));
  q = fma2(q, t, pk2(9.787139965e-05f, 9.787139965e-05f));
  q = fma2(q, t, pk2(-1.122678685e-03f, -1.122678685e-03f));
  q = fma2(q, t, pk2(9.833185488e-03f, 9.833185488e-03f));
  q = fma2(q, t, pk2(-6.633705714e-02f, -6.633705714e-02f));
  q = fma2(q, t, pk2(3.988837948e-01f, 3.988837948e-01f));
  float p0, p1;
  up2(fma2(xc, q, pk2(0.5f, 0.5f)), p0, p1);            // Phi(x), within 3e-5 of [0, 1]
  float e0, e1;                                          // phi(x) = 0.39894228 * 2^(-0.72134752 x^2)
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(-0.72134752f * x0 * x0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(-0.72134752f * x1 * x1));
  d0 = fmaf(x0 * 0.3989422804f, e0, p0);
  d1 = fmaf(x1 * 0.3989422804f, e1, p1);
}

// MODE 0: v = keep[m] * src[m,n]            (dst additionally * gamma[n])
// MODE 1: v = gelu(src[m,n])
// MODE 2: v = src[m,n] * gelu'(aux[m,n])    (src = dH, aux = pre-activation)
// dst  (M x N, bf16, nullable) = v (* gamma);  dstT (N x M, bf16, nullable) = v
template <typename ST, int MODE>
__global__ void __launch_bounds__(256)
transpose_op_kernel(const ST* __restrict__ src, const __nv_bfloat16* __restrict__ aux,
                    __nv_bfloat16* __restrict__ dst, __nv_bfloat16* __restrict__ dstT,
                    const float* __restrict__ keep, const float* __restrict__ gamma, int rows_per_sample, int M,
                    int N) {
  __shared__ float t[32][33];
  const int m0 = blockIdx.y * 32, n0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int m = m0 + i, n = n0 + threadIdx.x;
    float v = 0.f;
    if (m < M && n < N) {
      v = to_float(src[(int64_t)m * N + n]);
      if (MODE == 0 && keep) v *= keep[m / rows_per_sample];
      if (MODE == 1) v = gelu_erf(v);
      if (MODE == 2) v *= gelu_grad_f(__bfloat162float(aux[(int64_t)m * N + n]));
      // MODE 3: plain bf16 transpose / copy
      if (dst) dst[(int64_t)m * N + n] = __float2bfloat16_rn(MODE == 0 && gamma ? v * gamma[n] : v);
    }
    t[i][threadIdx.x] = v;
  }
  __syncthreads();
  if (dstT)
    for (int i = threadIdx.y; i < 32; i += 8) {
      const int n = n0 + i, m = m0 + threadIdx.x;
      if (n < N && m < M) dstT[(int64_t)n * M + m] = __float2bfloat16_rn(t[threadIdx.x][i]);
    }
}

// Same element-wise work without the transposed copy: 8 consecutive columns per thread (16-byte accesses).
__device__ __forceinline__ void load8f(const float* p, float (&f)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}
__device__ __forceinline__ void load8f(const __nv_bfloat16* p, float (&f)[8]) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = __bfloat1622float2(h[i]);
    f[2 * i] = t.x; f[2 * i + 1] = t.y;
  }
}
template <typename ST, int MODE>
__global__ void __launch_bounds__(256)
eltwise_op_kernel(const ST* __restrict__ src, const __nv_bfloat16* __restrict__ aux, __nv_bfloat16* __restrict__ dst,
                  const float* __restrict__ keep, const float* __restrict__ gamma, int rows_per_sample, int64_t total8,
                  int N) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total8) return;
  const int64_t e0 = i * 8;
  const int64_t m = e0 / N;
  const int n = (int)(e0 - m * N);
  float f[8];
  load8f(src + e0, f);
  if (MODE == 0) {
    const float k = keep ? keep[m / rows_per_sample] : 1.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) f[e] *= gamma ? k * gamma[n + e] : k;
  }
  if (MODE == 1) {
#pragma unroll
    for (int e = 0; e < 8; ++e) f[e] = gelu_erf(f[e]);
  }
  if (MODE == 2) {
    float a[8];
    load8f(aux + e0, a);
#pragma unroll
    for (int e = 0; e < 8; e += 2) {
      float d0, d1;
      gelu_grad_fast2(a[e], a[e + 1], d0, d1);
      f[e] *= d0; f[e + 1] *= d1;
    }
  }
  store8(dst + e0, f);
}

// The same element-wise pass that ALSO returns the column sums of what it writes (before the bf16 rounding): the
// bias gradient db1 = colsum(dH * gelu'(pre)) and the layer-scale / bias sum s = colsum(keep * g) used to be separate
// full passes over the (M x 4C) / (M x C) matrices (r2 profile: 3.4 ms of a 33 ms step).  CTA = RB rows x (TPR * 8)
// columns, thread = 8 columns x every RL-th row; fixed-order reduction over the row lanes in shared memory, one
// partial row per CTA row-block, summed by sum_parts_kernel (deterministic, no atomics).
template <typename ST, int MODE>
__global__ void __launch_bounds__(256)
eltwise_colsum_kernel(const ST* __restrict__ src, const __nv_bfloat16* __restrict__ aux, __nv_bfloat16* __restrict__ dst,
                      const float* __restrict__ keep, int rows_per_sample, float* __restrict__ part, int M, int N,
                      int tpr, int EC_RB) {
  __shared__ float red[256 * 8];
  const int tcol = threadIdx.x % tpr, rlane = threadIdx.x / tpr, rl = 256 / tpr;
  const int n = (blockIdx.x * tpr + tcol) * 8;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  // a CTA walks row blocks rb = blockIdx.y, + gridDim.y, ...: at most a few hundred partial rows whatever M is
  for (int r0 = blockIdx.y * EC_RB; r0 < M && n < N; r0 += gridDim.y * EC_RB) {
    const int r1 = min(M, r0 + EC_RB);
    // 4 rows per trip: all loads of a trip are issued before the first use (memory-level parallelism; a one-row loop
    // left each thread with a single 16-byte load in flight and ran at a third of the plain element-wise kernel)
    for (int mb = r0 + rlane; mb < r1; mb += 4 * rl) {
      float f[4][8], a[4][8];
      bool ok[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int m = mb + u * rl;
        ok[u] = m < r1;
        if (ok[u]) {
          load8f(src + (int64_t)m * N + n, f[u]);
          if (MODE == 2) load8f(aux + (int64_t)m * N + n, a[u]);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (!ok[u]) continue;
        const int m = mb + u * rl;
        if (MODE == 0) {
          const float k = keep ? keep[m / rows_per_sample] : 1.f;
#pragma unroll
          for (int e = 0; e < 8; ++e) f[u][e] *= k;
        }
        if (MODE == 2) {
#pragma unroll
          for (int e = 0; e < 8; e += 2) {
            float d0, d1;
            gelu_grad_fast2(a[u][e], a[u][e + 1], d0, d1);
            f[u][e] *= d0; f[u][e + 1] *= d1;
          }
        }
        store8(dst + (int64_t)m * N + n, f[u]);
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] += f[u][e];
      }
    }
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) red[(rlane * tpr + tcol) * 8 + e] = acc[e];
  __syncthreads();
  if (rlane == 0 && n < N) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      float v = 0.f;
      for (int q = 0; q < rl; ++q) v += red[(q * tpr + tcol) * 8 + e];
      part[(int64_t)blockIdx.y * N + n + e] = v;
    }
  }
}

// out[n] = sum_z part[z][n]: 32 columns x 8 row lanes per CTA, fixed-order tree (deterministic)
__global__ void __launch_bounds__(256)
colsum_parts_kernel(const float* __restrict__ part, float* __restrict__ out, int N, int S) {
  __shared__ float red[8][33];
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  const int n = blockIdx.x * 32 + cx;
  float v = 0.f;
  if (n < N)
    for (int z = ry; z < S; z += 8) v += part[(int64_t)z * N + n];
  red[ry][cx] = v;
  __syncthreads();
  if (ry == 0 && n < N) {
    float t = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) t += red[q][cx];
    out[n] = t;
  }
}

// column sums of a bf16 matrix: part[blk][n], then sum over blocks
__global__ void __launch_bounds__(256)
colsum_bf16_partial_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ part, int M, int N,
                           int rows_per_block) {
  __shared__ float red[8][32];
  const int n = blockIdx.x * 32 + (threadIdx.x & 31);
  const int r0 = blockIdx.y * rows_per_block, r1 = min(M, r0 + rows_per_block);
  float s = 0.f;
  if (n < N)
    for (int r = r0 + (threadIdx.x >> 5); r < r1; r += 8) s += __bfloat162float(x[(int64_t)r * N + n]);
  red[threadIdx.x >> 5][threadIdx.x & 31] = s;
  __syncthreads();
  if (threadIdx.x < 32 && n < N) {
    float tt = 0.f;
    for (int i = 0; i < 8; ++i) tt += red[i][threadIdx.x];
    part[(int64_t)blockIdx.y * N + n] = tt;
  }
}
__global__ void sum_parts_kernel(const float* __restrict__ part, float* __restrict__ out, int64_t n, int S,
                                 int64_t part_stride, int transpose_rows, int transpose_cols) {
  // out[i] = sum_z part[z][i];  with transpose_rows > 0 the (rows x cols) result is written transposed
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int z = 0; z < S; ++z) s += part[(int64_t)z * part_stride + i];
  if (transpose_rows > 0) {
    const int64_t r = i / transpose_cols, c = i - r * transpose_cols;
    out[c * transpose_rows + r] = s;
  } else {
    out[i] = s;
  }
}

int tc_gemm2_splitk(const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* B, int64_t ldb, float* partial, int M,
                    int N, int K, int splits, cudaStream_t s);

}  // namespace dgtd

using namespace dgtd;

extern "C" {

// mode 0: scale/cast (src fp32), 1: gelu (src bf16), 2: gelu backward (src = dH bf16, aux = pre bf16), 3: copy
int dgtd_transpose_op(const void* src, const void* aux, void* dst, void* dstT, const float* keep, const float* gamma,
                      int rows_per_sample, int M, int N, int mode, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(src && (dst || dstT) && M > 0 && N > 0 && mode >= 0 && mode <= 3, "transpose_op: bad args");
  DGTD_CHECK_ARG(mode != 2 || aux, "transpose_op: gelu backward needs the pre-activation");
  cudaStream_t s = (cudaStream_t)stream;
  const int rps = rows_per_sample > 0 ? rows_per_sample : 1;
  if (!dstT && N % 8 == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst) |
                               reinterpret_cast<uintptr_t>(aux)) & 15) == 0) {
    const int64_t total8 = (int64_t)M * N / 8;
    const unsigned blocks = (unsigned)cdiv(total8, (int64_t)256);
    __nv_bfloat16* d = (__nv_bfloat16*)dst;
    if (mode == 0)
      eltwise_op_kernel<float, 0><<<blocks, 256, 0, s>>>((const float*)src, nullptr, d, keep, gamma, rps, total8, N);
    else if (mode == 1)
      eltwise_op_kernel<__nv_bfloat16, 1><<<blocks, 256, 0, s>>>((const __nv_bfloat16*)src, nullptr, d, nullptr, nullptr,
                                                                  1, total8, N);
    else if (mode == 2)
      eltwise_op_kernel<__nv_bfloat16, 2><<<blocks, 256, 0, s>>>((const __nv_bfloat16*)src, (const __nv_bfloat16*)aux, d,
                                                                  nullptr, nullptr, 1, total8, N);
    else
      eltwise_op_kernel<__nv_bfloat16, 3><<<blocks, 256, 0, s>>>((const __nv_bfloat16*)src, nullptr, d, nullptr, nullptr,
                                                                  1, total8, N);
    DGTD_LAUNCH_CHECK("transpose_op(eltwise)");
    return 0;
  }
  dim3 grid(cdiv(N, 32), cdiv(M, 32)), block(32, 8);
  DGTD_CHECK_ARG(grid.y <= 65535, "transpose_op: too many rows for one launch");
  if (mode == 0)
    transpose_op_kernel<float, 0><<<grid, block, 0, s>>>((const float*)src, nullptr, (__nv_bfloat16*)dst,
                                                          (__nv_bfloat16*)dstT, keep, gamma, rps, M, N);
  else if (mode == 1)
    transpose_op_kernel<__nv_bfloat16, 1><<<grid, block, 0, s>>>((const __nv_bfloat16*)src, nullptr,
                                                                  (__nv_bfloat16*)dst, (__nv_bfloat16*)dstT, nullptr,
                                                                  nullptr, 1, M, N);
  else if (mode == 2)
    transpose_op_kernel<__nv_bfloat16, 2><<<grid, block, 0, s>>>((const __nv_bfloat16*)src, (const __nv_bfloat16*)aux,
                                                                  (__nv_bfloat16*)dst, (__nv_bfloat16*)dstT, nullptr,
                                                                  nullptr, 1, M, N);
  else
    transpose_op_kernel<__nv_bfloat16, 3><<<grid, block, 0, s>>>((const __nv_bfloat16*)src, nullptr,
                                                                  (__nv_bfloat16*)dst, (__nv_bfloat16*)dstT, nullptr,
                                                                  nullptr, 1, M, N);
  DGTD_LAUNCH_CHECK("transpose_op");
  return 0;
}

// rows per CTA trip: as many as leave ~4 CTAs per SM (592 in total), between one 4-row trip per row lane and 64 rows
// (with a fixed 64 the 9216 x 2048 matrices of stage 2 ran on 144 CTAs, one 8-warp CTA per SM)
static int ec_rows(int M, int N, int tpr) {
  const int gx = cdiv(N / 8, tpr), rl = 256 / tpr;
  int rb = cdiv((int64_t)M * gx, 592);
  const int unit = 4 * rl;
  rb = cdiv(rb, unit) * unit;
  if (rb < unit) rb = unit;
  if (rb > 64) rb = 64 / unit * unit > 0 ? 64 / unit * unit : unit;
  return rb;
}
static int ec_row_ctas(int M, int N, int tpr) {
  const int gx = cdiv(N / 8, tpr);
  int gy = cdiv(M, ec_rows(M, N, tpr));
  const int cap = 592 / gx > 1 ? 592 / gx : 1;       // ~4 CTAs per SM in total
  return gy < cap ? gy : cap;
}
static int ec_tpr(int N) {
  int tpr = 256;                          // threads per row: the largest power of two <= min(256, N / 8)
  while (tpr > N / 8) tpr >>= 1;
  return tpr < 1 ? 1 : tpr;
}
int dgtd_eltwise_colsum_ws_floats(int M, int N) { return ec_row_ctas(M, N, ec_tpr(N)) * N; }

int dgtd_eltwise_colsum(const void* src, const void* aux, void* dst, const float* keep, int rows_per_sample, float* ws,
                        float* colsum, int M, int N, int mode, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(src && dst && ws && colsum, "eltwise_colsum: null pointer");
  DGTD_CHECK_ARG(mode == 0 || mode == 2, "eltwise_colsum: mode must be 0 (keep * fp32 src) or 2 (src * gelu'(aux))");
  DGTD_CHECK_ARG(mode != 2 || aux, "eltwise_colsum: mode 2 needs aux");
  DGTD_CHECK_ARG(M > 0 && N > 0 && N % 8 == 0, "eltwise_colsum: N must be a multiple of 8 (M=%d N=%d)", M, N);
  cudaStream_t s = (cudaStream_t)stream;
  const int rps = rows_per_sample > 0 ? rows_per_sample : 1;
  const int tpr = ec_tpr(N);
  const dim3 grid(cdiv(N / 8, tpr), ec_row_ctas(M, N, tpr));
  if (mode == 0)
    eltwise_colsum_kernel<float, 0><<<grid, 256, 0, s>>>((const float*)src, nullptr, (__nv_bfloat16*)dst, keep, rps, ws, M,
                                                         N, tpr, ec_rows(M, N, tpr));
  else
    eltwise_colsum_kernel<__nv_bfloat16, 2><<<grid, 256, 0, s>>>((const __nv_bfloat16*)src, (const __nv_bfloat16*)aux,
                                                                 (__nv_bfloat16*)dst, nullptr, 1, ws, M, N, tpr,
                                                                 ec_rows(M, N, tpr));
  DGTD_LAUNCH_CHECK("eltwise_colsum");
  colsum_parts_kernel<<<cdiv(N, 32), 256, 0, s>>>(ws, colsum, N, (int)grid.y);
  DGTD_LAUNCH_CHECK("eltwise_colsum.reduce");
  return 0;
}

int dgtd_colsum_bf16(const void* x, float* ws, float* out, int M, int N, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(x && ws && out && M > 0 && N > 0, "colsum_bf16: bad args");
  cudaStream_t s = (cudaStream_t)stream;
  const int nb = cdiv(M, 1024);
  colsum_bf16_partial_kernel<<<dim3(cdiv(N, 32), nb), 256, 0, s>>>((const __nv_bfloat16*)x, ws, M, N, 1024);
  DGTD_LAUNCH_CHECK("colsum_bf16");
  sum_parts_kernel<<<cdiv(N, 256), 256, 0, s>>>(ws, out, N, nb, N, 0, 0);
  DGTD_LAUNCH_CHECK("colsum_bf16.reduce");
  return 0;
}

// Weight gradients (Mo x No fp32) reduce over the long Kr axis: it is split across CTA pairs and the partial products
// are summed in a fixed order.  ws: dgtd_wgrad_tc_ws_floats floats.
static int wgrad_splits(int Mo, int No, int Kr) {
  const int tiles = cdiv(Mo, 256) * cdiv(No, No % 256 == 0 ? 256 : 128);
  int s = cdiv(148, tiles);
  const int kb = cdiv(Kr, 64);
  if (s > kb / 4) s = kb / 4;
  if (s < 1) s = 1;
  if (s > 64) s = 64;
  const int kbps = cdiv(kb, s);
  return cdiv(kb, kbps);   // no empty split
}
int dgtd_wgrad_tc_ws_floats(int Mo, int No, int Kr) { return wgrad_splits(Mo, No, Kr) * cdiv(Mo, 256) * 256 * No; }

// Weight gradient from UN-transposed operands: out (Mo x No) = a[Kr, Mo]^T . b[Kr, No], a and b row-major
// activation matrices (pitches lda / ldb elements, column slices allowed), read as MN-major UMMA operands.
// transpose_out != 0 writes out as (No x Mo).
int dgtd_wgrad_tc_mn(const void* a, int lda, const void* b, int ldb, float* out, float* ws, int Mo, int No, int Kr,
                     int transpose_out, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(a && b && out && ws, "wgrad_tc_mn: null pointer");
  DGTD_CHECK_ARG(Mo >= 8 && No >= 8 && Mo % 8 == 0 && No % 8 == 0 && Kr >= 1 && lda >= Mo && ldb >= No && lda % 8 == 0 &&
                     ldb % 8 == 0,
                 "wgrad_tc_mn: need Mo, No, lda, ldb multiples of 8 (got Mo=%d No=%d Kr=%d lda=%d ldb=%d)", Mo, No, Kr,
                 lda, ldb);
  DGTD_CHECK_ARG(((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15) == 0,
                 "wgrad_tc_mn: operands must be 16-byte aligned");
  cudaStream_t s = (cudaStream_t)stream;
  const int S = wgrad_splits(Mo, No, Kr);
  int rc = tc_gemm2_splitk((const __nv_bfloat16*)a, lda, (const __nv_bfloat16*)b, ldb, ws, Mo, No, Kr, S, s);
  if (rc) return rc;
  DGTD_LAUNCH_CHECK("wgrad_tc");
  const int64_t n = (int64_t)Mo * No;
  sum_parts_kernel<<<cdiv(n, 256), 256, 0, s>>>(ws, out, n, S, (int64_t)cdiv(Mo, 256) * 256 * No,
                                                transpose_out ? Mo : 0, No);
  DGTD_LAUNCH_CHECK("wgrad_tc.reduce");
  return 0;
}

}  // extern "C"
