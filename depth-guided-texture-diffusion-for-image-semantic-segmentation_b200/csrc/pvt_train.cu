// Backward of the non-GEMM pieces of the PVT-v2 blocks (SURVEY.md 8f-1, training; cod.py:824-961): the attention
// core (cod.py:911-915) and Mlp's depthwise 3x3 + GELU (cod.py:852-854, 1520-1531).  The projections, LayerNorms and
// patch embeds reuse the gradient kernels of the trunk (train_ops.cu / train_tc.cu / decoder_train.cu).
//   attention_stats   per query row: lse = log sum_j exp(scale q.k_j) and D = dO . O  (one warp per query)
//   attention_bwd     CTA = (chunk of 256 queries, head, image); per 64-key tile the five 64x64x64 products
//                     S = Q K^T, dP = dO V^T, dQ += dS K, dK += dS^T Q, dV += P^T dO as register-blocked fp32
//                     CUDA-core GEMMs out of shared memory (N_kv <= a few hundred keys: the work is 5 x the forward's);
//                     dK / dV leave through fp32 atomics (one flush per CTA and key tile), dQ is owned by the CTA.
//   dwconv3_gelu_bwd  du = g * gelu'(conv3(x) + b) with the conv recomputed from the 9 neighbours that also give the
//                     tap gradients dw[k] = sum du * x[p + k]; the input gradient is the same depthwise conv of du
//                     with the taps rotated (dgtd_dwconv3_fwd).
#include "common.cuh"

namespace dgtd {
namespace {

template <typename T>
__device__ __forceinline__ float4 ldq(const T* p);
template <>
__device__ __forceinline__ float4 ldq<float>(const float* p) { return *reinterpret_cast<const float4*>(p); }
template <>
__device__ __forceinline__ float4 ldq<__nv_bfloat16>(const __nv_bfloat16* p) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
  const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
  return make_float4(a.x, a.y, b.x, b.y);
}

constexpr int AB_D = 64;     // head dim
constexpr int AB_T = 64;     // tile: queries per block, keys per tile
constexpr int AB_P = 65;     // shared-memory row pitch (floats)
constexpr int AB_QCH = 256;  // queries per CTA
constexpr int AS_QB = 32;    // queries per CTA of the stats kernel

// rows [r0, r0 + 64) x 64 columns of a (rows_total, ld) matrix at column col0 -> dst[64][65]; zero beyond rows_total
template <typename T>
__device__ __forceinline__ void stage_tile(float* dst, const T* src, int64_t r0, int64_t rows_total, int64_t ld) {
  for (int i = threadIdx.x; i < AB_T * (AB_D / 4); i += blockDim.x) {
    const int r = i / (AB_D / 4), c = (i % (AB_D / 4)) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r0 + r < rows_total) v = ldq<T>(src + (r0 + r) * ld + c);
    float* d = dst + r * AB_P + c;
    d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
attention_stats_kernel(const T* __restrict__ q, const T* __restrict__ kv, const T* __restrict__ o,
                       const float* __restrict__ dout, float* __restrict__ lse, float* __restrict__ dsum, int N, int Nk,
                       int C, float scale) {
  __shared__ float Ks[AB_T * AB_P];
  __shared__ float Qs[AS_QB][AB_D];
  const int hd = blockIdx.y, b = blockIdx.z, heads = gridDim.y;
  const int q0 = blockIdx.x * AS_QB;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int QPW = AS_QB / 8;
  for (int i = threadIdx.x; i < AS_QB * (AB_D / 4); i += 256) {
    const int r = i / (AB_D / 4), c = (i % (AB_D / 4)) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (q0 + r < N) v = ldq<T>(q + ((int64_t)b * N + q0 + r) * C + hd * AB_D + c);
    Qs[r][c] = v.x; Qs[r][c + 1] = v.y; Qs[r][c + 2] = v.z; Qs[r][c + 3] = v.w;
  }
  float m[QPW], l[QPW];
#pragma unroll
  for (int i = 0; i < QPW; ++i) { m[i] = -INFINITY; l[i] = 0.f; }
  const T* kb = kv + (int64_t)b * Nk * 2 * C + hd * AB_D;
  for (int k0 = 0; k0 < Nk; k0 += AB_T) {
    __syncthreads();
    stage_tile<T>(Ks, kb, k0, Nk, 2 * C);
    __syncthreads();
#pragma unroll
    for (int i = 0; i < QPW; ++i) {
      const float* qr = Qs[warp * QPW + i];
      float s0 = 0.f, s1 = 0.f;
#pragma unroll 16
      for (int d = 0; d < AB_D; ++d) {
        const float qv = qr[d];
        s0 = fmaf(qv, Ks[lane * AB_P + d], s0);
        s1 = fmaf(qv, Ks[(lane + 32) * AB_P + d], s1);
      }
      s0 = (k0 + lane < Nk) ? s0 * scale : -INFINITY;
      s1 = (k0 + lane + 32 < Nk) ? s1 * scale : -INFINITY;
      float mx = fmaxf(s0, s1);
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
      const float mn = fmaxf(m[i], mx);
      const float e = warp_sum(expf(s0 - mn) + expf(s1 - mn));
      l[i] = l[i] * expf(m[i] - mn) + e;
      m[i] = mn;
    }
  }
#pragma unroll
  for (int i = 0; i < QPW; ++i) {
    const int n = q0 + warp * QPW + i;
    if (n >= N) continue;
    const int64_t row = ((int64_t)b * N + n) * C + hd * AB_D;
    float acc = to_float(o[row + lane]) * dout[row + lane] + to_float(o[row + lane + 32]) * dout[row + lane + 32];
    acc = warp_sum(acc);
    if (lane == 0) {
      const int64_t idx = ((int64_t)b * heads + hd) * N + n;
      lse[idx] = m[i] + logf(l[i]);
      dsum[idx] = acc;
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
attention_bwd_kernel(const T* __restrict__ q, const T* __restrict__ kv, const float* __restrict__ dout,
                     const float* __restrict__ lse, const float* __restrict__ dsum, float* __restrict__ dq,
                     float* __restrict__ dkv, int N, int Nk, int C, float scale) {
  extern __shared__ float sm[];
  float* Qs = sm;
  float* dOs = Qs + AB_T * AB_P;
  float* Ps = dOs + AB_T * AB_P;
  float* dSs = Ps + AB_T * AB_P;
  float* Ks = dSs + AB_T * AB_P;
  float* Vs = Ks + AB_T * AB_P;
  float* Ls = Vs + AB_T * AB_P;   // [64] lse
  float* Ds = Ls + AB_T;          // [64] dO . O
  const int hd = blockIdx.y, b = blockIdx.z, heads = gridDim.y;
  const int qc0 = blockIdx.x * AB_QCH;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const T* qb = q + (int64_t)b * N * C + hd * AB_D;
  const float* dob = dout + (int64_t)b * N * C + hd * AB_D;
  float* dqb = dq + (int64_t)b * N * C + hd * AB_D;
  const T* kb = kv + (int64_t)b * Nk * 2 * C + hd * AB_D;
  float* dkb = dkv + (int64_t)b * Nk * 2 * C + hd * AB_D;
  const float* lb = lse + ((int64_t)b * heads + hd) * N;
  const float* db = dsum + ((int64_t)b * heads + hd) * N;

  for (int k0 = 0; k0 < Nk; k0 += AB_T) {
    __syncthreads();
    stage_tile<T>(Ks, kb, k0, Nk, 2 * C);
    stage_tile<T>(Vs, kb + C, k0, Nk, 2 * C);
    float dK[4][4], dV[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) { dK[i][j] = 0.f; dV[i][j] = 0.f; }

    for (int qo = 0; qo < AB_QCH; qo += AB_T) {
      const int q0 = qc0 + qo;
      if (q0 >= N) break;
      __syncthreads();   // previous block's readers of Qs / dOs / Ps / dSs are done
      stage_tile<T>(Qs, qb, q0, N, C);
      stage_tile<float>(dOs, dob, q0, N, C);
      if (threadIdx.x < AB_T) {
        const bool ok = q0 + (int)threadIdx.x < N;
        Ls[threadIdx.x] = ok ? lb[q0 + threadIdx.x] : 0.f;
        Ds[threadIdx.x] = ok ? db[q0 + threadIdx.x] : 0.f;
      }
      __syncthreads();
      {  // S = Q K^T and dP = dO V^T for (q = ty + 16 i, key = tx + 16 j)
        float s[4][4], dp[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) { s[i][j] = 0.f; dp[i][j] = 0.f; }
#pragma unroll 4
        for (int d = 0; d < AB_D; ++d) {
          float qv[4], gv[4], kk[4], vv[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) { qv[i] = Qs[(ty + 16 * i) * AB_P + d]; gv[i] = dOs[(ty + 16 * i) * AB_P + d]; }
#pragma unroll
          for (int j = 0; j < 4; ++j) { kk[j] = Ks[(tx + 16 * j) * AB_P + d]; vv[j] = Vs[(tx + 16 * j) * AB_P + d]; }
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) { s[i][j] = fmaf(qv[i], kk[j], s[i][j]); dp[i][j] = fmaf(gv[i], vv[j], dp[i][j]); }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int qi = ty + 16 * i;
          const float L = Ls[qi], Dq = Ds[qi];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int kj = tx + 16 * j;
            const bool ok = (q0 + qi < N) && (k0 + kj < Nk);
            const float p = ok ? expf(s[i][j] * scale - L) : 0.f;
            Ps[qi * AB_P + kj] = p;
            dSs[qi * AB_P + kj] = p * (dp[i][j] - Dq) * scale;
          }
        }
      }
      __syncthreads();
      {  // dQ (q = ty + 16 i, d = tx + 16 j) += dS K
        float a[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) a[i][j] = 0.f;
#pragma unroll 4
        for (int k = 0; k < AB_T; ++k) {
          float sv[4], kk[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) sv[i] = dSs[(ty + 16 * i) * AB_P + k];
#pragma unroll
          for (int j = 0; j < 4; ++j) kk[j] = Ks[k * AB_P + tx + 16 * j];
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) a[i][j] = fmaf(sv[i], kk[j], a[i][j]);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int qi = q0 + ty + 16 * i;
          if (qi >= N) continue;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float* dst = dqb + (int64_t)qi * C + tx + 16 * j;
            *dst = (k0 == 0) ? a[i][j] : *dst + a[i][j];   // this CTA owns its query rows
          }
        }
      }
      // dK (key = ty + 16 i, d = tx + 16 j) += dS^T Q;  dV += P^T dO
#pragma unroll 4
      for (int r = 0; r < AB_T; ++r) {
        float sv[4], pv[4], qv[4], gv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { sv[i] = dSs[r * AB_P + ty + 16 * i]; pv[i] = Ps[r * AB_P + ty + 16 * i]; }
#pragma unroll
        for (int j = 0; j < 4; ++j) { qv[j] = Qs[r * AB_P + tx + 16 * j]; gv[j] = dOs[r * AB_P + tx + 16 * j]; }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) { dK[i][j] = fmaf(sv[i], qv[j], dK[i][j]); dV[i][j] = fmaf(pv[i], gv[j], dV[i][j]); }
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int kj = k0 + ty + 16 * i;
      if (kj >= Nk) continue;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        atomicAdd(dkb + (int64_t)kj * 2 * C + tx + 16 * j, dK[i][j]);
        atomicAdd(dkb + (int64_t)kj * 2 * C + C + tx + 16 * j, dV[i][j]);
      }
    }
  }
}

__device__ __forceinline__ float gelu_grad_exact(float x) {
  const float phi = 0.3989422804014327f * expf(-0.5f * x * x);
  return 0.5f * (1.0f + erff(x * 0.70710678118654752440f)) + x * phi;
}

// block = 64 channel quads x 4 sub-strips of DW_PIX / 4 pixels; grid = (C / 256, pixel strips)
constexpr int DW_PIX = 128;
template <typename T>
__global__ void __launch_bounds__(256)
dwconv3_gelu_bwd_kernel(const T* __restrict__ x, const float* __restrict__ wT, const float* __restrict__ bias,
                        const float* __restrict__ g, float* __restrict__ du, float* __restrict__ dwT,
                        float* __restrict__ dbias, int64_t M, int h, int w, int C) {
  __shared__ float red[3][64][41];
  const int quad = threadIdx.x & 63, sub = threadIdx.x >> 6;
  const int c = (blockIdx.x * 64 + quad) * 4;
  const bool live = c < C;
  float4 tap[9], bs = make_float4(0.f, 0.f, 0.f, 0.f);
  float acc[10][4];
#pragma unroll
  for (int k = 0; k < 10; ++k)
#pragma unroll
    for (int e = 0; e < 4; ++e) acc[k][e] = 0.f;
  if (live) {
#pragma unroll
    for (int k = 0; k < 9; ++k) tap[k] = *reinterpret_cast<const float4*>(wT + (int64_t)k * C + c);
    bs = *reinterpret_cast<const float4*>(bias + c);
    const int64_t p0 = (int64_t)blockIdx.y * DW_PIX + sub * (DW_PIX / 4);
    for (int t = 0; t < DW_PIX / 4; ++t) {
      const int64_t p = p0 + t;
      if (p >= M) break;
      const int px = (int)(p % w), py = (int)((p / w) % h);
      float4 nb[9];
      float4 u = bs;
#pragma unroll
      for (int k = 0; k < 9; ++k) {
        const int yy = py + k / 3 - 1, xx = px + k % 3 - 1;
        nb[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (yy >= 0 && yy < h && xx >= 0 && xx < w) nb[k] = ldq<T>(x + (p + (int64_t)(k / 3 - 1) * w + (k % 3 - 1)) * C + c);
        u.x = fmaf(tap[k].x, nb[k].x, u.x); u.y = fmaf(tap[k].y, nb[k].y, u.y);
        u.z = fmaf(tap[k].z, nb[k].z, u.z); u.w = fmaf(tap[k].w, nb[k].w, u.w);
      }
      const float4 gv = *reinterpret_cast<const float4*>(g + p * C + c);
      float4 d;
      d.x = gv.x * gelu_grad_exact(u.x); d.y = gv.y * gelu_grad_exact(u.y);
      d.z = gv.z * gelu_grad_exact(u.z); d.w = gv.w * gelu_grad_exact(u.w);
      *reinterpret_cast<float4*>(du + p * C + c) = d;
#pragma unroll
      for (int k = 0; k < 9; ++k) {
        acc[k][0] = fmaf(d.x, nb[k].x, acc[k][0]); acc[k][1] = fmaf(d.y, nb[k].y, acc[k][1]);
        acc[k][2] = fmaf(d.z, nb[k].z, acc[k][2]); acc[k][3] = fmaf(d.w, nb[k].w, acc[k][3]);
      }
      acc[9][0] += d.x; acc[9][1] += d.y; acc[9][2] += d.z; acc[9][3] += d.w;
    }
  }
  if (sub > 0) {
#pragma unroll
    for (int k = 0; k < 10; ++k)
#pragma unroll
      for (int e = 0; e < 4; ++e) red[sub - 1][quad][k * 4 + e] = acc[k][e];
  }
  __syncthreads();
  if (sub == 0 && live) {
#pragma unroll
    for (int k = 0; k < 10; ++k)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float v = acc[k][e] + red[0][quad][k * 4 + e] + red[1][quad][k * 4 + e] + red[2][quad][k * 4 + e];
        atomicAdd(k < 9 ? dwT + (int64_t)k * C + c + e : dbias + c + e, v);
      }
  }
}

}  // namespace
}  // namespace dgtd

namespace dgtd {
int64_t attention_bwd_tc_ws_floats(int B, int N, int Nk, int heads);   // attn_bwd_tc.cu
int attention_bwd_tc(const void* q, const void* kv, const void* o, const float* dout, float* dq, float* dkv, float* ws, int B,
                     int N, int Nk, int heads, float scale, cudaStream_t s);
int64_t dwconv3_gelu_bwd_tma_ws_floats();   // dwconv3_tma.cu
int dwconv3_gelu_bwd_tma(const void* x, const float* wT, const float* bias, const float* g, float* du, float* dwT,
                         float* dbias, float* ws, int B, int h, int w, int C, cudaStream_t s);
}
using namespace dgtd;

extern "C" {

int64_t dgtd_attention_bwd_ws_floats(int B, int N, int Nk, int heads) { return attention_bwd_tc_ws_floats(B, N, Nk, heads); }

int dgtd_attention_bwd(const void* q, const void* kv, const void* out, const float* dout, float* dq, float* dkv, float* ws,
                       int dtype, int B, int N, int Nk, int heads, float scale, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(q && kv && out && dout && dq && dkv && ws && B > 0 && N > 0 && Nk > 0 && heads > 0 && heads <= 65535 &&
                     B <= 65535,
                 "attention_bwd: bad args");
  DGTD_CHECK_ARG(dtype == DGTD_F32 || dtype == DGTD_BF16, "attention_bwd: bad dtype %d", dtype);
  const int C = heads * AB_D;
  cudaStream_t s = (cudaStream_t)stream;
  if (dtype == DGTD_BF16) {   // mma.sync path, no atomics (attn_bwd_tc.cu)
    const int rc = attention_bwd_tc(q, kv, out, dout, dq, dkv, ws, B, N, Nk, heads, scale, s);
    if (rc) return rc;
    DGTD_LAUNCH_CHECK("attention_bwd(tc)");
    return 0;
  }
  float* lse = ws;
  float* dsum = ws + (int64_t)B * N * heads;
  cudaError_t e = cudaMemsetAsync(dkv, 0, (size_t)B * Nk * 2 * C * sizeof(float), s);
  DGTD_CHECK_ARG(e == cudaSuccess, "attention_bwd: memset failed: %s", cudaGetErrorString(e));
  const size_t smem = (size_t)(6 * AB_T * AB_P + 2 * AB_T) * sizeof(float);
  dim3 gs(cdiv(N, AS_QB), heads, B), gb(cdiv(N, AB_QCH), heads, B);
  e = cudaFuncSetAttribute(attention_bwd_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  DGTD_CHECK_ARG(e == cudaSuccess, "attention_bwd: cannot opt in to %zu B smem", smem);
  attention_stats_kernel<<<gs, 256, 0, s>>>((const float*)q, (const float*)kv, (const float*)out, dout, lse, dsum, N, Nk,
                                             C, scale);
  DGTD_LAUNCH_CHECK("attention_stats");
  attention_bwd_kernel<<<gb, 256, smem, s>>>((const float*)q, (const float*)kv, dout, lse, dsum, dq, dkv, N, Nk, C, scale);
  DGTD_LAUNCH_CHECK("attention_bwd");
  return 0;
}

int64_t dgtd_dwconv3_gelu_bwd_ws_floats(void) { return dwconv3_gelu_bwd_tma_ws_floats(); }

int dgtd_dwconv3_gelu_bwd(const void* x, const float* wT, const float* bias, const float* g, float* du, float* dwT,
                          float* dbias, float* ws, int dtype, int B, int h, int w, int C, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(x && wT && bias && g && du && dwT && dbias && B > 0 && h > 0 && w > 0 && C > 0 && C % 4 == 0,
                 "dwconv3_gelu_bwd: bad args (C % 4)");
  DGTD_CHECK_ARG(dtype == DGTD_F32 || dtype == DGTD_BF16, "dwconv3_gelu_bwd: bad dtype %d", dtype);
  cudaStream_t s = (cudaStream_t)stream;
  if (dtype == DGTD_BF16) {   // persistent TMA-staged kernel, per-CTA partial tap gradients summed in order (no atomics)
    const int rc = dwconv3_gelu_bwd_tma(x, wT, bias, g, du, dwT, dbias, ws, B, h, w, C, s);
    if (rc < 0) return rc;
    if (rc == 0) {
      DGTD_LAUNCH_CHECK("dwconv3_gelu_bwd(tma)");
      count_launch();
      return 0;
    }
  }
  cudaError_t e1 = cudaMemsetAsync(dwT, 0, (size_t)9 * C * sizeof(float), s);
  cudaError_t e2 = cudaMemsetAsync(dbias, 0, (size_t)C * sizeof(float), s);
  DGTD_CHECK_ARG(e1 == cudaSuccess && e2 == cudaSuccess, "dwconv3_gelu_bwd: memset failed");
  const int64_t M = (int64_t)B * h * w;
  const int64_t strips = (M + DW_PIX - 1) / DW_PIX;
  DGTD_CHECK_ARG(strips <= 65535, "dwconv3_gelu_bwd: too many pixels for one launch");
  dim3 grid(cdiv(C / 4, 64), (unsigned)strips);
  if (dtype == DGTD_BF16)
    dwconv3_gelu_bwd_kernel<<<grid, 256, 0, s>>>((const __nv_bfloat16*)x, wT, bias, g, du, dwT, dbias, M, h, w, C);
  else
    dwconv3_gelu_bwd_kernel<<<grid, 256, 0, s>>>((const float*)x, wT, bias, g, du, dwT, dbias, M, h, w, C);
  DGTD_LAUNCH_CHECK("dwconv3_gelu_bwd");
  return 0;
}

}  // extern "C"
