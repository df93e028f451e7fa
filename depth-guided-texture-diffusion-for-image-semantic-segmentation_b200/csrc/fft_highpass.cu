// a2: prompt_encoder.fft (cod.py:1256-1271) without an FFT.
//
// Zeroing the centred (2*line)^2 block of the shifted spectrum removes the projection of the
// image onto the frequency band k in [-line, line-1] of each axis, so
//     out = | x - Re( P_h x P_w^T ) |,   P = E E^H / n  (n x n, Hermitian, circulant)
//         = | x - (A_h x A_w^T - B_h x B_w^T) |,   A = Re P,  B = Im P.
// A is a real symmetric circulant (dense product on the fp32 FMA pipe: two GEMMs per plane);
// B comes only from the unpaired bin k = -line:  B[a,b] = -sin(th_a - th_b)/n with
// th_a = 2 pi line a / n, i.e. rank 2, so B_h x B_w^T collapses to four scalars per plane.
#include "simt_gemm.cuh"

namespace dgtd {

// row 0 of A: r[d] = (1/n) sum_{k=-line}^{line-1} cos(2 pi k d / n); sc = [sin th | cos th].
__global__ void projector_row_kernel(float* __restrict__ P, float* __restrict__ sc, int n, int line) {
  int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= n) return;
  const double two_pi = 6.283185307179586476925286766559;
  double acc = 0.0;
  for (int k = -line; k < line; ++k) {
    long long r = ((long long)k * d) % n;  // exact angle reduction
    if (r < 0) r += n;
    acc += cos(two_pi * (double)r / (double)n);
  }
  P[d] = (float)(acc / n);
  long long r = ((long long)line * d) % n;
  double th = two_pi * (double)r / (double)n;
  sc[d] = (float)sin(th);
  sc[n + d] = (float)cos(th);
}
// A[a,b] = r[(a-b) mod n] (r even, so row 0 is r itself)
__global__ void projector_fill_kernel(float* __restrict__ P, int n) {
  int b = blockIdx.x * blockDim.x + threadIdx.x, a = blockIdx.y + 1;
  if (b >= n || a >= n) return;
  int d = a - b;
  if (d < 0) d += n;
  P[(int64_t)a * n + b] = P[d];
}

// coef[z] = {Qcc, Qcs, Qsc, Qss} / (H*W),  Qcs = sum_{b,c} cos_h[b] x[b,c] sin_w[c], ...
// Two levels so that the reduction fills the GPU at any batch (one CTA per plane left 3 CTAs at batch 1 and two
// uneven waves at batch 64: 237 us for 113 MB): COEF_CHUNKS CTAs per plane write partial sums, a second kernel adds
// them in a fixed order (bit-stable) and normalises.
constexpr int COEF_CHUNKS = 16;
__global__ void __launch_bounds__(256)
imag_coef_partial_kernel(const float* __restrict__ x, const float* __restrict__ sc_h, const float* __restrict__ sc_w,
                         float* __restrict__ partial, int H, int W, int vec) {
  __shared__ float red[4][8];
  const int plane = blockIdx.y, chunk = blockIdx.x;
  const int total = H * W, len = (total + COEF_CHUNKS - 1) / COEF_CHUNKS;
  const int i0 = chunk * len, i1 = min(total, i0 + len);
  const float* p = x + (int64_t)plane * total;
  float q[4] = {0.f, 0.f, 0.f, 0.f};
  if (vec && (W & 3) == 0 && (len & 3) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0) {
    // four columns of one row per step (W % 4 == 0): one division and one 16-byte load per four elements
#pragma unroll 3
    for (int i = i0 + threadIdx.x * 4; i < i1; i += 1024) {
      const int r = i / W, c = i - r * W;
      const float4 v = __ldg(reinterpret_cast<const float4*>(p + i));
      const float sh = __ldg(sc_h + r), ch = __ldg(sc_h + H + r);
      const float4 sw = __ldg(reinterpret_cast<const float4*>(sc_w + c)), cw = __ldg(reinterpret_cast<const float4*>(sc_w + W + c));
      const float vc = (cw.x * v.x + cw.y * v.y) + (cw.z * v.z + cw.w * v.w);
      const float vs = (sw.x * v.x + sw.y * v.y) + (sw.z * v.z + sw.w * v.w);
      q[0] = fmaf(ch, vc, q[0]);
      q[1] = fmaf(ch, vs, q[1]);
      q[2] = fmaf(sh, vc, q[2]);
      q[3] = fmaf(sh, vs, q[3]);
    }
  } else {
    for (int i = i0 + threadIdx.x; i < i1; i += 256) {
      int r = i / W, c = i - r * W;
      float v = p[i];
      float sh = sc_h[r], ch = sc_h[H + r], sw = sc_w[c], cw = sc_w[W + c];
      q[0] = fmaf(ch * cw, v, q[0]);
      q[1] = fmaf(ch * sw, v, q[1]);
      q[2] = fmaf(sh * cw, v, q[2]);
      q[3] = fmaf(sh * sw, v, q[3]);
    }
  }
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float s = warp_sum(q[j]);
    if (lane == 0) red[j][wid] = s;
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    float s = 0.f;
    for (int i = 0; i < 8; ++i) s += red[threadIdx.x][i];
    partial[((int64_t)plane * COEF_CHUNKS + chunk) * 4 + threadIdx.x] = s;
  }
}

__global__ void imag_coef_final_kernel(const float* __restrict__ partial, float* __restrict__ coef, int n, float hw) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;   // i = plane * 4 + j
  if (i >= n) return;
  const int plane = i >> 2, j = i & 3;
  float s = 0.f;
  for (int k = 0; k < COEF_CHUNKS; ++k) s += partial[((int64_t)plane * COEF_CHUNKS + k) * 4 + j];
  coef[i] = s / hw;
}

// `scratch`: >= planes * COEF_CHUNKS * 4 floats that nothing reads before the next kernel of the caller overwrites it
// vec = 1: four columns per step (the tensor-core variant).  The exact fp32 entry keeps the element-wise summation
// order its golden vectors and the 1e-4 gradient tests were validated with: the two orders agree to 2e-7, but the
// decoders behind this operator are ReLU networks and a pre-activation within that distance of zero flips its mask
// against the float64 oracle (seen once: one conv1 weight gradient of the 128^2 backbone test off by 1e-2).
static int launch_imag_coef(const float* x, const float* sc_h, const float* sc_w, float* scratch, float* coef, int planes,
                            int H, int W, cudaStream_t s, int vec) {
  imag_coef_partial_kernel<<<dim3(COEF_CHUNKS, planes), 256, 0, s>>>(x, sc_h, sc_w, scratch, H, W, vec);
  DGTD_LAUNCH_CHECK("fft_highpass.coef(partial)");
  imag_coef_final_kernel<<<cdiv(planes * 4, 256), 256, 0, s>>>(scratch, coef, planes * 4, (float)H * (float)W);
  DGTD_LAUNCH_CHECK("fft_highpass.coef");
  return 0;
}

struct EpiStore {
  float* out;
  int64_t ld, bs;
  __device__ __forceinline__ void operator()(int m, int n, int z, float4 v) const {
    store4(out + z * bs + (int64_t)m * ld + n, v.x, v.y, v.z, v.w);
  }
};

// out = | x - acc + (s_a s'_d Qcc - s_a c'_d Qcs - c_a s'_d Qsc + c_a c'_d Qss) |
struct EpiHighpass {
  const float* x;
  const float* sc_h;
  const float* sc_w;
  const float* coef;
  float* out;
  int H, W;
  __device__ __forceinline__ void operator()(int m, int n, int z, float4 v) const {
    const int64_t o = ((int64_t)z * H + m) * W + n;
    float4 xv = load4(x + o);
    float sa = sc_h[m], ca = sc_h[H + m];
    float4 q = load4(coef + z * 4);
    float4 sd = load4(sc_w + n), cd = load4(sc_w + W + n);
    float u = sa * q.x - ca * q.z;   // multiplies s'_d
    float t = ca * q.w - sa * q.y;   // multiplies c'_d
    store4(out + o, fabsf(xv.x - v.x + (u * sd.x + t * cd.x)), fabsf(xv.y - v.y + (u * sd.y + t * cd.y)),
           fabsf(xv.z - v.z + (u * sd.z + t * cd.z)), fabsf(xv.w - v.w + (u * sd.w + t * cd.w)));
  }
};


// ---- tensor-core variant (bf16 mode of the path): the two projector products as tcgen05 GEMMs over ALL planes,
// fp32-accurate through a two-term bf16 split of both operands:
//     x = x_hi + x_lo,  A = A_hi + A_lo   ->   x A  ~=  x_hi A_hi + x_hi A_lo + x_lo A_hi     (|err| ~ 2^-16 |x||A|)
// Each split product is ONE K-concatenated GEMM (one fp32 accumulation in TMEM, no accumulator round trips):
//   [x_hi | x_lo | x_hi] . [A_hi | A_hi | A_lo]^T = x_hi A_hi + x_lo A_hi + x_hi A_lo
// rows of 3 * W bf16; x_hi is stored twice (57 MB more written at batch 64) against two fp32 read-modify-write
// passes over the 113 MB accumulator per product when the three terms are accumulated by separate GEMMs.
// The second product contracts over image rows, so the intermediate is transposed per plane (fused with its split)
// and the result comes out transposed; the finishing kernel transposes back while applying the rank-2 imaginary
// term, the subtraction and |.|.
__global__ void split3_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ a3, int64_t rows, int W4) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // float4 index
  if (i >= rows * W4) return;
  const int64_t r = i / W4;
  const int c = (int)(i - r * W4) * 4, W = W4 * 4;
  const float4 v = *reinterpret_cast<const float4*>(x + i * 4);
  const float f[4] = {v.x, v.y, v.z, v.w};
  float h[4], l[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    h[e] = __bfloat162float(__float2bfloat16_rn(f[e]));
    l[e] = f[e] - h[e];
  }
  __nv_bfloat16* o = a3 + r * 3 * W + c;
  store4(o, h[0], h[1], h[2], h[3]);
  store4(o + W, l[0], l[1], l[2], l[3]);
  store4(o + 2 * W, h[0], h[1], h[2], h[3]);
}
// per plane (R x C fp32) -> (C rows) x [hi(R) | lo(R) | hi(R)] bf16.  64 x 32 tiles: eight loads in flight per thread,
// two adjacent r per lane on the way out (4-byte bf16x2 stores, 128 B per warp instruction).  R even.
__global__ void __launch_bounds__(256)
transpose_split3_kernel(const float* __restrict__ t, __nv_bfloat16* __restrict__ a3, int R, int C) {
  __shared__ float tile[64][33];
  const int64_t pb = (int64_t)blockIdx.z * R * C;
  const int r0 = blockIdx.y * 64, c0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  float v[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int rr = r0 + ty + 8 * e;
    v[e] = (rr < R && c0 + tx < C) ? __ldg(t + pb + (int64_t)rr * C + c0 + tx) : 0.f;
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) tile[ty + 8 * e][tx] = v[e];
  __syncthreads();
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int cl = ty + 8 * e, c = c0 + cl, r = r0 + 2 * tx;
    if (c < C && r < R) {
      const float v0 = tile[2 * tx][cl], v1 = tile[2 * tx + 1][cl];
      const __nv_bfloat162 h = __floats2bfloat162_rn(v0, v1);
      const float2 hf = __bfloat1622float2(h);
      const __nv_bfloat162 l = __floats2bfloat162_rn(v0 - hf.x, v1 - hf.y);
      __nv_bfloat16* o = a3 + ((int64_t)blockIdx.z * C + c) * 3 * R + r;
      *reinterpret_cast<__nv_bfloat162*>(o) = h;
      *reinterpret_cast<__nv_bfloat162*>(o + R) = l;
      *reinterpret_cast<__nv_bfloat162*>(o + 2 * R) = h;
    }
  }
}
// out[p][i][j] = | x[p][i][j] - yt[p][j][i] + (u_i * sin_w[j] + t_i * cos_w[j]) |   (EpiHighpass, transposed input)
__global__ void __launch_bounds__(256)
highpass_finish_kernel(const float* __restrict__ x, const float* __restrict__ yt, const float* __restrict__ sc_h,
                       const float* __restrict__ sc_w, const float* __restrict__ coef, float* __restrict__ out, int H,
                       int W) {
  __shared__ float tile[32][33];
  const int pl = blockIdx.z;
  const int64_t pb = (int64_t)pl * H * W;
  const int i0 = blockIdx.y * 32, j0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  // both operands are requested before the barrier: eight independent loads in flight per thread instead of four
  float yv[4], xv[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int k = ty + 8 * e;
    yv[e] = (j0 + k < W && i0 + tx < H) ? __ldg(yt + pb + (int64_t)(j0 + k) * H + i0 + tx) : 0.f;   // yt rows = j, columns = i
    xv[e] = (i0 + k < H && j0 + tx < W) ? __ldg(x + pb + (int64_t)(i0 + k) * W + j0 + tx) : 0.f;
  }
#pragma unroll
  for (int e = 0; e < 4; ++e) tile[ty + 8 * e][tx] = yv[e];
  __syncthreads();
  const float4 q = load4(coef + pl * 4);
  const int j = j0 + tx;
  const float sj = j < W ? sc_w[j] : 0.f, cj = j < W ? sc_w[W + j] : 0.f;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int k = ty + 8 * e, i = i0 + k;
    if (i < H && j < W) {
      const float sa = sc_h[i], ca = sc_h[H + i];
      const float u = sa * q.x - ca * q.z, t = ca * q.w - sa * q.y;
      out[pb + (int64_t)i * W + j] = fabsf(xv[e] - tile[tx][k] + (u * sj + t * cj));
    }
  }
}

}  // namespace dgtd

using namespace dgtd;

extern "C" {

int dgtd_lowpass_projector(float* P, float* sc, int n, int line, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(P && sc && n > 0 && line >= 0 && 2 * line <= n, "lowpass_projector: bad args");
  cudaStream_t s = (cudaStream_t)stream;
  projector_row_kernel<<<cdiv(n, 128), 128, 0, s>>>(P, sc, n, line);
  DGTD_LAUNCH_CHECK("lowpass_projector.row");
  if (n > 1) {
    projector_fill_kernel<<<dim3(cdiv(n, 128), n - 1), 128, 0, s>>>(P, n);
    DGTD_LAUNCH_CHECK("lowpass_projector.fill");
  }
  return 0;
}

int dgtd_fft_highpass_fwd(const float* x, const float* Ph, const float* Pw, const float* sc_h,
                          const float* sc_w, float* tmp, float* coef, float* out, int planes,
                          int H, int W, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(x && Ph && Pw && sc_h && sc_w && tmp && coef && out, "fft_highpass: null pointer");
  DGTD_CHECK_ARG(planes > 0 && H > 0 && W > 0 && (W % 4) == 0 && (H % 4) == 0,
                 "fft_highpass: H and W must be multiples of 4 (got %dx%d)", H, W);
  DGTD_CHECK_ARG(planes <= 65535, "fft_highpass: too many planes");
  cudaStream_t s = (cudaStream_t)stream;
  {  // partial sums live in `tmp` until the first GEMM overwrites it (H*W >= 64 floats per plane)
    int rc0 = launch_imag_coef(x, sc_h, sc_w, tmp, coef, planes, H, W, s, 0);
    if (rc0) return rc0;
  }
  {  // tmp = x . A_w^T over all (plane,row) rows at once
    RowMajorLoader al{x, W, 0, planes * H, W};
    RowMajorLoader bl{Pw, W, 0, W, W};
    EpiStore ep{tmp, W, 0};
    launch_simt_gemm<true, true>(al, bl, ep, planes * H, W, W, 1, s);
    DGTD_LAUNCH_CHECK("fft_highpass.rows");
  }
  {  // per plane: A_h . tmp, fused with the rank-2 imaginary term, the subtraction and |.|
    RowMajorLoader al{Ph, H, 0, H, H};
    RowMajorLoader bl{tmp, W, (int64_t)H * W, H, W};  // (K x N) row major, N contiguous
    EpiHighpass ep{x, sc_h, sc_w, coef, out, H, W};
    launch_simt_gemm<true, false>(al, bl, ep, H, W, H, planes, s);
    DGTD_LAUNCH_CHECK("fft_highpass.cols");
  }
  return 0;
}

// bf16-mode variant on the tcgen05 GEMMs, each split product as ONE K-concatenated GEMM (see above).
// Ph_cat / Pw_cat: [P_hi | P_hi | P_lo] per row (H x 3H, W x 3W bf16); ws_a: planes*H*W*3 bf16; ws_f32: planes*H*W fp32.
int dgtd_fft_highpass_tc3_fwd(const float* x, const void* Ph_cat, const void* Pw_cat, const float* sc_h, const float* sc_w,
                              void* ws_a, float* ws_f32, float* coef, float* out, int planes, int H, int W,
                              dgtd_stream_t stream) {
  DGTD_CHECK_ARG(x && Ph_cat && Pw_cat && sc_h && sc_w && ws_a && ws_f32 && coef && out, "fft_highpass_tc3: null pointer");
  DGTD_CHECK_ARG(planes > 0 && planes <= 65535 && H > 0 && W > 0 && (W % 8) == 0 && (H % 8) == 0,
                 "fft_highpass_tc3: H and W must be multiples of 8 (got %dx%d)", H, W);
  cudaStream_t s = (cudaStream_t)stream;
  __nv_bfloat16* a3 = (__nv_bfloat16*)ws_a;
  {  // partial sums live in ws_f32 until the first GEMM overwrites it
    int rc0 = launch_imag_coef(x, sc_h, sc_w, ws_f32, coef, planes, H, W, s, 1);
    if (rc0) return rc0;
  }
  const int64_t R = (int64_t)planes * H, R2 = (int64_t)planes * W;
  DGTD_CHECK_ARG(R < (1ll << 31) && R2 < (1ll << 31), "fft_highpass_tc3: too many rows");
  split3_bf16_kernel<<<(unsigned)cdiv(R * (W / 4), (int64_t)256), 256, 0, s>>>(x, a3, R, W / 4);
  DGTD_LAUNCH_CHECK("fft_highpass_tc3.split");
  int rc;
  // T[(p,i), j] = sum_k x[(p,i), k] A_w[j, k]
  if ((rc = dgtd_linear_fwd(a3, Pw_cat, nullptr, ws_f32, (int)R, W, 3 * W, W, DGTD_BF16, DGTD_F32, DGTD_ACT_NONE, stream))) return rc;
  // per plane transpose (+ split): Tt[(p,j), i] = T[(p,i), j]
  transpose_split3_kernel<<<dim3(cdiv(W, 32), cdiv(H, 64), planes), 256, 0, s>>>(ws_f32, a3, H, W);
  DGTD_LAUNCH_CHECK("fft_highpass_tc3.transpose");
  // Yt[(p,j), i'] = sum_i Tt[(p,j), i] A_h[i', i]
  if ((rc = dgtd_linear_fwd(a3, Ph_cat, nullptr, ws_f32, (int)R2, H, 3 * H, H, DGTD_BF16, DGTD_F32, DGTD_ACT_NONE, stream))) return rc;
  highpass_finish_kernel<<<dim3(cdiv(W, 32), cdiv(H, 32), planes), 256, 0, s>>>(x, ws_f32, sc_h, sc_w, coef, out, H, W);
  DGTD_LAUNCH_CHECK("fft_highpass_tc3.finish");
  return 0;
}

}  // extern "C"
