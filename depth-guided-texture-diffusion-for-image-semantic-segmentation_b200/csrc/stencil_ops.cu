// Memory/latency-bound pieces of the texture diffuser: surface normals (a1), the fused
// diffusion front (a3..a6), the stand-alone MessagePassing operator fwd/bwd (a6), and the
// small NCHW helpers that make every nn.Module of the path callable on its own.
#include <math_constants.h>

#include "common.cuh"

namespace dgtd {

constexpr int KS = 7, KK = 49, KR = 3;

// ------------------------------------------------------------------------------------ a1
// cod.py:96-109.  torch.gradient: central differences inside, one-sided at the edges.
__global__ void surface_normals_kernel(const float* __restrict__ d, float* __restrict__ out, int H,
                                       int W) {
  int b = blockIdx.z;
  int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
  if (x >= W || y >= H) return;
  const float* p = d + (int64_t)b * H * W;
  float gh, gw;
  if (H == 1) gh = 0.f;
  else if (y == 0) gh = p[W + x] - p[x];
  else if (y == H - 1) gh = p[(int64_t)y * W + x] - p[(int64_t)(y - 1) * W + x];
  else gh = (p[(int64_t)(y + 1) * W + x] - p[(int64_t)(y - 1) * W + x]) * 0.5f;
  if (W == 1) gw = 0.f;
  else if (x == 0) gw = p[(int64_t)y * W + 1] - p[(int64_t)y * W];
  else if (x == W - 1) gw = p[(int64_t)y * W + x] - p[(int64_t)y * W + x - 1];
  else gw = (p[(int64_t)y * W + x + 1] - p[(int64_t)y * W + x - 1]) * 0.5f;
  float nx = -gh, ny = -gw;
  float norm = sqrtf(nx * nx + ny * ny + 1.0f);
  float* o = out + (int64_t)b * 3 * H * W + (int64_t)y * W + x;
  o[0] = nx / norm;
  o[(int64_t)H * W] = ny / norm;
  o[(int64_t)2 * H * W] = 1.0f / norm;
}

// ------------------------------------------------------------------------------------ a3..a6
// One CTA per (image, latent channel); one thread per grid cell.  Each thread keeps its 49
// normalised weights in registers, the channel plane ping-pongs in shared memory, so the T
// iterations never touch HBM (cod.py:1201-1205).  FUSED = weights generated on chip from the
// nearest-sampled high-pass image (cod.py:1295-1296) and state from the depth taps
// (cod.py:1297-1298); otherwise weights / state are read from global (stand-alone operator).
template <bool FUSED, int MAXT>
__global__ void __launch_bounds__(MAXT)
diffuse_plane_kernel(const float* __restrict__ emb1, const float* __restrict__ depth,
                     const float* __restrict__ reg_w, const float* __restrict__ reg_b,
                     const float* __restrict__ enc_w, const float* __restrict__ enc_b,
                     const float* __restrict__ x_in, const float* __restrict__ weight,
                     float* __restrict__ out, float* __restrict__ save_states,
                     float* __restrict__ save_wn, int C, int H, int W, int gh, int gw, int wc, int T,
                     float eps) {
  extern __shared__ float sm[];  // 2 planes with a 3-cell zero halo
  const int pw = gw + 2 * KR, ph = gh + 2 * KR, plane = pw * ph;
  float* buf0 = sm;
  float* buf1 = sm + plane;
  const int c = blockIdx.x, b = blockIdx.y;
  const int p = threadIdx.x, hw = gh * gw;
  const bool live = p < hw;
  const int py = live ? p / gw : 0, px = live ? p - py * gw : 0;

  for (int i = threadIdx.x; i < 2 * plane; i += blockDim.x) sm[i] = 0.f;

  float wn[KK];
  float x0 = 0.f;
  if (live) {
    if (FUSED) {
      // nearest sample (ATen: src = min(floor(dst * in/out), in-1))
      int sy = min((int)floorf(py * ((float)H / gh)), H - 1);
      int sx = min((int)floorf(px * ((float)W / gw)), W - 1);
      const float* e = emb1 + (int64_t)b * 3 * H * W + (int64_t)sy * W + sx;
      float g0 = e[0], g1 = e[(int64_t)H * W], g2 = e[(int64_t)2 * H * W];
      float s = 0.f;
#pragma unroll
      for (int k = 0; k < KK; ++k) {
        const float* rw = reg_w + (int64_t)(c * KK + k) * 3;
        float v = fmaf(rw[2], g2, fmaf(rw[1], g1, fmaf(rw[0], g0, reg_b[c * KK + k])));
        v = sigmoidf_acc(v);
        wn[k] = v;
        s += v;
      }
      float inv = 1.0f / (s + eps);
#pragma unroll
      for (int k = 0; k < KK; ++k) wn[k] *= inv;
      // depth -> bilinear down (align_corners = False) -> per-channel affine
      int y0, y1, x0i, x1i;
      float ly, lx;
      bilinear_src(py, (float)H / gh, H, y0, y1, ly);
      bilinear_src(px, (float)W / gw, W, x0i, x1i, lx);
      const float* dp = depth + (int64_t)b * H * W;
      float d00 = dp[(int64_t)y0 * W + x0i], d01 = dp[(int64_t)y0 * W + x1i];
      float d10 = dp[(int64_t)y1 * W + x0i], d11 = dp[(int64_t)y1 * W + x1i];
      // the reference interpolates conv1x1(depth); the affine map commutes with the taps
      float e00 = fmaf(enc_w[c], d00, enc_b[c]), e01 = fmaf(enc_w[c], d01, enc_b[c]);
      float e10 = fmaf(enc_w[c], d10, enc_b[c]), e11 = fmaf(enc_w[c], d11, enc_b[c]);
      x0 = (1.f - ly) * ((1.f - lx) * e00 + lx * e01) + ly * ((1.f - lx) * e10 + lx * e11);
    } else {
      const int cw = (wc == 1) ? 0 : c;
      const float* wp = weight + ((int64_t)b * wc + cw) * KK * hw + p;
      float s = 0.f;
#pragma unroll
      for (int k = 0; k < KK; ++k) {
        wn[k] = wp[(int64_t)k * hw];
        s += wn[k];
      }
      float inv = 1.0f / (s + eps);   // cod.py:1201 divides; 1/x then multiply differs by <=1ulp
#pragma unroll
      for (int k = 0; k < KK; ++k) wn[k] = wn[k] * inv;
      x0 = x_in[((int64_t)b * C + c) * hw + p];
    }
    if (save_wn) {
      float* o = save_wn + ((int64_t)b * C + c) * KK * hw + p;
#pragma unroll
      for (int k = 0; k < KK; ++k) o[(int64_t)k * hw] = wn[k];
    }
  }
  __syncthreads();
  if (live) buf0[(py + KR) * pw + px + KR] = x0;
  if (live && save_states) save_states[(((int64_t)b * (T + 1)) * C + c) * hw + p] = x0;
  __syncthreads();

  float* cur = buf0;
  float* nxt = buf1;
  float v = x0;
  for (int t = 0; t < T; ++t) {
    if (live) {
      float acc = 0.f;
#pragma unroll
      for (int ki = 0; ki < KS; ++ki)
#pragma unroll
        for (int kj = 0; kj < KS; ++kj)
          acc = fmaf(wn[ki * KS + kj], cur[(py + ki) * pw + px + kj], acc);
      v = acc;
      nxt[(py + KR) * pw + px + KR] = v;
      if (save_states) save_states[(((int64_t)b * (T + 1) + t + 1) * C + c) * hw + p] = v;
    }
    __syncthreads();
    float* tmp = cur; cur = nxt; nxt = tmp;
  }
  if (live && out) out[((int64_t)b * C + c) * hw + p] = v;
}

// 1x1 conv C -> Cout on the tiny (B,C,G,G) state (message_passing.conv, cod.py:1206), also the
// generic NCHW 1x1 conv (+sigmoid) for the stand-alone modules.
template <bool SIGMOID>
__global__ void conv1x1_nchw_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                    const float* __restrict__ bias, float* __restrict__ out, int Cin,
                                    int Cout, int HW, int64_t x_batch_stride) {
  int b = blockIdx.z, co = blockIdx.y;
  int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  const float* xp = x + (int64_t)b * x_batch_stride + p;
  const float* wp = w + (int64_t)co * Cin;
  float acc = bias ? bias[co] : 0.f;
  for (int ci = 0; ci < Cin; ++ci) acc = fmaf(wp[ci], xp[(int64_t)ci * HW], acc);
  if (SIGMOID) acc = sigmoidf_acc(acc);
  out[((int64_t)b * Cout + co) * HW + p] = acc;
}

// bilinear sample (align_corners=False) of the (h, w) plane p at output pixel (oy, ox) of an (oh, ow) resize
__device__ __forceinline__ float bilinear_at(const float* __restrict__ p, int h, int w, int oh, int ow, int oy, int ox) {
  int y0, y1, x0, x1;
  float ly, lx;
  bilinear_src(oy, (float)h / oh, h, y0, y1, ly);
  bilinear_src(ox, (float)w / ow, w, x0, x1, lx);
  return (1.f - ly) * ((1.f - lx) * p[(int64_t)y0 * w + x0] + lx * p[(int64_t)y0 * w + x1]) +
         ly * ((1.f - lx) * p[(int64_t)y1 * w + x0] + lx * p[(int64_t)y1 * w + x1]);
}

__global__ void resize_nchw_kernel(const float* __restrict__ x, float* __restrict__ out, int h, int w,
                                   int oh, int ow, int bilinear) {
  int plane = blockIdx.z;
  int ox = blockIdx.x * blockDim.x + threadIdx.x, oy = blockIdx.y * blockDim.y + threadIdx.y;
  if (ox >= ow || oy >= oh) return;
  const float* p = x + (int64_t)plane * h * w;
  float v;
  if (bilinear) {
    v = bilinear_at(p, h, w, oh, ow, oy, ox);
  } else {
    int sy = min((int)floorf(oy * ((float)h / oh)), h - 1);
    int sx = min((int)floorf(ox * ((float)w / ow)), w - 1);
    v = p[(int64_t)sy * w + sx];
  }
  out[((int64_t)plane * oh + oy) * ow + ox] = v;
}

// Predict head for images of different sizes: plane b (h, w) -> sigmoid of its bilinear resize to sizes[b] = (H_b, W_b)
// in the top-left of an (Hmax, Wmax) plane, 0 in the rest.  Per image the same arithmetic as resize_nchw_kernel then
// sigmoid_kernel; a plane already at (H_b, W_b) is copied, as `Hitnet.predict_logits` skips that resize.  A size
// outside [2, Hmax] x [2, Wmax] fills the whole plane with NaN.
__global__ void resize_sigmoid_sized_kernel(const float* __restrict__ x, float* __restrict__ out,
                                            const int* __restrict__ sizes, int h, int w, int Hmax, int Wmax) {
  const int b = blockIdx.z;
  const int ox = blockIdx.x * blockDim.x + threadIdx.x, oy = blockIdx.y * blockDim.y + threadIdx.y;
  if (ox >= Wmax || oy >= Hmax) return;
  const int oh = sizes[2 * b], ow = sizes[2 * b + 1];
  float v = 0.f;
  if (!(oh >= 2 && oh <= Hmax && ow >= 2 && ow <= Wmax)) {
    v = CUDART_NAN_F;
  } else if (oy < oh && ox < ow) {
    const float* p = x + (int64_t)b * h * w;
    v = sigmoidf_acc((oh == h && ow == w) ? p[(int64_t)oy * w + ox] : bilinear_at(p, h, w, oh, ow, oy, ox));
  }
  out[((int64_t)b * Hmax + oy) * Wmax + ox] = v;
}

// Generic LayerNorm over the middle dim of (outer, C, inner); one warp per (outer, inner) row,
// two-pass statistics (cod.py:1045-1047 / F.layer_norm).
__global__ void layer_norm_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                  const float* __restrict__ b, float* __restrict__ out, int64_t rows,
                                  int C, int64_t inner, float eps) {
  int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  int lane = threadIdx.x & 31;
  int64_t o = row / inner, i = row - o * inner;
  const float* xp = x + o * C * inner + i;
  float s = 0.f;
  for (int c = lane; c < C; c += 32) s += xp[(int64_t)c * inner];
  float mean = warp_sum(s) / C;
  float q = 0.f;
  for (int c = lane; c < C; c += 32) {
    float d = xp[(int64_t)c * inner] - mean;
    q = fmaf(d, d, q);
  }
  float rstd = 1.0f / sqrtf(warp_sum(q) / C + eps);
  float* op = out + o * C * inner + i;
  for (int c = lane; c < C; c += 32)
    op[(int64_t)c * inner] = (xp[(int64_t)c * inner] - mean) * rstd * w[c] + b[c];
}

// ------------------------------------------------------------------------------------ a6 bwd
// One CTA per (n, channel).  Re-normalises the raw weights into registers, then walks the saved
// states backwards:  dWn[k,p] += g[p] * x_t[p+d_k];  g_prev[q] = sum_k Wn[k,q-d_k] * g[q-d_k].
// The scatter is done as a gather through a (49 x plane) shared product table so the
// reduction order is fixed (bit-stable gradients).  Finally through Wn = W / (sum W + eps).
template <int MAXT>
__global__ void __launch_bounds__(MAXT)
diffuse_plane_bwd_kernel(const float* __restrict__ grad_out, const float* __restrict__ weight,
                         const float* __restrict__ states, float* __restrict__ grad_x,
                         float* __restrict__ grad_weight, int C, int gh, int gw, int wc, int T,
                         float eps) {
  extern __shared__ float sm[];
  const int pw = gw + 2 * KR, ph = gh + 2 * KR, plane = pw * ph, hw = gh * gw;
  float* xs = sm;               // padded state plane
  float* prod = sm + plane;     // [49][hw] products Wn[k,p]*g[p]
  const int c = blockIdx.x, b = blockIdx.y, p = threadIdx.x;
  const bool live = p < hw;
  const int py = live ? p / gw : 0, px = live ? p - py * gw : 0;
  for (int i = threadIdx.x; i < plane; i += blockDim.x) xs[i] = 0.f;

  float wn[KK], dwn[KK];
  float inv = 0.f, g = 0.f;
  const int cw = (wc == 1) ? 0 : c;
  if (live) {
    const float* wp = weight + ((int64_t)b * wc + cw) * KK * hw + p;
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < KK; ++k) {
      wn[k] = wp[(int64_t)k * hw];
      s += wn[k];
      dwn[k] = 0.f;
    }
    inv = 1.0f / (s + eps);
#pragma unroll
    for (int k = 0; k < KK; ++k) wn[k] *= inv;
    g = grad_out[((int64_t)b * C + c) * hw + p];
  }
  __syncthreads();
  for (int t = T - 1; t >= 0; --t) {
    if (live) {
      xs[(py + KR) * pw + px + KR] = states[(((int64_t)b * (T + 1) + t) * C + c) * hw + p];
#pragma unroll
      for (int k = 0; k < KK; ++k) prod[k * hw + p] = wn[k] * g;
    }
    __syncthreads();
    if (live) {
      float gp = 0.f;
#pragma unroll
      for (int ki = 0; ki < KS; ++ki)
#pragma unroll
        for (int kj = 0; kj < KS; ++kj) {
          dwn[ki * KS + kj] = fmaf(g, xs[(py + ki) * pw + px + kj], dwn[ki * KS + kj]);
          // output pixel (qy,qx) = (py-ki+3, px-kj+3) read this pixel through tap (ki,kj)
          int qy = py - ki + KR, qx = px - kj + KR;
          if ((unsigned)qy < (unsigned)gh && (unsigned)qx < (unsigned)gw)
            gp += prod[(ki * KS + kj) * hw + qy * gw + qx];
        }
      g = gp;
    }
    __syncthreads();
  }
  if (live) {
    grad_x[((int64_t)b * C + c) * hw + p] = g;
    // W_k -> Wn_k = W_k / S:  dW_k = (dWn_k - sum_j dWn_j Wn_j) / S
    float dot = 0.f;
#pragma unroll
    for (int k = 0; k < KK; ++k) dot = fmaf(dwn[k], wn[k], dot);
    float* gwp = grad_weight + ((int64_t)b * wc + cw) * KK * hw + p;
#pragma unroll
    for (int k = 0; k < KK; ++k) {
      float v = (dwn[k] - dot) * inv;
      if (wc == 1) atomicAdd(gwp + (int64_t)k * hw, v);   // shared weights: sum over channels
      else gwp[(int64_t)k * hw] = v;
    }
  }
}

// ------------------------------------------------------------------------------------ small backward ops
// 1x1 conv NCHW backward.  y_out non-null => the forward applied a sigmoid: g <- g * y (1 - y).
// dx: thread per (b, ci, p);  dw/db: one CTA per (input, output) channel pair, fixed-order reduction.
__global__ void conv1x1_nchw_bwd_dx_kernel(const float* __restrict__ g, const float* __restrict__ y_out,
                                           const float* __restrict__ w, float* __restrict__ dx, int Cin,
                                           int Cout, int HW) {
  int b = blockIdx.z, ci = blockIdx.y;
  int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  const float* gp = g + (int64_t)b * Cout * HW + p;
  const float* yp = y_out ? y_out + (int64_t)b * Cout * HW + p : nullptr;
  float acc = 0.f;
  for (int co = 0; co < Cout; ++co) {
    float gv = gp[(int64_t)co * HW];
    if (yp) {
      float yv = yp[(int64_t)co * HW];
      gv *= yv * (1.f - yv);
    }
    acc = fmaf(w[(int64_t)co * Cin + ci], gv, acc);
  }
  dx[((int64_t)b * Cin + ci) * HW + p] = acc;
}

__global__ void __launch_bounds__(256)
conv1x1_nchw_bwd_dw_kernel(const float* __restrict__ g, const float* __restrict__ y_out,
                           const float* __restrict__ x, float* __restrict__ dw, float* __restrict__ db, int B,
                           int Cin, int Cout, int HW) {
  // CTA = one (ci, co) pair (blockIdx.x == 0: bias gradient); fixed-order reduction
  __shared__ float red[8];
  const int co = blockIdx.y, ci = (int)blockIdx.x - 1;
  float acc = 0.f;
  for (int b = 0; b < B; ++b) {
    const float* gp = g + ((int64_t)b * Cout + co) * HW;
    const float* yp = y_out ? y_out + ((int64_t)b * Cout + co) * HW : nullptr;
    const float* xp = ci < 0 ? nullptr : x + ((int64_t)b * Cin + ci) * HW;
    for (int p = threadIdx.x; p < HW; p += 256) {
      float gv = gp[p];
      if (yp) {
        const float yv = yp[p];
        gv *= yv * (1.f - yv);
      }
      acc += xp ? gv * xp[p] : gv;
    }
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i];
    if (ci < 0) { if (db) db[co] = t; }
    else dw[(int64_t)co * Cin + ci] = t;
  }
}

// adjoint of the bilinear resize (gather form, deterministic): one thread per INPUT pixel walks
// the output window that can reference it.
__global__ void resize_bilinear_nchw_bwd_kernel(const float* __restrict__ g, float* __restrict__ dx, int h,
                                                int w, int oh, int ow) {
  int plane = blockIdx.z;
  int ix = blockIdx.x * blockDim.x + threadIdx.x, iy = blockIdx.y * blockDim.y + threadIdx.y;
  if (ix >= w || iy >= h) return;
  const float sy = (float)h / oh, sx = (float)w / ow;
  int oy_lo = (int)floorf((iy - 1 + 0.5f) / sy - 0.5f) - 1, oy_hi = (int)ceilf((iy + 1 + 0.5f) / sy - 0.5f) + 1;
  int ox_lo = (int)floorf((ix - 1 + 0.5f) / sx - 0.5f) - 1, ox_hi = (int)ceilf((ix + 1 + 0.5f) / sx - 0.5f) + 1;
  if (iy == 0) oy_lo = 0;             // clamped source coordinates pile up on the border pixels
  if (ix == 0) ox_lo = 0;
  if (iy == h - 1) oy_hi = oh - 1;
  if (ix == w - 1) ox_hi = ow - 1;
  oy_lo = max(oy_lo, 0); ox_lo = max(ox_lo, 0);
  oy_hi = min(oy_hi, oh - 1); ox_hi = min(ox_hi, ow - 1);
  const float* gp = g + (int64_t)plane * oh * ow;
  float acc = 0.f;
  for (int oy = oy_lo; oy <= oy_hi; ++oy) {
    int y0, y1;
    float ly;
    bilinear_src(oy, sy, h, y0, y1, ly);
    float wy = (y0 == iy ? 1.f - ly : 0.f) + (y1 == iy ? ly : 0.f);
    if (wy == 0.f) continue;
    for (int ox = ox_lo; ox <= ox_hi; ++ox) {
      int x0, x1;
      float lx;
      bilinear_src(ox, sx, w, x0, x1, lx);
      float wx = (x0 == ix ? 1.f - lx : 0.f) + (x1 == ix ? lx : 0.f);
      if (wx != 0.f) acc = fmaf(wy * wx, gp[(int64_t)oy * ow + ox], acc);
    }
  }
  dx[((int64_t)plane * h + iy) * w + ix] = acc;
}

}  // namespace dgtd

using namespace dgtd;

extern "C" {

int dgtd_surface_normals_fwd(const float* depth, float* normals, int B, int H, int W,
                             dgtd_stream_t stream) {
  DGTD_CHECK_ARG(depth && normals && B > 0 && H > 0 && W > 0, "surface_normals: bad args");
  dim3 block(32, 8), grid(cdiv(W, 32), cdiv(H, 8), B);
  surface_normals_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(depth, normals, H, W);
  DGTD_LAUNCH_CHECK("surface_normals");
  return 0;
}

static int plane_threads(int hw) { return ((hw + 31) / 32) * 32; }

int dgtd_diffusion_front_fwd(const float* emb1, const float* depth, const float* reg_w,
                             const float* reg_b, const float* enc_w, const float* enc_b,
                             const float* conv_w, const float* conv_b, float* out_grid,
                             float* save_states, float* save_wn, int B, int H, int W, int G, int C,
                             int T, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(emb1 && depth && reg_w && reg_b && enc_w && enc_b && conv_w && conv_b && out_grid,
                 "diffusion_front: null pointer");
  DGTD_CHECK_ARG(B > 0 && H >= G && W >= G && G > 0 && G * G <= 1024 && C > 0 && T >= 0,
                 "diffusion_front: bad shape B=%d H=%d W=%d G=%d C=%d T=%d", B, H, W, G, C, T);
  DGTD_CHECK_ARG(save_states != nullptr, "diffusion_front: save_states (B,T+1,C,G,G) is required "
                 "(its last slice is the operand of the 1x1 conv)");
  cudaStream_t s = (cudaStream_t)stream;
  const int hw = G * G;
  size_t smem = 2 * (size_t)(G + 6) * (G + 6) * sizeof(float);
  if (hw <= 256)
    diffuse_plane_kernel<true, 256><<<dim3(C, B), plane_threads(hw), smem, s>>>(
        emb1, depth, reg_w, reg_b, enc_w, enc_b, nullptr, nullptr, /*out=*/nullptr, save_states,
        save_wn, C, H, W, G, G, C, T, 1e-5f);
  else
    diffuse_plane_kernel<true, 1024><<<dim3(C, B), plane_threads(hw), smem, s>>>(
        emb1, depth, reg_w, reg_b, enc_w, enc_b, nullptr, nullptr, /*out=*/nullptr, save_states,
        save_wn, C, H, W, G, G, C, T, 1e-5f);
  DGTD_LAUNCH_CHECK("diffusion_front");
  // message_passing.conv (cod.py:1206) over the final state slice states[:, T]
  conv1x1_nchw_kernel<false><<<dim3(cdiv(hw, 128), 3, B), 128, 0, s>>>(
      save_states + (int64_t)T * C * hw, conv_w, conv_b, out_grid, C, 3, hw,
      (int64_t)(T + 1) * C * hw);
  DGTD_LAUNCH_CHECK("diffusion_front.conv");
  return 0;
}

int dgtd_message_passing_fwd(const float* x, const float* weight, float* out, float* save_states,
                             int n, int c, int h, int w, int wc, int T, float eps,
                             dgtd_stream_t stream) {
  DGTD_CHECK_ARG(x && weight && out, "message_passing: null pointer");
  DGTD_CHECK_ARG(n > 0 && c > 0 && h > 0 && w > 0 && T >= 0, "message_passing: bad shape");
  DGTD_CHECK_ARG(wc == 1 || wc == c, "message_passing: weight channels %d must be 1 or %d", wc, c);
  DGTD_CHECK_ARG(h * w <= 1024, "message_passing: plane %dx%d exceeds the on-chip variant "
                 "(h*w <= 1024); use dgtd_message_passing_tiled_fwd", h, w);
  size_t smem = 2 * (size_t)(h + 6) * (w + 6) * sizeof(float);
  if (h * w <= 256)
    diffuse_plane_kernel<false, 256><<<dim3(c, n), plane_threads(h * w), smem, (cudaStream_t)stream>>>(
        nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, x, weight, out, save_states, nullptr,
        c, 0, 0, h, w, wc, T, eps);
  else
    diffuse_plane_kernel<false, 1024><<<dim3(c, n), plane_threads(h * w), smem, (cudaStream_t)stream>>>(
        nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, x, weight, out, save_states, nullptr,
        c, 0, 0, h, w, wc, T, eps);
  DGTD_LAUNCH_CHECK("message_passing");
  return 0;
}

int dgtd_message_passing_bwd(const float* grad_out, const float* weight, const float* states,
                             float* grad_x, float* grad_weight, int n, int c, int h, int w, int wc,
                             int T, float eps, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(grad_out && weight && states && grad_x && grad_weight,
                 "message_passing_bwd: null pointer");
  DGTD_CHECK_ARG(wc == 1 || wc == c, "message_passing_bwd: bad wc");
  DGTD_CHECK_ARG(h * w <= 1024, "message_passing_bwd: plane too large for the on-chip variant");
  cudaStream_t s = (cudaStream_t)stream;
  const int hw = h * w;
  size_t smem = ((size_t)(h + 6) * (w + 6) + (size_t)49 * hw) * sizeof(float);
  DGTD_CHECK_ARG(smem <= 227 * 1024, "message_passing_bwd: plane needs %zu B of shared memory", smem);
  if (wc == 1) {
    cudaError_t e = cudaMemsetAsync(grad_weight, 0, (size_t)n * 49 * hw * sizeof(float), s);
    DGTD_CHECK_ARG(e == cudaSuccess, "message_passing_bwd: memset failed");
  }
  if (hw <= 256) {
    if (smem > 48 * 1024) {
      cudaError_t e = cudaFuncSetAttribute(diffuse_plane_bwd_kernel<256>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      DGTD_CHECK_ARG(e == cudaSuccess, "message_passing_bwd: cannot opt in to %zu B smem", smem);
    }
    diffuse_plane_bwd_kernel<256><<<dim3(c, n), plane_threads(hw), smem, s>>>(
        grad_out, weight, states, grad_x, grad_weight, c, h, w, wc, T, eps);
  } else {
    cudaError_t e = cudaFuncSetAttribute(diffuse_plane_bwd_kernel<1024>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    DGTD_CHECK_ARG(e == cudaSuccess, "message_passing_bwd: cannot opt in to %zu B smem", smem);
    diffuse_plane_bwd_kernel<1024><<<dim3(c, n), plane_threads(hw), smem, s>>>(
        grad_out, weight, states, grad_x, grad_weight, c, h, w, wc, T, eps);
  }
  DGTD_LAUNCH_CHECK("message_passing_bwd");
  return 0;
}

int dgtd_conv1x1_nchw_fwd(const float* x, const float* w, const float* b, float* out, int B,
                          int Cin, int Cout, int HW, int sigmoid, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(x && w && out && B > 0 && Cin > 0 && Cout > 0 && HW > 0, "conv1x1_nchw: bad args");
  DGTD_CHECK_ARG(Cout <= 65535 && B <= 65535, "conv1x1_nchw: grid too large");
  dim3 grid(cdiv(HW, 128), Cout, B);
  cudaStream_t s = (cudaStream_t)stream;
  if (sigmoid)
    conv1x1_nchw_kernel<true><<<grid, 128, 0, s>>>(x, w, b, out, Cin, Cout, HW, (int64_t)Cin * HW);
  else
    conv1x1_nchw_kernel<false><<<grid, 128, 0, s>>>(x, w, b, out, Cin, Cout, HW, (int64_t)Cin * HW);
  DGTD_LAUNCH_CHECK("conv1x1_nchw");
  return 0;
}

int dgtd_conv1x1_nchw_bwd(const float* grad_out, const float* y_out, const float* x, const float* w,
                          float* grad_x, float* grad_w, float* grad_b, int B, int Cin, int Cout, int HW,
                          dgtd_stream_t stream) {
  DGTD_CHECK_ARG(grad_out && x && w && B > 0 && Cin > 0 && Cout > 0 && HW > 0, "conv1x1_nchw_bwd: bad args");
  DGTD_CHECK_ARG(Cin <= 65535 && B <= 65535 && Cout <= 65535, "conv1x1_nchw_bwd: grid too large");
  cudaStream_t s = (cudaStream_t)stream;
  if (grad_x) {
    conv1x1_nchw_bwd_dx_kernel<<<dim3(cdiv(HW, 128), Cin, B), 128, 0, s>>>(grad_out, y_out, w, grad_x, Cin, Cout, HW);
    DGTD_LAUNCH_CHECK("conv1x1_nchw_bwd.dx");
  }
  if (grad_w) {
    conv1x1_nchw_bwd_dw_kernel<<<dim3(Cin + 1, Cout), 256, 0, s>>>(grad_out, y_out, x, grad_w, grad_b, B, Cin, Cout, HW);
    DGTD_LAUNCH_CHECK("conv1x1_nchw_bwd.dw");
  }
  return 0;
}

int dgtd_resize_bilinear_nchw_bwd(const float* grad_out, float* grad_x, int planes, int h, int w, int oh,
                                  int ow, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(grad_out && grad_x && planes > 0 && h > 0 && w > 0 && oh > 0 && ow > 0, "resize_bwd: bad args");
  DGTD_CHECK_ARG(planes <= 65535, "resize_bwd: too many planes");
  dim3 block(16, 8), grid(cdiv(w, 16), cdiv(h, 8), planes);
  resize_bilinear_nchw_bwd_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(grad_out, grad_x, h, w, oh, ow);
  DGTD_LAUNCH_CHECK("resize_bilinear_nchw_bwd");
  return 0;
}

int dgtd_resize_nchw_fwd(const float* x, float* out, int planes, int h, int w, int oh, int ow,
                         int bilinear, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(x && out && planes > 0 && h > 0 && w > 0 && oh > 0 && ow > 0, "resize_nchw: bad args");
  DGTD_CHECK_ARG(planes <= 65535, "resize_nchw: too many planes");
  dim3 block(32, 8), grid(cdiv(ow, 32), cdiv(oh, 8), planes);
  resize_nchw_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(x, out, h, w, oh, ow, bilinear);
  DGTD_LAUNCH_CHECK("resize_nchw");
  return 0;
}

int dgtd_resize_sigmoid_sized_fwd(const float* x, float* out, const int32_t* sizes, int B, int h, int w, int Hmax,
                                  int Wmax, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(x && out && sizes && B > 0 && h > 0 && w > 0 && Hmax > 1 && Wmax > 1, "resize_sigmoid_sized: bad args");
  DGTD_CHECK_ARG(B <= 65535, "resize_sigmoid_sized: too many planes");
  dim3 block(32, 8), grid(cdiv(Wmax, 32), cdiv(Hmax, 8), B);
  resize_sigmoid_sized_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(x, out, sizes, h, w, Hmax, Wmax);
  DGTD_LAUNCH_CHECK("resize_sigmoid_sized");
  return 0;
}

int dgtd_layer_norm_fwd(const float* x, const float* w, const float* b, float* out, int64_t outer,
                        int C, int64_t inner, float eps, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(x && w && b && out && outer > 0 && C > 0 && inner > 0, "layer_norm: bad args");
  int64_t rows = outer * inner;
  layer_norm_kernel<<<cdiv(rows, 8), 256, 0, (cudaStream_t)stream>>>(x, w, b, out, rows, C, inner, eps);
  DGTD_LAUNCH_CHECK("layer_norm");
  return 0;
}

}  // extern "C"
