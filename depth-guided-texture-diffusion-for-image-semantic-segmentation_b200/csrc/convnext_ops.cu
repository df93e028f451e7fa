// CUDA-core pieces of ShapePropEncoder (cod.py:1119-1177): stem (a7), LayerNorm + 2x2 patch
// gather (a7), depthwise 7x7 + channels-last LayerNorm (a8), fusion head tail (a9).
// Activations are NHWC; the residual stream is fp32.
#include "common.cuh"

namespace dgtd {

// ------------------------------------------------------------------------------------ a7 stem
// (bilinear-up(grid) + image) -> conv 4x4 stride 4 (3 -> Cout) -> LayerNorm over channels.
// CTA = 16 consecutive output pixels of one output row; thread = output channel.
constexpr int STEM_PX = 16;

constexpr int STEM_TILES_PER_CTA = 12;

__global__ void __launch_bounds__(256)
stem_kernel(const float* __restrict__ image, const float* __restrict__ grid, int G,
            const float* __restrict__ w, const float* __restrict__ bias,
            const float* __restrict__ ln_w, const float* __restrict__ ln_b, float* __restrict__ out,
            int H, int W, int oh, int ow, int Cout, float eps, int total_tiles) {
  extern __shared__ float sm[];
  float* in = sm;                    // [STEM_PX][48]
  float* ys = sm + STEM_PX * 48;     // [STEM_PX][Cout]
  const int tiles_x = (ow + STEM_PX - 1) / STEM_PX;
  const int c = threadIdx.x;
  float wr[48];
#pragma unroll
  for (int k = 0; k < 48; ++k) wr[k] = w[(int64_t)c * 48 + k];
  const float bc = bias[c];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;

  for (int it = 0; it < STEM_TILES_PER_CTA; ++it) {
    int tile = blockIdx.x * STEM_TILES_PER_CTA + it;
    if (tile >= total_tiles) break;               // block-uniform
    const int tx = tile % tiles_x;
    tile /= tiles_x;
    const int oy = tile % oh, b = tile / oh;
    const int ox0 = tx * STEM_PX;
    // gather the 4 x (4*STEM_PX) x 3 input patch, adding the up-sampled diffusion result
    for (int e = threadIdx.x; e < 3 * 4 * 4 * STEM_PX; e += blockDim.x) {
      int ci = e / (16 * STEM_PX), r = e - ci * 16 * STEM_PX;
      int ky = r / (4 * STEM_PX), j = r - ky * 4 * STEM_PX;
      int px = j >> 2, kx = j & 3;
      int iy = oy * 4 + ky, ix = ox0 * 4 + j;
      float v = 0.f;
      if (ox0 + px < ow) {
        v = image[(((int64_t)b * 3 + ci) * H + iy) * W + ix];
        if (grid) {
          int y0, y1, x0, x1;
          float ly, lx;
          bilinear_src(iy, (float)G / H, G, y0, y1, ly);
          bilinear_src(ix, (float)G / W, G, x0, x1, lx);
          const float* g = grid + ((int64_t)b * 3 + ci) * G * G;
          v += (1.f - ly) * ((1.f - lx) * g[y0 * G + x0] + lx * g[y0 * G + x1]) +
               ly * ((1.f - lx) * g[y1 * G + x0] + lx * g[y1 * G + x1]);
        }
      }
      in[px * 48 + ci * 16 + ky * 4 + kx] = v;
    }
    __syncthreads();
#pragma unroll 4
    for (int px = 0; px < STEM_PX; ++px) {
      float acc = bc;
#pragma unroll
      for (int k4 = 0; k4 < 12; ++k4) {
        float4 v = *reinterpret_cast<const float4*>(&in[px * 48 + k4 * 4]);
        acc = fmaf(wr[k4 * 4 + 0], v.x, acc);
        acc = fmaf(wr[k4 * 4 + 1], v.y, acc);
        acc = fmaf(wr[k4 * 4 + 2], v.z, acc);
        acc = fmaf(wr[k4 * 4 + 3], v.w, acc);
      }
      ys[px * Cout + c] = acc;
    }
    __syncthreads();
    // LayerNorm(channels_first) == per-pixel LN over channels (cod.py:1045-1048)
    for (int px = wid; px < STEM_PX; px += nw) {
      if (ox0 + px >= ow) continue;
      float s = 0.f;
      for (int cc = lane; cc < Cout; cc += 32) s += ys[px * Cout + cc];
      float mean = warp_sum(s) / Cout;
      float q = 0.f;
      for (int cc = lane; cc < Cout; cc += 32) {
        float d = ys[px * Cout + cc] - mean;
        q = fmaf(d, d, q);
      }
      float rstd = 1.0f / sqrtf(warp_sum(q) / Cout + eps);
      float* o = out + (((int64_t)b * oh + oy) * ow + ox0 + px) * Cout;
      for (int cc = lane; cc < Cout; cc += 32)
        o[cc] = (ys[px * Cout + cc] - mean) * rstd * ln_w[cc] + ln_b[cc];
    }
    __syncthreads();   // ys / in are rewritten by the next tile
  }
}

// ------------------------------------------------------------------------------------ a7 downsample
// LayerNorm(channels_first) then scatter into 2x2 patch rows: one warp per input pixel.
template <typename OT, int VPL>  // VPL = C / 32 values per lane
__global__ void __launch_bounds__(256)
ln_patchify_kernel(const float* __restrict__ x, const float* __restrict__ ln_w,
                   const float* __restrict__ ln_b, OT* __restrict__ out, int B, int h, int w, int C,
                   float eps) {
  const int h2 = h >> 1, w2 = w >> 1;
  int64_t pix = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  int64_t total = (int64_t)B * h2 * 2 * w2 * 2;
  if (pix >= total) return;
  const int lane = threadIdx.x & 31;
  int xx = (int)(pix % (w2 * 2));
  int64_t t = pix / (w2 * 2);
  int yy = (int)(t % (h2 * 2));
  int b = (int)(t / (h2 * 2));
  const float* p = x + (((int64_t)b * h + yy) * w + xx) * C;
  float v[VPL];
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < VPL; ++j) {
    v[j] = p[lane + 32 * j];
    s += v[j];
  }
  float mean = warp_sum(s) / C;
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < VPL; ++j) {
    float d = v[j] - mean;
    q = fmaf(d, d, q);
  }
  float rstd = 1.0f / sqrtf(warp_sum(q) / C + eps);
  OT* o = out + (((int64_t)b * h2 + (yy >> 1)) * w2 + (xx >> 1)) * (4 * (int64_t)C) +
          (int64_t)((yy & 1) * 2 + (xx & 1)) * C;
#pragma unroll
  for (int j = 0; j < VPL; ++j) {
    int cc = lane + 32 * j;
    o[cc] = from_float<OT>((v[j] - mean) * rstd * ln_w[cc] + ln_b[cc]);
  }
}

// The same operator for C = 128 * V4 with 16-byte accesses: a warp owns R consecutive pixels in PATCH-MAJOR order
// (pixel index = ((b * h2 + y2) * w2 + x2) * 4 + 2 * (y & 1) + (x & 1), which is also its output row), so that its
// R * V4 = 4 loads per lane are in flight together and its stores cover R * C contiguous outputs.
template <typename OT, int V4, int R>
__global__ void __launch_bounds__(256)
ln_patchify_v4_kernel(const float* __restrict__ x, const float* __restrict__ ln_w, const float* __restrict__ ln_b,
                      OT* __restrict__ out, int B, int h, int w, int C, float eps) {
  const int h2 = h >> 1, w2 = w >> 1;
  const int64_t total = (int64_t)B * h2 * w2 * 4;
  const int64_t pix0 = ((int64_t)blockIdx.x * 8 + (threadIdx.x >> 5)) * R;
  if (pix0 >= total) return;
  const int lane = threadIdx.x & 31;
  float4 v[R][V4];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int64_t pix = pix0 + r;
    const int r4 = (int)(pix & 3);
    int64_t t = pix >> 2;
    const int x2 = (int)(t % w2);
    t /= w2;
    const int y2 = (int)(t % h2), b = (int)(t / h2);
    const float* p = x + (((int64_t)b * h + 2 * y2 + (r4 >> 1)) * w + 2 * x2 + (r4 & 1)) * C;
#pragma unroll
    for (int j = 0; j < V4; ++j)
      v[r][j] = pix < total ? __ldg(reinterpret_cast<const float4*>(p + (j * 32 + lane) * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  float4 g[V4], be[V4];
#pragma unroll
  for (int j = 0; j < V4; ++j) {
    g[j] = __ldg(reinterpret_cast<const float4*>(ln_w + (j * 32 + lane) * 4));
    be[j] = __ldg(reinterpret_cast<const float4*>(ln_b + (j * 32 + lane) * 4));
  }
  const float inv_c = 1.0f / C;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < V4; ++j) s += (v[r][j].x + v[r][j].y) + (v[r][j].z + v[r][j].w);
    const float mean = warp_sum(s) * inv_c;
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < V4; ++j) {
      const float a = v[r][j].x - mean, bb = v[r][j].y - mean, c = v[r][j].z - mean, d = v[r][j].w - mean;
      q += (a * a + bb * bb) + (c * c + d * d);
    }
    const float rstd = 1.0f / sqrtf(warp_sum(q) * inv_c + eps);
    if (pix0 + r < total) {
      OT* o = out + (pix0 + r) * C;
#pragma unroll
      for (int j = 0; j < V4; ++j)
        store4(o + (j * 32 + lane) * 4, (v[r][j].x - mean) * rstd * g[j].x + be[j].x, (v[r][j].y - mean) * rstd * g[j].y + be[j].y,
               (v[r][j].z - mean) * rstd * g[j].z + be[j].z, (v[r][j].w - mean) * rstd * g[j].w + be[j].w);
    }
  }
}

// ------------------------------------------------------------------------------------ a8 dwconv + LN
// CTA = TH x 8 output pixels x all C channels.  thread = channel (coalesced NHWC), 49 taps in
// registers, TH x 8 accumulators, every input row loaded once and reused by up to TH output
// rows and 7 taps (FMA : load = 16 : 1).  Results go to shared memory, then one warp per pixel
// does the two-pass LayerNorm over C (cod.py:1106-1108).
template <typename OT, int TH>
__global__ void __launch_bounds__(256, 2)
dwconv7_ln_kernel(const float* __restrict__ x, const float* __restrict__ dw_w,
                  const float* __restrict__ dw_b, const float* __restrict__ ln_w,
                  const float* __restrict__ ln_b, OT* __restrict__ out, int h, int w, int C,
                  float eps) {
  constexpr int TW = 8, NPX = TH * TW;
  extern __shared__ float ys[];  // [NPX][C]
  const int tiles_x = (w + TW - 1) / TW, tiles_y = (h + TH - 1) / TH;
  int bid = blockIdx.x;
  const int tx = bid % tiles_x;
  bid /= tiles_x;
  const int ty = bid % tiles_y, b = bid / tiles_y;
  const int x0 = tx * TW, y0 = ty * TH;
  const float* xb = x + (int64_t)b * h * w * C;

  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float wr[49];
#pragma unroll
    for (int k = 0; k < 49; ++k) wr[k] = dw_w[(int64_t)c * 49 + k];
    float acc[TH][TW];
    const float bc = dw_b[c];
#pragma unroll
    for (int i = 0; i < TH; ++i)
#pragma unroll
      for (int j = 0; j < TW; ++j) acc[i][j] = bc;
#pragma unroll
    for (int iy = 0; iy < TH + 6; ++iy) {
      const int gy = y0 + iy - 3;
      if (gy < 0 || gy >= h) continue;   // zero padding row (block-uniform branch)
      float in[TW + 6];
      const float* row = xb + (int64_t)gy * w * C + c;
#pragma unroll
      for (int j = 0; j < TW + 6; ++j) {
        int gx = x0 + j - 3;
        in[j] = (gx >= 0 && gx < w) ? row[(int64_t)gx * C] : 0.f;
      }
#pragma unroll
      for (int oy = 0; oy < TH; ++oy) {
        const int ky = iy - oy;
        if (ky < 0 || ky >= 7) continue;
#pragma unroll
        for (int ox = 0; ox < TW; ++ox)
#pragma unroll
          for (int kx = 0; kx < 7; ++kx) acc[oy][ox] = fmaf(wr[ky * 7 + kx], in[ox + kx], acc[oy][ox]);
      }
      asm volatile("" ::: "memory");  // keep only one input row live (bounds register pressure)
    }
#pragma unroll
    for (int i = 0; i < TH; ++i)
#pragma unroll
      for (int j = 0; j < TW; ++j) ys[(i * TW + j) * C + c] = acc[i][j];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int px = wid; px < NPX; px += nw) {
    const int oy = y0 + px / TW, ox = x0 + px % TW;
    if (oy >= h || ox >= w) continue;
    const float* yp = ys + px * C;
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s += yp[c];
    const float mean = warp_sum(s) / C;
    float q = 0.f;
    for (int c = lane; c < C; c += 32) {
      float d = yp[c] - mean;
      q = fmaf(d, d, q);
    }
    const float rstd = 1.0f / sqrtf(warp_sum(q) / C + eps);
    OT* o = out + (((int64_t)b * h + oy) * w + ox) * C;
    for (int c = lane; c < C; c += 32)
      o[c] = from_float<OT>((yp[c] - mean) * rstd * ln_w[c] + ln_b[c]);
  }
}

// ------------------------------------------------------------------------------------ a9 head tail
// ShapePropEncoder head with the 1x1 fusion conv already applied per level (it commutes with the bilinear up-sample
// and is folded into the head projections on the host): out[p] = bias + sum_lv bilinear_up(z_lv)[p].
// thread = (pixel, 4 channels); quads beyond C only zero-fill the padded bf16 copy.
__global__ void __launch_bounds__(256)
fusion_sum_kernel(const float* __restrict__ z0, const float* __restrict__ z1, const float* __restrict__ z2,
                  const float* __restrict__ z3, int h0, int w0, int h1, int w1, int h2, int w2, int h3, int w3,
                  const float* __restrict__ bias, float* __restrict__ out_nhwc, float* __restrict__ out_nchw,
                  __nv_bfloat16* __restrict__ out_pad, int C, int Cpad, int quads, int64_t total) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int cq = (int)(i % quads);
  const int64_t p = i / quads;
  const int c = cq * 4;
  if (c >= C) {   // padding channels of the bf16 copy
    if (out_pad && c < Cpad) store4(out_pad + p * Cpad + c, 0.f, 0.f, 0.f, 0.f);
    return;
  }
  const int ox = (int)(p % w0);
  const int64_t t = p / w0;
  const int oy = (int)(t % h0), b = (int)(t / h0);
  float4 acc = load4(bias + c);
  {
    const float4 v = load4(z0 + p * C + c);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
#pragma unroll
  for (int lv = 1; lv < 4; ++lv) {
    const float* src = lv == 1 ? z1 : lv == 2 ? z2 : z3;
    const int hh = lv == 1 ? h1 : lv == 2 ? h2 : h3;
    const int ww = lv == 1 ? w1 : lv == 2 ? w2 : w3;
    int y0, y1, x0, x1;
    float ly, lx;
    bilinear_src(oy, (float)hh / h0, hh, y0, y1, ly);
    bilinear_src(ox, (float)ww / w0, ww, x0, x1, lx);
    const float* sb = src + (int64_t)b * hh * ww * C + c;
    const float4 a = load4(sb + ((int64_t)y0 * ww + x0) * C), bq = load4(sb + ((int64_t)y0 * ww + x1) * C);
    const float4 cc = load4(sb + ((int64_t)y1 * ww + x0) * C), d = load4(sb + ((int64_t)y1 * ww + x1) * C);
    const float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
    acc.x += w00 * a.x + w01 * bq.x + w10 * cc.x + w11 * d.x;
    acc.y += w00 * a.y + w01 * bq.y + w10 * cc.y + w11 * d.y;
    acc.z += w00 * a.z + w01 * bq.z + w10 * cc.z + w11 * d.z;
    acc.w += w00 * a.w + w01 * bq.w + w10 * cc.w + w11 * d.w;
  }
  if (out_nhwc) store4(out_nhwc + p * C + c, acc.x, acc.y, acc.z, acc.w);
  if (out_pad) store4(out_pad + p * Cpad + c, acc.x, acc.y, acc.z, acc.w);
  if (out_nchw) {
    const int64_t hw = (int64_t)h0 * w0, r = p - (int64_t)b * hw;
    float* o = out_nchw + ((int64_t)b * C + c) * hw + r;
    o[0] = acc.x; o[hw] = acc.y; o[2 * hw] = acc.z; o[3 * hw] = acc.w;
  }
}

// ------------------------------------------------------------------------------------ a11 resize
template <typename IT, typename OT>
__global__ void resize_nhwc_kernel(const IT* __restrict__ x, OT* __restrict__ out, int h, int w, int C,
                                   int oh, int ow, int64_t total) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c4 = C >> 2;
  int cq = (int)(i % c4);
  int64_t t = i / c4;
  int ox = (int)(t % ow);
  t /= ow;
  int oy = (int)(t % oh), b = (int)(t / oh);
  int y0, y1, x0, x1;
  float ly, lx;
  bilinear_src(oy, (float)h / oh, h, y0, y1, ly);
  bilinear_src(ox, (float)w / ow, w, x0, x1, lx);
  const IT* xb = x + (int64_t)b * h * w * C + cq * 4;
  float4 a = load4(xb + ((int64_t)y0 * w + x0) * C), bq = load4(xb + ((int64_t)y0 * w + x1) * C);
  float4 cc = load4(xb + ((int64_t)y1 * w + x0) * C), d = load4(xb + ((int64_t)y1 * w + x1) * C);
  float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
  store4(out + (((int64_t)b * oh + oy) * ow + ox) * C + cq * 4,
         w00 * a.x + w01 * bq.x + w10 * cc.x + w11 * d.x, w00 * a.y + w01 * bq.y + w10 * cc.y + w11 * d.y,
         w00 * a.z + w01 * bq.z + w10 * cc.z + w11 * d.z, w00 * a.w + w01 * bq.w + w10 * cc.w + w11 * d.w);
}

}  // namespace dgtd

namespace dgtd {
int ln_rows_any(const float* y, const float* ln_w, const float* ln_b, void* out, int out_dtype, int64_t rows, int C,
                float eps, cudaStream_t s);
int dwconv7_ln_tma(const float* x, const float* wT, const float* dw_b, const float* ln_w, const float* ln_b,
                   float* ws, void* out, int out_dtype, int B, int h, int w, int C, float eps, cudaStream_t s);
int dwconv7_stats_tma(const float* x, const float* wT, const float* dw_b, __nv_bfloat16* y, float2* stats, int B, int h,
                      int w, int C, float eps, cudaStream_t s);
}
using namespace dgtd;

extern "C" {

int dgtd_stem_fwd(const float* image, const float* grid, int G, const float* w, const float* b,
                  const float* ln_w, const float* ln_b, float* out, int B, int H, int W, int Cout,
                  float eps, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(image && w && b && ln_w && ln_b && out, "stem: null pointer");
  DGTD_CHECK_ARG(B > 0 && H >= 4 && W >= 4 && Cout >= 32 && Cout <= 256 && Cout % 32 == 0,
                 "stem: bad shape B=%d H=%d W=%d Cout=%d", B, H, W, Cout);
  DGTD_CHECK_ARG(!grid || G > 0, "stem: bad grid size");
  const int oh = H / 4, ow = W / 4;
  size_t smem = (size_t)(STEM_PX * 48 + STEM_PX * Cout) * sizeof(float);
  const int total_tiles = cdiv(ow, STEM_PX) * oh * B;
  stem_kernel<<<cdiv(total_tiles, STEM_TILES_PER_CTA), Cout, smem, (cudaStream_t)stream>>>(
      image, grid, G, w, b, ln_w, ln_b, out, H, W, oh, ow, Cout, eps, total_tiles);
  DGTD_LAUNCH_CHECK("stem");
  return 0;
}

}  // extern "C"

template <typename OT>
static int ln_patchify_dispatch(const float* x, const float* ln_w, const float* ln_b, OT* out, int B,
                                int h, int w, int C, float eps, cudaStream_t s) {
  int64_t pix = (int64_t)B * (h / 2) * 2 * (w / 2) * 2;
  if (C % 128 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 &&
      (reinterpret_cast<uintptr_t>(ln_w) & 15) == 0 && (reinterpret_cast<uintptr_t>(ln_b) & 15) == 0) {
    switch (C / 128) {   // pixels per block = 8 warps x R
      case 1: ln_patchify_v4_kernel<OT, 1, 4><<<cdiv(pix, 32), 256, 0, s>>>(x, ln_w, ln_b, out, B, h, w, C, eps); return 0;
      case 2: ln_patchify_v4_kernel<OT, 2, 2><<<cdiv(pix, 16), 256, 0, s>>>(x, ln_w, ln_b, out, B, h, w, C, eps); return 0;
      case 4: ln_patchify_v4_kernel<OT, 4, 1><<<cdiv(pix, 8), 256, 0, s>>>(x, ln_w, ln_b, out, B, h, w, C, eps); return 0;
      case 8: ln_patchify_v4_kernel<OT, 8, 1><<<cdiv(pix, 8), 256, 0, s>>>(x, ln_w, ln_b, out, B, h, w, C, eps); return 0;
      default: break;
    }
  }
  int blocks = cdiv(pix, 8);
  switch (C / 32) {
    case 1: ln_patchify_kernel<OT, 1><<<blocks, 256, 0, s>>>(x, ln_w, ln_b, out, B, h, w, C, eps); break;
    case 2: ln_patchify_kernel<OT, 2><<<blocks, 256, 0, s>>>(x, ln_w, ln_b, out, B, h, w, C, eps); break;
    case 4: ln_patchify_kernel<OT, 4><<<blocks, 256, 0, s>>>(x, ln_w, ln_b, out, B, h, w, C, eps); break;
    case 8: ln_patchify_kernel<OT, 8><<<blocks, 256, 0, s>>>(x, ln_w, ln_b, out, B, h, w, C, eps); break;
    case 16: ln_patchify_kernel<OT, 16><<<blocks, 256, 0, s>>>(x, ln_w, ln_b, out, B, h, w, C, eps); break;
    case 32: ln_patchify_kernel<OT, 32><<<blocks, 256, 0, s>>>(x, ln_w, ln_b, out, B, h, w, C, eps); break;
    default:
      set_error("ln_patchify: C=%d must be 32*{1,2,4,8,16,32}", C);
      return -1;
  }
  return 0;
}

extern "C" int dgtd_ln_patchify_fwd(const float* x, const float* ln_w, const float* ln_b, void* out,
                         int out_dtype, int B, int h, int w, int C, float eps,
                         dgtd_stream_t stream) {
  DGTD_CHECK_ARG(x && ln_w && ln_b && out && B > 0 && h >= 2 && w >= 2 && C % 32 == 0,
                 "ln_patchify: bad args");
  int rc = out_dtype == DGTD_BF16
               ? ln_patchify_dispatch(x, ln_w, ln_b, (__nv_bfloat16*)out, B, h, w, C, eps, (cudaStream_t)stream)
               : ln_patchify_dispatch(x, ln_w, ln_b, (float*)out, B, h, w, C, eps, (cudaStream_t)stream);
  if (rc) return rc;
  DGTD_LAUNCH_CHECK("ln_patchify");
  return 0;
}

template <typename OT>
static int dwconv_launch(const float* x, const float* dw_w, const float* dw_b, const float* ln_w,
                         const float* ln_b, OT* out, int B, int h, int w, int C, float eps,
                         cudaStream_t s) {
  constexpr int TH = 4;
  size_t smem = (size_t)TH * 8 * C * sizeof(float);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(dwconv7_ln_kernel<OT, TH>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      set_error("dwconv7_ln: cannot opt in to %zu B smem: %s", smem, cudaGetErrorString(e));
      return -2;
    }
  }
  int threads = C < 256 ? C : 256;
  int64_t blocks = (int64_t)B * cdiv(h, TH) * cdiv(w, 8);
  dwconv7_ln_kernel<OT, TH><<<(unsigned)blocks, threads, smem, s>>>(x, dw_w, dw_b, ln_w, ln_b, out, h,
                                                                    w, C, eps);
  return 0;
}

extern "C" {

int dgtd_dwconv7_ln_fwd(const float* x, const float* dw_w, const float* dw_b, const float* ln_w,
                        const float* ln_b, void* out, int out_dtype, int B, int h, int w, int C,
                        float eps, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(x && dw_w && dw_b && ln_w && ln_b && out, "dwconv7_ln: null pointer");
  DGTD_CHECK_ARG(B > 0 && h > 0 && w > 0 && C >= 32 && C % 32 == 0 && C <= 1024,
                 "dwconv7_ln: bad shape B=%d h=%d w=%d C=%d", B, h, w, C);
  int rc = out_dtype == DGTD_BF16
               ? dwconv_launch(x, dw_w, dw_b, ln_w, ln_b, (__nv_bfloat16*)out, B, h, w, C, eps, (cudaStream_t)stream)
               : dwconv_launch(x, dw_w, dw_b, ln_w, ln_b, (float*)out, B, h, w, C, eps, (cudaStream_t)stream);
  if (rc) return rc;
  DGTD_LAUNCH_CHECK("dwconv7_ln");
  return 0;
}

int dgtd_dwconv7_ln_tma_fwd(const float* x, const float* dw_wT, const float* dw_b, const float* ln_w,
                            const float* ln_b, float* ws, void* out, int out_dtype, int B, int h, int w,
                            int C, float eps, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(x && dw_wT && dw_b && ln_w && ln_b && ws && out, "dwconv7_ln_tma: null pointer");
  DGTD_CHECK_ARG(B > 0 && h > 0 && w > 0 && C >= 128 && C % 128 == 0 && C <= 1024,
                 "dwconv7_ln_tma: bad shape B=%d h=%d w=%d C=%d (C must be a multiple of 128)", B, h, w, C);
  int rc = dwconv7_ln_tma(x, dw_wT, dw_b, ln_w, ln_b, ws, out, out_dtype, B, h, w, C, eps, (cudaStream_t)stream);
  if (rc > 0) {
    set_error("dwconv7_ln_tma: shape not supported by the TMA variant");
    return -1;
  }
  if (rc) return rc;
  DGTD_LAUNCH_CHECK("dwconv7_ln_tma.ln");
  return 0;
}

int dgtd_dwconv7_stats_tma_fwd(const float* x, const float* dw_wT, const float* dw_b, void* y, float* stats, int B, int h,
                               int w, int C, float eps, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(x && dw_wT && dw_b && y && stats, "dwconv7_stats_tma: null pointer");
  DGTD_CHECK_ARG(B > 0 && h > 0 && w > 0 && C >= 128 && C % 128 == 0 && C <= 1024,
                 "dwconv7_stats_tma: bad shape B=%d h=%d w=%d C=%d (C must be a multiple of 128)", B, h, w, C);
  DGTD_CHECK_ARG((reinterpret_cast<uintptr_t>(stats) & 7) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0,
                 "dwconv7_stats_tma: y must be 16-byte, stats 8-byte aligned");
  int rc = dwconv7_stats_tma(x, dw_wT, dw_b, (__nv_bfloat16*)y, (float2*)stats, B, h, w, C, eps, (cudaStream_t)stream);
  if (rc > 0) {
    set_error("dwconv7_stats_tma: shape not supported by the TMA variant");
    return -1;
  }
  return rc;
}

int dgtd_ln_rows_fwd(const float* y, const float* ln_w, const float* ln_b, void* out, int out_dtype, int64_t rows,
                     int C, float eps, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(y && ln_w && ln_b && out && rows > 0 && C % 128 == 0 && C <= 1024, "ln_rows: bad args");
  int rc = ln_rows_any(y, ln_w, ln_b, out, out_dtype, rows, C, eps, (cudaStream_t)stream);
  if (rc) return rc;
  DGTD_LAUNCH_CHECK("ln_rows");
  return 0;
}

int dgtd_fusion_sum_fwd(const float* z0, const float* z1, const float* z2, const float* z3, const int* hw,
                        const float* bias, float* out_nhwc, float* out_nchw, void* out_pad, int Cpad, int B, int C,
                        dgtd_stream_t stream) {
  DGTD_CHECK_ARG(z0 && z1 && z2 && z3 && hw && bias, "fusion_sum: null pointer");
  DGTD_CHECK_ARG(C > 0 && C % 4 == 0, "fusion_sum: C must be a multiple of 4");
  DGTD_CHECK_ARG(out_nhwc || out_nchw || out_pad, "fusion_sum: no output requested");
  DGTD_CHECK_ARG(!out_pad || (Cpad >= C && Cpad % 4 == 0), "fusion_sum: Cpad must be a multiple of 4 and >= C");
  const int quads = (out_pad && Cpad > C ? Cpad : C) / 4;
  const int64_t total = (int64_t)B * hw[0] * hw[1] * quads;
  fusion_sum_kernel<<<(unsigned)cdiv(total, (int64_t)256), 256, 0, (cudaStream_t)stream>>>(
      z0, z1, z2, z3, hw[0], hw[1], hw[2], hw[3], hw[4], hw[5], hw[6], hw[7], bias, out_nhwc, out_nchw,
      (__nv_bfloat16*)out_pad, C, Cpad, quads, total);
  DGTD_LAUNCH_CHECK("fusion_sum");
  return 0;
}

int dgtd_resize_nhwc_fwd(const void* x, void* out, int B, int h, int w, int C, int oh, int ow,
                         int dtype_in, int dtype_out, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(x && out && B > 0 && h > 0 && w > 0 && oh > 0 && ow > 0 && C % 4 == 0,
                 "resize_nhwc: bad args (C must be a multiple of 4)");
  int64_t total = (int64_t)B * oh * ow * (C / 4);
  cudaStream_t s = (cudaStream_t)stream;
  int blocks = cdiv(total, 256);
  if (dtype_in == DGTD_F32 && dtype_out == DGTD_F32)
    resize_nhwc_kernel<<<blocks, 256, 0, s>>>((const float*)x, (float*)out, h, w, C, oh, ow, total);
  else if (dtype_in == DGTD_BF16 && dtype_out == DGTD_BF16)
    resize_nhwc_kernel<<<blocks, 256, 0, s>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)out, h, w, C, oh, ow, total);
  else if (dtype_in == DGTD_BF16 && dtype_out == DGTD_F32)
    resize_nhwc_kernel<<<blocks, 256, 0, s>>>((const __nv_bfloat16*)x, (float*)out, h, w, C, oh, ow, total);
  else
    resize_nhwc_kernel<<<blocks, 256, 0, s>>>((const float*)x, (__nv_bfloat16*)out, h, w, C, oh, ow, total);
  DGTD_LAUNCH_CHECK("resize_nhwc");
  return 0;
}

}  // extern "C"
