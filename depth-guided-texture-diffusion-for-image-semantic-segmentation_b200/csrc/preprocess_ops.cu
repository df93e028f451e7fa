// Preprocessing of decoded RGB-D images on the GPU, bit-identical to the datasets' host transforms (SURVEY §2 row 11):
// PIL 12.2's bilinear Image.resize of an 8-bit image, convert('L') for a colour depth rendering, torchvision's
// ToTensor and Normalize.  DESIGN §14 states the arithmetic and how it was established; oracle/preprocess_ref.py
// restates it in numpy.
//
// Input: one packed uint8 buffer.  At its head B descriptors of kDescFields int64 (RGB byte offset, H, W, depth byte
// offset, H', W', depth channels), then every image's RGB (HWC) and depth planes back to back, no padding.
//
// Launches, all on the caller's stream, none per image:
//   plan   one block: validates the descriptors, carves the workspace per image (a serial prefix over 256 chunks),
//          picks each plane's pass order and fills the 4 x 256 output lookup;
//   coef   (B, 4) blocks: PIL's fixed-point coefficient tables, per image, for the RGB and depth axes;
//   pass1  (tiles, B, 2): the first resampling pass of every RGB and depth plane into a uint8 intermediate;
//   pass2  (tiles, B, 2): the second pass, written as fp32 NCHW through the lookup.
// A scale-1 pass has weights (2^22, 0) and reproduces its input, so running both passes where PIL skips an axis
// gives PIL's bits with one code path.  Integer arithmetic after the coefficients, no atomics: an image's output does
// not depend on the batch it is in.
#include <math.h>

#include "common.cuh"

namespace dgtd {
namespace {

constexpr int kPrecBits = 22;                  // PIL PRECISION_BITS = 32 - 8 - 2
constexpr int kDescFields = 7;
constexpr int kMaxSide = 65535;
constexpr int kPlanThreads = 256;
constexpr int kTileW = 64, kTileH = 16, kBlockRows = 4;   // pass block: 64 x 4 threads, 4 rows each

struct Plan {
  int64_t src[2];      // byte offsets in the packed buffer: RGB, depth
  int64_t coef[4];     // byte offsets in ws of the tables: RGB x, RGB y, depth x, depth y
  int64_t inter[2];    // byte offsets in ws of the intermediates: RGB (3 planes), depth (1 plane)
  int32_t h[2], w[2];  // source sizes: RGB, depth
  int32_t ks[4];       // taps per output index of each table
  int32_t ch;          // depth channels (1, or 3 = converted to 'L' on read)
  int32_t vfirst[2];   // vertical pass first: RGB, depth
  int32_t valid;
};

struct Norm {
  float mean[3], std[3];
};

// PIL precompute_coeffs: ksize = ceil(support) * 2 + 1 with support = max(in / out, 1) (bilinear support is 1).
// The division is correctly rounded on host and device alike, so both sides size the tables the same way.
__host__ __device__ inline int ksize_of(int in, int out) {
  double fs = (double)in / (double)out;
  if (fs < 1.0) fs = 1.0;
  return (int)ceil(fs) * 2 + 1;
}
// Pillow's Image.resize: a source more than 100 times taller than wide that gets shorter is resized vertically first.
__host__ __device__ inline bool vfirst_of(int h, int w, int out_h) { return h > 100ll * w && out_h < h; }
__host__ __device__ inline int64_t align16(int64_t x) { return (x + 15) & ~(int64_t)15; }
// one table: out x {xmin, n} then out x ks weights, int32
__host__ __device__ inline int64_t table_bytes(int in, int out) {
  return align16((int64_t)out * (2 + ksize_of(in, out)) * 4);
}
__host__ __device__ inline int64_t inter_bytes(int h, int w, int oh, int ow, int planes) {
  return align16(vfirst_of(h, w, oh) ? (int64_t)planes * oh * w : (int64_t)planes * h * ow);
}
__host__ __device__ inline int64_t image_ws_bytes(const int64_t* d, int oh, int ow) {
  const int h = (int)d[1], w = (int)d[2], hd = (int)d[4], wd = (int)d[5];
  return table_bytes(w, ow) + table_bytes(h, oh) + table_bytes(wd, ow) + table_bytes(hd, oh) +
         inter_bytes(h, w, oh, ow, 3) + inter_bytes(hd, wd, oh, ow, 1);
}
__host__ __device__ inline bool side_ok(int64_t v, int64_t max) { return v >= 1 && v <= max; }
// sizes and channel count; with packed_bytes > 0 also that both planes lie inside the packed buffer
__host__ __device__ inline bool desc_ok(const int64_t* d, int64_t packed_bytes, int64_t max_h, int64_t max_w) {
  if (!(side_ok(d[1], max_h) && side_ok(d[2], max_w) && side_ok(d[4], max_h) && side_ok(d[5], max_w))) return false;
  if (d[6] != 1 && d[6] != 3) return false;
  if (d[0] < 0 || d[3] < 0) return false;
  if (packed_bytes <= 0) return true;
  return d[0] + d[1] * d[2] * 3 <= packed_bytes && d[3] + d[4] * d[5] * d[6] <= packed_bytes;
}
inline int64_t head_bytes(int B) {
  return ((int64_t)B * (int64_t)sizeof(Plan) + 255) / 256 * 256 + 4 * 256 * (int64_t)sizeof(float);
}

__device__ __forceinline__ uint8_t clip8(int acc) {
  const int v = acc >> kPrecBits;
  return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v));
}

// One output sample of a resampling pass over n taps p[0], p[step], ...: acc = 2^21 + sum u8 * k in int32 (PIL
// ImagingResample{Horizontal,Vertical}_8bpc).  NIN channels cstride apart; LUMA turns 3 interleaved channels into one
// with convert('L')'s (19595 R + 38470 G + 7471 B + 0x8000) >> 16 before it is weighted.
template <int NIN, bool LUMA>
__device__ __forceinline__ void resample_one(const uint8_t* __restrict__ p, int64_t step, int64_t cstride,
                                             const int* __restrict__ k, int n, int (&acc)[LUMA ? 1 : NIN]) {
#pragma unroll
  for (int c = 0; c < (LUMA ? 1 : NIN); ++c) acc[c] = 1 << (kPrecBits - 1);
  for (int i = 0; i < n; ++i, p += step) {
    const int kv = __ldg(k + i);
    if (LUMA) {
      acc[0] += ((19595 * (int)p[0] + 38470 * (int)p[1] + 7471 * (int)p[2] + 0x8000) >> 16) * kv;
    } else {
#pragma unroll
      for (int c = 0; c < NIN; ++c) acc[c] += (int)p[c * cstride] * kv;
    }
  }
}

__global__ void __launch_bounds__(kPlanThreads) prep_plan_kernel(const int64_t* __restrict__ desc, int64_t packed_bytes,
                                                                 int B, int oh, int ow, int max_h, int max_w,
                                                                 int64_t ws_bytes, int64_t head, Norm norm,
                                                                 Plan* __restrict__ plan, float* __restrict__ lut) {
  __shared__ int64_t base[kPlanThreads];
  const int t = threadIdx.x, per = (B + kPlanThreads - 1) / kPlanThreads;
  const int b0 = min(B, t * per), b1 = min(B, b0 + per);
  int64_t need = 0;
  for (int b = b0; b < b1; ++b) {
    const int64_t* d = desc + (int64_t)b * kDescFields;
    if (desc_ok(d, packed_bytes, max_h, max_w)) need += image_ws_bytes(d, oh, ow);
  }
  base[t] = need;
  __syncthreads();
  if (t == 0) {
    int64_t run = head;
    for (int i = 0; i < kPlanThreads; ++i) {
      const int64_t v = base[i];
      base[i] = run;
      run += v;
    }
  }
  __syncthreads();
  int64_t off = base[t];
  for (int b = b0; b < b1; ++b) {
    const int64_t* d = desc + (int64_t)b * kDescFields;
    Plan p = {};
    if (desc_ok(d, packed_bytes, max_h, max_w)) {
      const int64_t bytes = image_ws_bytes(d, oh, ow);
      p.valid = off + bytes <= ws_bytes;
      p.src[0] = d[0];
      p.src[1] = d[3];
      p.h[0] = (int)d[1], p.w[0] = (int)d[2], p.h[1] = (int)d[4], p.w[1] = (int)d[5];
      p.ch = (int)d[6];
      int64_t o = off;
      for (int k = 0; k < 2; ++k) {
        p.vfirst[k] = vfirst_of(p.h[k], p.w[k], oh);
        p.ks[2 * k] = ksize_of(p.w[k], ow);
        p.ks[2 * k + 1] = ksize_of(p.h[k], oh);
        p.coef[2 * k] = o;
        o += table_bytes(p.w[k], ow);
        p.coef[2 * k + 1] = o;
        o += table_bytes(p.h[k], oh);
      }
      for (int k = 0; k < 2; ++k) {
        p.inter[k] = o;
        o += inter_bytes(p.h[k], p.w[k], oh, ow, k == 0 ? 3 : 1);
      }
      off += bytes;
    }
    plan[b] = p;
  }
  // ToTensor: u / 255; Normalize: (x - mean) / std -- correctly rounded fp32, as torch computes them on the host
  for (int i = t; i < 4 * 256; i += kPlanThreads) {
    const int c = i >> 8;
    const float x = __fdiv_rn((float)(i & 255), 255.0f);
    lut[i] = c < 3 ? __fdiv_rn(__fsub_rn(x, norm.mean[c]), norm.std[c]) : x;
  }
}

__device__ __forceinline__ double tri_weight(int x, double center, double ss) {
  double t = __dmul_rn(__dadd_rn(__dsub_rn((double)x, center), 0.5), ss);   // (x + xmin - center + 0.5) * ss
  t = t < 0.0 ? -t : t;
  return t < 1.0 ? __dsub_rn(1.0, t) : 0.0;
}

// PIL precompute_coeffs + normalize_coeffs_8bpc for one (image, table); thread = output index.  Every operation is a
// separately rounded float64 intrinsic so that nvcc cannot contract it into an FMA; the order is PIL's.
__global__ void __launch_bounds__(128) prep_coef_kernel(const Plan* __restrict__ plan, uint8_t* __restrict__ ws,
                                                        int oh, int ow) {
  const Plan& P = plan[blockIdx.x];
  if (!P.valid) return;
  const int t = blockIdx.y, k = t >> 1;
  const bool vert = t & 1;
  const int in = vert ? P.h[k] : P.w[k], out = vert ? oh : ow, ks = P.ks[t];
  int* bounds = reinterpret_cast<int*>(ws + P.coef[t]);
  int* kk = bounds + 2 * out;
  const double scale = __ddiv_rn((double)in, (double)out);
  const double fs = scale < 1.0 ? 1.0 : scale;   // filterscale; support = 1 * fs
  const double ss = __ddiv_rn(1.0, fs);
  for (int o = threadIdx.x; o < out; o += blockDim.x) {
    const double center = __dmul_rn(__dadd_rn((double)o, 0.5), scale);
    const int xmin = max(__double2int_rz(__dadd_rn(__dsub_rn(center, fs), 0.5)), 0);
    const int n = min(__double2int_rz(__dadd_rn(__dadd_rn(center, fs), 0.5)), in) - xmin;
    double ww = 0.0;
    for (int x = 0; x < n; ++x) ww = __dadd_rn(ww, tri_weight(x + xmin, center, ss));
    for (int x = 0; x < ks; ++x) {
      int v = 0;
      if (x < n) {
        double w = tri_weight(x + xmin, center, ss);
        if (ww != 0.0) w = __ddiv_rn(w, ww);
        v = __double2int_rz(__dadd_rn(0.5, __dmul_rn(w, (double)(1 << kPrecBits))));
      }
      kk[(int64_t)o * ks + x] = v;
    }
    bounds[2 * o] = xmin;
    bounds[2 * o + 1] = n;
  }
}

// First pass of plane kind z (0 = RGB, 1 = depth) of image blockIdx.y from the packed source into its intermediate:
// horizontal (output h x ow) or, for vfirst, vertical (output oh x w).
__global__ void __launch_bounds__(kTileW * kBlockRows) prep_pass1_kernel(const uint8_t* __restrict__ packed,
                                                                          uint8_t* __restrict__ ws,
                                                                          const Plan* __restrict__ plan, int oh,
                                                                          int ow) {
  const Plan& P = plan[blockIdx.y];
  const int z = blockIdx.z;
  if (!P.valid) return;
  const int h = P.h[z], w = P.w[z];
  const bool vf = P.vfirst[z];
  const int R = vf ? oh : h, C = vf ? w : ow;
  const int tiles_x = (C + kTileW - 1) / kTileW;
  const int ty = blockIdx.x / tiles_x, c = (blockIdx.x - ty * tiles_x) * kTileW + threadIdx.x;
  if (ty * kTileH >= R || c >= C) return;
  const int t = 2 * z + (vf ? 1 : 0);
  const int* bounds = reinterpret_cast<const int*>(ws + P.coef[t]);
  const int* kk = bounds + 2 * (vf ? oh : ow);
  const int ks = P.ks[t], nch = z == 0 ? 3 : P.ch;
  const uint8_t* src = packed + P.src[z];
  uint8_t* dst = ws + P.inter[z];
  const int64_t plane = (int64_t)R * C, pix = nch, row = (int64_t)w * nch;
  for (int r = ty * kTileH + threadIdx.y; r < min(R, (ty + 1) * kTileH); r += kBlockRows) {
    const int o = vf ? r : c;                       // index along the resampled axis
    const int lo = __ldg(bounds + 2 * o), n = __ldg(bounds + 2 * o + 1);
    const int* kw = kk + (int64_t)o * ks;
    const uint8_t* p = vf ? src + (int64_t)lo * row + (int64_t)c * pix : src + (int64_t)r * row + (int64_t)lo * pix;
    const int64_t step = vf ? row : pix, at = (int64_t)r * C + c;
    if (z == 0) {
      int a[3];
      resample_one<3, false>(p, step, 1, kw, n, a);
      dst[at] = clip8(a[0]);
      dst[plane + at] = clip8(a[1]);
      dst[2 * plane + at] = clip8(a[2]);
    } else if (nch == 3) {
      int a[1];
      resample_one<3, true>(p, step, 1, kw, n, a);
      dst[at] = clip8(a[0]);
    } else {
      int a[1];
      resample_one<1, false>(p, step, 0, kw, n, a);
      dst[at] = clip8(a[0]);
    }
  }
}

// Second pass along the other axis, from the intermediate to fp32 NCHW through the lookup: image (B, 3, oh, ow) for
// z = 0, depth (B, 1, oh, ow) for z = 1.  An image whose descriptor was rejected gets NaN.
__global__ void __launch_bounds__(kTileW * kBlockRows) prep_pass2_kernel(const uint8_t* __restrict__ ws,
                                                                          const Plan* __restrict__ plan,
                                                                          const float* __restrict__ lut,
                                                                          float* __restrict__ image,
                                                                          float* __restrict__ depth, int oh, int ow) {
  const Plan& P = plan[blockIdx.y];
  const int z = blockIdx.z, nch = z == 0 ? 3 : 1;
  const int tiles_x = (ow + kTileW - 1) / kTileW;
  const int ty = blockIdx.x / tiles_x, c = (blockIdx.x - ty * tiles_x) * kTileW + threadIdx.x;
  if (ty * kTileH >= oh || c >= ow) return;
  const int64_t oplane = (int64_t)oh * ow;
  float* out = z == 0 ? image + (int64_t)blockIdx.y * 3 * oplane : depth + (int64_t)blockIdx.y * oplane;
  const int r_end = min(oh, (ty + 1) * kTileH);
  if (!P.valid) {
    for (int r = ty * kTileH + threadIdx.y; r < r_end; r += kBlockRows)
      for (int ch = 0; ch < nch; ++ch) out[ch * oplane + (int64_t)r * ow + c] = __int_as_float(0x7fc00000);
    return;
  }
  const bool horiz = P.vfirst[z];                     // the axis the first pass left
  const int Ri = horiz ? oh : P.h[z], Ci = horiz ? P.w[z] : ow;
  const int t = 2 * z + (horiz ? 0 : 1);
  const int* bounds = reinterpret_cast<const int*>(ws + P.coef[t]);
  const int* kk = bounds + 2 * (horiz ? ow : oh);
  const int ks = P.ks[t];
  const uint8_t* src = ws + P.inter[z];
  const int64_t iplane = (int64_t)Ri * Ci;
  const float* lz = lut + (z == 0 ? 0 : 3 * 256);
  for (int r = ty * kTileH + threadIdx.y; r < r_end; r += kBlockRows) {
    const int o = horiz ? c : r;
    const int lo = __ldg(bounds + 2 * o), n = __ldg(bounds + 2 * o + 1);
    const int* kw = kk + (int64_t)o * ks;
    const uint8_t* p = horiz ? src + (int64_t)r * Ci + lo : src + (int64_t)lo * Ci + c;
    const int64_t step = horiz ? 1 : Ci, at = (int64_t)r * ow + c;
    if (z == 0) {
      int a[3];
      resample_one<3, false>(p, step, iplane, kw, n, a);
#pragma unroll
      for (int ch = 0; ch < 3; ++ch) out[ch * oplane + at] = __ldg(lz + ch * 256 + clip8(a[ch]));
    } else {
      int a[1];
      resample_one<1, false>(p, step, 0, kw, n, a);
      out[at] = __ldg(lz + clip8(a[0]));
    }
  }
}

}  // namespace
}  // namespace dgtd

using namespace dgtd;

extern "C" {

int64_t dgtd_rgbd_preprocess_ws_bytes(const int64_t* desc, int B, int out_h, int out_w) {
  DGTD_CHECK_ARG(desc && B > 0 && B <= 65535, "rgbd_preprocess: need 1 <= B <= 65535 descriptors");
  DGTD_CHECK_ARG(side_ok(out_h, kMaxSide) && side_ok(out_w, kMaxSide), "rgbd_preprocess: bad output size %d x %d",
                 out_h, out_w);
  int64_t total = head_bytes(B);
  for (int b = 0; b < B; ++b) {
    const int64_t* d = desc + (int64_t)b * kDescFields;
    DGTD_CHECK_ARG(desc_ok(d, 0, kMaxSide, kMaxSide), "rgbd_preprocess: descriptor %d is out of range", b);
    total += image_ws_bytes(d, out_h, out_w);
  }
  return total;
}

int dgtd_rgbd_preprocess_fwd(const void* packed, int64_t packed_bytes, int B, int max_h, int max_w, int out_h,
                             int out_w, float mean0, float mean1, float mean2, float std0, float std1, float std2,
                             void* ws, int64_t ws_bytes, float* image, float* depth, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(packed && ws && image && depth, "rgbd_preprocess: null pointer");
  DGTD_CHECK_ARG(B > 0 && B <= 65535, "rgbd_preprocess: need 1 <= B <= 65535, got %d", B);
  DGTD_CHECK_ARG(side_ok(out_h, kMaxSide) && side_ok(out_w, kMaxSide), "rgbd_preprocess: bad output size %d x %d",
                 out_h, out_w);
  DGTD_CHECK_ARG(side_ok(max_h, kMaxSide) && side_ok(max_w, kMaxSide), "rgbd_preprocess: bad max size %d x %d", max_h,
                 max_w);
  DGTD_CHECK_ARG(((uintptr_t)packed & 7) == 0 && packed_bytes >= (int64_t)B * kDescFields * 8,
                 "rgbd_preprocess: the packed buffer must be 8-byte aligned and hold the descriptors");
  DGTD_CHECK_ARG(((uintptr_t)ws & 255) == 0 && ws_bytes >= head_bytes(B),
                 "rgbd_preprocess: workspace must be 256-byte aligned, of dgtd_rgbd_preprocess_ws_bytes bytes");
  DGTD_CHECK_ARG(std0 != 0.f && std1 != 0.f && std2 != 0.f, "rgbd_preprocess: std must not be 0");
  cudaStream_t s = (cudaStream_t)stream;
  uint8_t* w8 = (uint8_t*)ws;
  Plan* plan = (Plan*)ws;
  float* lut = (float*)(w8 + head_bytes(B) - 4 * 256 * (int64_t)sizeof(float));
  const Norm norm = {{mean0, mean1, mean2}, {std0, std1, std2}};
  prep_plan_kernel<<<1, kPlanThreads, 0, s>>>((const int64_t*)packed, packed_bytes, B, out_h, out_w, max_h, max_w,
                                              ws_bytes, head_bytes(B), norm, plan, lut);
  DGTD_LAUNCH_CHECK("rgbd_preprocess plan");
  prep_coef_kernel<<<dim3(B, 4), 128, 0, s>>>(plan, w8, out_h, out_w);
  DGTD_LAUNCH_CHECK("rgbd_preprocess coef");
  const int64_t t1 = (int64_t)cdiv(max(max_h, out_h), kTileH) * cdiv(max(max_w, out_w), kTileW);
  const int64_t t2 = (int64_t)cdiv(out_h, kTileH) * cdiv(out_w, kTileW);
  DGTD_CHECK_ARG(t1 < (1ll << 31), "rgbd_preprocess: sizes too large");
  const dim3 block(kTileW, kBlockRows);
  prep_pass1_kernel<<<dim3((unsigned)t1, B, 2), block, 0, s>>>((const uint8_t*)packed, w8, plan, out_h, out_w);
  DGTD_LAUNCH_CHECK("rgbd_preprocess pass1");
  prep_pass2_kernel<<<dim3((unsigned)t2, B, 2), block, 0, s>>>(w8, plan, lut, image, depth, out_h, out_w);
  DGTD_LAUNCH_CHECK("rgbd_preprocess pass2");
  return 0;
}

}  // extern "C"
