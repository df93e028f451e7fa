// a6 at microbench scale (BASELINE configs[3]: 1024 x 1024 x 256, k = 7, T sweep):
// MessagePassing.forward core (cod.py:1190-1205) with shared weights (wc == 1) on NHWC maps.
//
// One launch per diffusion step (at C = 256 a step is already past the crossover between the HBM
// and the on-chip roofs, so fusing steps would only add halo recomputation).  Per CTA:
//   * 8 x 16 output pixels; the 49 raw weights of each pixel are read once (coalesced planes),
//     random-walk normalised (W / (sum W + eps), cod.py:1201) and kept in shared memory for ALL
//     channel chunks -- the reference re-reads a 49x unfolded copy of x instead;
//   * x streams through in chunks of 32*RC channels (256 B per pixel): one 4-D TMA box
//     (14 x 22 pixels, zero fill outside the map == unfold's zero padding) per chunk, double
//     buffered;
//   * warp = 2 x 8 pixel sub-tile (8 warps), lane = RC adjacent channels (fp32: 2, bf16
//     storage: 4): each input row is read once (8-byte shared loads, conflict free) and feeds up
//     to 2 output rows.
// The per-pixel weights are warp-uniform, so every FMA instruction needs one broadcast word from
// shared memory; with RC channels per lane that is 1/RC shared-memory wavefronts per FMA
// instruction against the 0.25 the FMA pipes can absorb -- the kernel is bound by shared-memory
// bandwidth, not HBM (DESIGN.md, profiles/).
// Algorithmic HBM traffic per step: (2*C*sizeof(T) + 49*4) * H * W bytes.
#include "blackwell.cuh"
#include "common.cuh"

namespace dgtd {

constexpr int MP_TH = 8, MP_TW = 16, MP_PH = MP_TH + 6, MP_PW = MP_TW + 6;
constexpr int MP_TILE_BYTES = MP_PH * MP_PW * 256;
constexpr int MP_WN_FLOATS = MP_TH * MP_TW * 56;   // [pixel][ky][8] (7 taps + 1 pad)
constexpr int MP_SMEM = 2 * MP_TILE_BYTES + MP_WN_FLOATS * 4 + 128;

template <int RC> struct MpVec;
template <> struct MpVec<2> {   // fp32 storage: 2 channels = 8 bytes
  using T = float;
  static __device__ __forceinline__ void load(const uint8_t* p, float (&v)[2]) {
    float2 t = *reinterpret_cast<const float2*>(p);
    v[0] = t.x; v[1] = t.y;
  }
  static __device__ __forceinline__ void store(float* p, const float (&v)[2]) {
    *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]);
  }
};
template <> struct MpVec<4> {   // bf16 storage: 4 channels = 8 bytes, fp32 accumulate
  using T = __nv_bfloat16;
  static __device__ __forceinline__ void load(const uint8_t* p, float (&v)[4]) {
    uint2 u = *reinterpret_cast<const uint2*>(p);
    float2 a = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&u.x));
    float2 b = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&u.y));
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&v)[4]) {
    store4(p, v[0], v[1], v[2], v[3]);
  }
};

template <int RC>
__global__ void __launch_bounds__(256, 1)
mp_tiled_kernel(const __grid_constant__ CUtensorMap tmX, const float* __restrict__ weight,
                typename MpVec<RC>::T* __restrict__ out, int h, int w, int C, float eps) {
  using V = MpVec<RC>;
  extern __shared__ __align__(128) uint8_t xs[];   // TMA destination; keeps ld.shared addressing
  float* wn = reinterpret_cast<float*>(xs + 2 * MP_TILE_BYTES);
  __shared__ uint64_t bar[2];

  const int tiles_x = (w + MP_TW - 1) / MP_TW, tiles_y = (h + MP_TH - 1) / MP_TH;
  int bid = blockIdx.x;
  const int tx = bid % tiles_x; bid /= tiles_x;
  const int ty = bid % tiles_y;
  const int n = bid / tiles_y;
  const int x0 = tx * MP_TW, y0 = ty * MP_TH;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sy = warp >> 1, sx = warp & 1;   // 4 x 2 sub-tiles of 2 x 8 pixels
  const int nchunks = C / (32 * RC);

  if (threadIdx.x == 0) {
    bw::prefetch_tmap(&tmX);
    bw::mbar_init(&bar[0], 1);
    bw::mbar_init(&bar[1], 1);
    bw::fence_mbar_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    bw::mbar_arrive_expect_tx(&bar[0], MP_TILE_BYTES);
    bw::tma_load_4d(&tmX, &bar[0], xs, 0, x0 - 3, y0 - 3, n);
  }
  if (threadIdx.x < MP_TH * MP_TW) {  // normalised weights of this tile: thread = pixel (row-major 8 x 16)
    const int py = threadIdx.x >> 4, px = threadIdx.x & 15;
    const int gy = y0 + py, gx = x0 + px;
    float wv[49];
    float s = 0.f;
    const bool ok = gy < h && gx < w;
    const float* wp = weight + ((int64_t)n * 49 * h + gy) * w + gx;
#pragma unroll
    for (int k = 0; k < 49; ++k) {
      wv[k] = ok ? __ldg(wp + (int64_t)k * h * w) : 0.f;
      s += wv[k];
    }
    const float inv = 1.0f / (s + eps);
    float* dst = wn + threadIdx.x * 56;
#pragma unroll
    for (int ky = 0; ky < 7; ++ky) {
#pragma unroll
      for (int kx = 0; kx < 7; ++kx) dst[ky * 8 + kx] = wv[ky * 7 + kx] * inv;
      dst[ky * 8 + 7] = 0.f;
    }
  }
  __syncthreads();

  const float* wbase = wn + ((2 * sy) * MP_TW + 8 * sx) * 56;
#pragma unroll 1
  for (int i = 0; i < nchunks; ++i) {
    if (threadIdx.x == 0 && i + 1 < nchunks) {
      bw::fence_proxy_async_smem();
      bw::mbar_arrive_expect_tx(&bar[(i + 1) & 1], MP_TILE_BYTES);
      bw::tma_load_4d(&tmX, &bar[(i + 1) & 1], xs + ((i + 1) & 1) * MP_TILE_BYTES, (i + 1) * 32 * RC, x0 - 3, y0 - 3, n);
    }
    float acc[2][8][RC];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int j = 0; j < 8; ++j)
#pragma unroll
        for (int r = 0; r < RC; ++r) acc[a][j][r] = 0.f;
    bw::mbar_wait(&bar[i & 1], (i >> 1) & 1);
    const uint8_t* base = xs + (i & 1) * MP_TILE_BYTES + ((2 * sy) * MP_PW + 8 * sx) * 256 + lane * 8;
#pragma unroll
    for (int iy = 0; iy < 8; ++iy) {
      float in[14][RC];
#pragma unroll
      for (int j = 0; j < 14; ++j) V::load(base + (iy * MP_PW + j) * 256, in[j]);
#pragma unroll
      for (int oy = 0; oy < 2; ++oy) {
        const int ky = iy - oy;
        if (ky < 0 || ky >= 7) continue;
#pragma unroll
        for (int ox = 0; ox < 8; ++ox) {
          const float* wp = wbase + (oy * MP_TW + ox) * 56 + ky * 8;
#pragma unroll
          for (int kx = 0; kx < 7; ++kx) {
            const float wv = wp[kx];           // warp-uniform: one broadcast wavefront
#pragma unroll
            for (int r = 0; r < RC; ++r) acc[oy][ox][r] = fmaf(wv, in[ox + kx][r], acc[oy][ox][r]);
          }
        }
      }
      asm volatile("" ::: "memory");   // one input row in flight: bounds the register footprint
    }
    const int c = (i * 32 + lane) * RC;
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      const int oy = y0 + 2 * sy + a;
      if (oy >= h) continue;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int ox = x0 + 8 * sx + j;
        if (ox < w) V::store(out + (((int64_t)n * h + oy) * w + ox) * C + c, acc[a][j]);
      }
    }
    __syncthreads();
  }
}

template <int RC>
static int mp_step(const void* x, const float* weight, void* out, int n, int h, int w, int c, float eps,
                   cudaStream_t s) {
  using T = typename MpVec<RC>::T;
  CUtensorMap tm;
  PFN_tmapEncodeTiled enc = get_tmap_encoder();
  if (!enc) return -3;
  const size_t es = sizeof(T);
  cuuint64_t gd[4] = {(cuuint64_t)c, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)n};
  cuuint64_t gs[3] = {(cuuint64_t)c * es, (cuuint64_t)w * c * es, (cuuint64_t)h * w * c * es};
  cuuint32_t bx[4] = {(cuuint32_t)(32 * RC), MP_PW, MP_PH, 1};
  cuuint32_t est[4] = {1, 1, 1, 1};
  CUresult r = enc(&tm, es == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4,
                   const_cast<void*>(x), gd, gs, bx, est, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("message_passing_tiled: cuTensorMapEncodeTiled failed (%d)", (int)r);
    return -3;
  }
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(mp_tiled_kernel<RC>, cudaFuncAttributeMaxDynamicSharedMemorySize, MP_SMEM);
    if (e != cudaSuccess) {
      set_error("message_passing_tiled: cannot opt in to %d B smem: %s", MP_SMEM, cudaGetErrorString(e));
      return -2;
    }
    configured = true;
  }
  const int64_t blocks = (int64_t)n * cdiv(h, MP_TH) * cdiv(w, MP_TW);
  mp_tiled_kernel<RC><<<(unsigned)blocks, 256, MP_SMEM, s>>>(tm, weight, (T*)out, h, w, c, eps);
  return 0;
}

// mp_tc.cu: one step on the tensor pipe (banded GEMM); returns 1 when the shape is not handled there
int mp_tc_step_bf16(const void* x, const float* weight, void* out, int n, int h, int w, int c, float eps, cudaStream_t s);
// mp_tc_f32.cu: the same step for fp32 storage (three bf16 products, fp32-level accuracy)
int mp_tc_step_f32(const void* x, const float* weight, void* out, int n, int h, int w, int c, float eps, cudaStream_t s);

}  // namespace dgtd

using namespace dgtd;

extern "C" int dgtd_message_passing_tc_fwd(const void* x, const float* weight, void* out, void* tmp, int n, int h, int w,
                                           int c, int T, float eps, int dtype, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(x && weight && out, "message_passing_tc: null pointer");
  DGTD_CHECK_ARG(dtype == DGTD_BF16 || dtype == DGTD_F32, "message_passing_tc: bad dtype %d", dtype);
  DGTD_CHECK_ARG(n > 0 && h > 0 && w > 0 && c >= 256 && c % 256 == 0 && T >= 1,
                 "message_passing_tc: bad shape n=%d h=%d w=%d c=%d T=%d (c must be a multiple of 256)", n, h, w, c, T);
  DGTD_CHECK_ARG(T == 1 || tmp, "message_passing_tc: tmp buffer required for T > 1");
  DGTD_CHECK_ARG(!(reinterpret_cast<uintptr_t>(x) & 15) && !(reinterpret_cast<uintptr_t>(out) & 15) &&
                     !(reinterpret_cast<uintptr_t>(tmp) & 15),
                 "message_passing_tc: buffers must be 16-byte aligned");
  cudaStream_t s = (cudaStream_t)stream;
  const void* src = x;   // ping-pong so that the last step lands in `out`
  for (int t = 0; t < T; ++t) {
    void* dst = ((T - 1 - t) % 2 == 0) ? out : tmp;
    int rc = dtype == DGTD_BF16 ? mp_tc_step_bf16(src, weight, dst, n, h, w, c, eps, s)
                                : mp_tc_step_f32(src, weight, dst, n, h, w, c, eps, s);
    if (rc > 0) {
      set_error("message_passing_tc: shape not supported");
      return -1;
    }
    if (rc) return rc;
    DGTD_LAUNCH_CHECK("message_passing_tc");
    src = dst;
  }
  return 0;
}

static int mp_tiled_simt(const void* x, const float* weight, void* out, void* tmp, int n, int h, int w, int c, int T,
                         float eps, int dtype, dgtd_stream_t stream, bool allow_tc);

extern "C" int dgtd_message_passing_tiled_fwd(const void* x, const float* weight, void* out, void* tmp, int n,
                                              int h, int w, int c, int T, float eps, int dtype,
                                              dgtd_stream_t stream) {
  return mp_tiled_simt(x, weight, out, tmp, n, h, w, c, T, eps, dtype, stream, true);
}
extern "C" int dgtd_message_passing_tiled_simt_fwd(const void* x, const float* weight, void* out, void* tmp, int n,
                                                   int h, int w, int c, int T, float eps, int dtype,
                                                   dgtd_stream_t stream) {
  return mp_tiled_simt(x, weight, out, tmp, n, h, w, c, T, eps, dtype, stream, false);
}

static int mp_tiled_simt(const void* x, const float* weight, void* out, void* tmp, int n, int h, int w, int c, int T,
                         float eps, int dtype, dgtd_stream_t stream, bool allow_tc) {
  DGTD_CHECK_ARG(x && weight && out, "message_passing_tiled: null pointer");
  DGTD_CHECK_ARG(dtype == DGTD_F32 || dtype == DGTD_BF16, "message_passing_tiled: bad dtype %d", dtype);
  const int cmul = dtype == DGTD_F32 ? 64 : 128;
  DGTD_CHECK_ARG(n > 0 && h > 0 && w > 0 && c >= cmul && c % cmul == 0 && T >= 1,
                 "message_passing_tiled: bad shape n=%d h=%d w=%d c=%d T=%d (c must be a multiple of %d)", n, h, w,
                 c, T, cmul);
  DGTD_CHECK_ARG(T == 1 || tmp, "message_passing_tiled: tmp buffer required for T > 1");
  DGTD_CHECK_ARG(!(reinterpret_cast<uintptr_t>(x) & 15) && !(reinterpret_cast<uintptr_t>(out) & 15),
                 "message_passing_tiled: buffers must be 16-byte aligned");
  // bf16 storage with C % 256 == 0 runs on the tensor pipe (mp_tc.cu); everything else on the SIMT kernel below
  if (allow_tc && c % 256 == 0 && (int64_t)h * w * 49 < ((int64_t)1 << 31) && (dtype == DGTD_BF16 || w % 4 == 0))
    return dgtd_message_passing_tc_fwd(x, weight, out, tmp, n, h, w, c, T, eps, dtype, stream);
  cudaStream_t s = (cudaStream_t)stream;
  const void* src = x;   // ping-pong so that the last step lands in `out`
  for (int t = 0; t < T; ++t) {
    void* dst = ((T - 1 - t) % 2 == 0) ? out : tmp;
    int rc = dtype == DGTD_F32 ? mp_step<2>(src, weight, dst, n, h, w, c, eps, s)
                               : mp_step<4>(src, weight, dst, n, h, w, c, eps, s);
    if (rc) return rc;
    DGTD_LAUNCH_CHECK("message_passing_tiled");
    src = dst;
  }
  return 0;
}
