// Mlp's depthwise 3x3 (pad 1) + bias + GELU on the bf16 hidden tokens of the PVT-v2 blocks (cod.py:852-854,
// 1520-1531), forward and backward, as persistent TMA-staged kernels (SURVEY.md 8f-1).
//
// CTA = 256 threads, tile = 8 x 16 output pixels x 64 channels (128 B of bf16 per pixel).  The 10 x 18 halo tile is ONE
// 4-D TMA box (zero fill outside the image == the conv's padding, so the kernel has no border tests on its inputs and no
// per-thread address arithmetic), double buffered: the box of the CTA's next tile is in flight while this one is
// computed.  A CTA keeps its 64-channel group for all its tiles (grid = multiple of C / 64; tiles enumerate the channel
// group fastest so that co-resident CTAs read the same pixels' full rows), taps + bias sit in shared memory.
// thread = 8 channels x 4 consecutive pixels of one tile row: 3 x 6 16-byte shared loads (a quarter warp reads 128
// contiguous bytes: conflict-free) feed 4 x 8 outputs through packed fp32x2 FMAs.
//
//   MODE_FWD  out = gelu(conv3(x) + b)                 bf16, the polynomial GELU of the GEMM epilogues (2.8e-5)
//   MODE_BWD  du = g * gelu'(conv3(x) + b)             fp32 (exact erf form), and in the same pass the tap / bias gradients
//             dw[k] = sum_p du[p] x[p + k], db = sum_p du[p]: 80 accumulators per thread carried across the CTA's tiles,
//             reduced over the CTA through shared memory once, written as per-CTA partials that a second kernel sums in
//             a fixed order (no atomics).  The input gradient is the depthwise conv of du with rotated taps
//             (dgtd_dwconv3_fwd), as before.
#include "tc_common.cuh"

namespace dgtd {

PFN_tmapEncodeTiled get_tmap_encoder();   // tc_gemm.cu
int sm_count();                           // tc_gemm.cu

namespace {

constexpr int D3_TH = 8, D3_TW = 16, D3_PH = D3_TH + 2, D3_PW = D3_TW + 2;
constexpr uint32_t D3_TILE_BYTES = D3_PH * D3_PW * 128;   // 23040
constexpr int MODE_FWD = 0, MODE_BWD = 1;

__device__ __forceinline__ float gelu_grad_erf(float x) {
  const float phi = 0.3989422804014327f * expf(-0.5f * x * x);
  return 0.5f * (1.0f + erff(x * 0.70710678118654752440f)) + x * phi;
}

__device__ __forceinline__ void unpack8(const uint4& raw, uint64_t (&v)[4]) {
  const uint32_t u[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
  for (int e = 0; e < 4; ++e)   // bf16 pair -> fp32 pair: low half << 16, high half masked
    v[e] = pk2(__uint_as_float(u[e] << 16), __uint_as_float(u[e] & 0xffff0000u));
}

template <int MODE>
__global__ void __launch_bounds__(256, MODE == MODE_FWD ? 2 : 1)
dwconv3_tma_kernel(const __grid_constant__ CUtensorMap tmX, const float* __restrict__ wT, const float* __restrict__ bias,
                   const float* __restrict__ g, void* __restrict__ outp, float* __restrict__ part, int h, int w, int C,
                   int tiles_x, int tiles_y, int ntiles) {
  extern __shared__ __align__(128) uint8_t xs[];   // 2 TMA stages
  __shared__ uint64_t bar[2];
  __shared__ __align__(16) float ws[10][64];       // 9 taps + bias of this CTA's channel group
  const int cgs = C >> 6;
  const int cg = blockIdx.x % cgs;                 // gridDim.x % cgs == 0: fixed for the CTA's lifetime
  const int tid = threadIdx.x;
  for (int i = tid; i < 640; i += 256) {
    const int j = i >> 6, cc = i & 63;
    ws[j][cc] = j < 9 ? wT[(int64_t)j * C + cg * 64 + cc] : bias[cg * 64 + cc];
  }
  if (tid == 0) {
    bw::prefetch_tmap(&tmX);
    bw::mbar_init(&bar[0], 1);
    bw::mbar_init(&bar[1], 1);
    bw::fence_mbar_init();
  }
  __syncthreads();

  // tile = blockIdx.x + n * gridDim.x with a fixed channel group: the spatial index advances by gridDim.x / cgs per
  // step; (tx, ty, b) are carried as mixed-radix digits (no division inside the loop)
  const uint32_t step = gridDim.x / cgs;
  const uint32_t sx = step % tiles_x, sy = (step / tiles_x) % tiles_y, sb = step / (tiles_x * tiles_y);
  uint32_t sp0 = blockIdx.x / cgs;
  uint32_t tx = sp0 % tiles_x, ty = (sp0 / tiles_x) % tiles_y, b = sp0 / (tiles_x * tiles_y);
  auto advance = [&](uint32_t& ax, uint32_t& ay, uint32_t& ab) {
    ax += sx;
    if (ax >= (uint32_t)tiles_x) { ax -= tiles_x; ++ay; }
    ay += sy;
    if (ay >= (uint32_t)tiles_y) { ay -= tiles_y; ++ab; }
    ab += sb;
  };
  auto issue = [&](uint32_t ax, uint32_t ay, uint32_t ab, int stage) {
    bw::mbar_arrive_expect_tx(&bar[stage], D3_TILE_BYTES);
    bw::tma_load_4d(&tmX, &bar[stage], xs + stage * D3_TILE_BYTES, cg * 64, (int)ax * D3_TW - 1, (int)ay * D3_TH - 1, (int)ab);
  };
  int tile = blockIdx.x;
  if (tid == 0 && tile < ntiles) issue(tx, ty, b, 0);

  const int oct = tid & 7, grp = tid >> 3;
  const int gx = grp & 3, gy = grp >> 2;
  const int co = oct * 8;
  // gradient accumulators (MODE_BWD): dwa[k][e] pairs for the 9 taps, dba[e] for the bias
  uint64_t dwa[MODE == MODE_BWD ? 9 : 1][4], dba[4];
  if (MODE == MODE_BWD) {
#pragma unroll
    for (int k = 0; k < 9; ++k)
#pragma unroll
      for (int e = 0; e < 4; ++e) dwa[k][e] = 0ull;
#pragma unroll
    for (int e = 0; e < 4; ++e) dba[e] = 0ull;
  }

#pragma unroll 1
  for (int it = 0; tile < ntiles; tile += gridDim.x, ++it) {
    const int stage = it & 1;
    const int oy = (int)ty * D3_TH + gy, ox0 = (int)tx * D3_TW + gx * 4;
    const int bcur = (int)b;
    advance(tx, ty, b);                  // -> the CTA's next tile
    if (tid == 0 && tile + (int)gridDim.x < ntiles) {   // stage ^ 1 was released by the __syncthreads of the previous iteration
      bw::fence_proxy_async_smem();
      issue(tx, ty, b, stage ^ 1);
    }

    uint64_t acc[4][4];
    {
      float bs[8];
      const float4 b0 = *reinterpret_cast<const float4*>(&ws[9][co]), b1 = *reinterpret_cast<const float4*>(&ws[9][co + 4]);
      bs[0] = b0.x; bs[1] = b0.y; bs[2] = b0.z; bs[3] = b0.w; bs[4] = b1.x; bs[5] = b1.y; bs[6] = b1.z; bs[7] = b1.w;
#pragma unroll
      for (int p = 0; p < 4; ++p)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[p][e] = pk2(bs[2 * e], bs[2 * e + 1]);
    }
    bw::mbar_wait(&bar[stage], (it >> 1) & 1);
    const uint8_t* win = xs + stage * D3_TILE_BYTES + ((gy * D3_PW) + gx * 4) * 128 + oct * 16;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      uint64_t k[3][4];
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const float4 k0 = *reinterpret_cast<const float4*>(&ws[ky * 3 + kx][co]);
        const float4 k1 = *reinterpret_cast<const float4*>(&ws[ky * 3 + kx][co + 4]);
        k[kx][0] = pk2(k0.x, k0.y); k[kx][1] = pk2(k0.z, k0.w); k[kx][2] = pk2(k1.x, k1.y); k[kx][3] = pk2(k1.z, k1.w);
      }
#pragma unroll
      for (int j = 0; j < 6; ++j) {
        uint64_t v[4];
        unpack8(*reinterpret_cast<const uint4*>(win + (ky * D3_PW + j) * 128), v);
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const int p = j - kx;
          if (p < 0 || p >= 4) continue;
#pragma unroll
          for (int e = 0; e < 4; ++e) acc[p][e] = fma2(v[e], k[kx][e], acc[p][e]);
        }
      }
    }
    const bool row_ok = oy < h;
    if (MODE == MODE_FWD) {
      __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(outp);
      if (row_ok) {
#pragma unroll
        for (int p = 0; p < 4; ++p) {
          if (ox0 + p >= w) break;
          float r[8];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            up2(acc[p][e], r[2 * e], r[2 * e + 1]);
            gelu_fast2(r[2 * e], r[2 * e + 1]);
          }
          store8(out + (((int64_t)bcur * h + oy) * w + ox0 + p) * C + cg * 64 + co, r);
        }
      }
    } else {
      float* du = reinterpret_cast<float*>(outp);
      // acc <- du = g * gelu'(u) (0 outside the image: those pixels contribute nothing to the gradients)
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const bool ok = row_ok && ox0 + p < w;
        float d[8];
        if (ok) {
          const int64_t off = (((int64_t)bcur * h + oy) * w + ox0 + p) * C + cg * 64 + co;
          const float4 g0 = *reinterpret_cast<const float4*>(g + off), g1 = *reinterpret_cast<const float4*>(g + off + 4);
          const float gv[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            float u0, u1;
            up2(acc[p][e], u0, u1);
            d[2 * e] = gv[2 * e] * gelu_grad_erf(u0);
            d[2 * e + 1] = gv[2 * e + 1] * gelu_grad_erf(u1);
          }
          *reinterpret_cast<float4*>(du + off) = make_float4(d[0], d[1], d[2], d[3]);
          *reinterpret_cast<float4*>(du + off + 4) = make_float4(d[4], d[5], d[6], d[7]);
        } else {
#pragma unroll
          for (int e = 0; e < 8; ++e) d[e] = 0.f;
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          acc[p][e] = pk2(d[2 * e], d[2 * e + 1]);
          dba[e] = add2(dba[e], acc[p][e]);
        }
      }
      // tap gradients: the same window walk with the roles of taps and outputs exchanged
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
        for (int j = 0; j < 6; ++j) {
          uint64_t v[4];
          unpack8(*reinterpret_cast<const uint4*>(win + (ky * D3_PW + j) * 128), v);
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) {
            const int p = j - kx;
            if (p < 0 || p >= 4) continue;
#pragma unroll
            for (int e = 0; e < 4; ++e) dwa[ky * 3 + kx][e] = fma2(v[e], acc[p][e], dwa[ky * 3 + kx][e]);
          }
        }
      }
    }
    __syncthreads();   // every thread is done with this stage before it is refilled
  }

  if (MODE == MODE_BWD) {
    // reduce the 80 accumulators over the 32 pixel groups of the CTA (two passes of 40 through the stage buffers)
    float* red = reinterpret_cast<float*>(xs);   // [40][256]
    float vals[80];
#pragma unroll
    for (int k = 0; k < 9; ++k)
#pragma unroll
      for (int e = 0; e < 4; ++e) up2(dwa[k][e], vals[k * 8 + 2 * e], vals[k * 8 + 2 * e + 1]);
#pragma unroll
    for (int e = 0; e < 4; ++e) up2(dba[e], vals[72 + 2 * e], vals[72 + 2 * e + 1]);
#pragma unroll
    for (int half = 0; half < 2; ++half) {
#pragma unroll
      for (int f = 0; f < 40; ++f) red[f * 256 + tid] = vals[half * 40 + f];
      __syncthreads();
      for (int i = tid; i < 40 * 8; i += 256) {       // (f, octet): sum over the 32 groups in order
        const int f = i >> 3, o = i & 7;
        float s = 0.f;
        for (int gq = 0; gq < 32; ++gq) s += red[f * 256 + gq * 8 + o];
        const int ff = half * 40 + f;                 // = tap * 8 + e (tap 9 = bias)
        part[((int64_t)blockIdx.x * 10 + (ff >> 3)) * 64 + o * 8 + (ff & 7)] = s;
      }
      __syncthreads();
    }
  }
}

// dwT[k][c] = sum over the CTAs of channel group c / 64 (cta = cg + n * cgs, n ascending) of part[cta][k][c % 64]
__global__ void dwconv3_wgrad_finalize_kernel(const float* __restrict__ part, int nctas, int cgs, int C,
                                              float* __restrict__ dwT, float* __restrict__ dbias) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 10 * C) return;
  const int k = i / C, c = i - k * C;
  const int cg = c >> 6, cc = c & 63;
  float s = 0.f;
  for (int cta = cg; cta < nctas; cta += cgs) s += part[((int64_t)cta * 10 + k) * 64 + cc];
  if (k < 9) dwT[(int64_t)k * C + c] = s;
  else dbias[c] = s;
}

int d3_grid(int ntiles, int cgs, int ctas_per_sm) {
  int grid = ctas_per_sm * sm_count();
  if (grid > ntiles) grid = ntiles;
  grid = grid / cgs * cgs;
  return grid < cgs ? cgs : grid;
}

int d3_make_tmap(CUtensorMap* tm, const void* x, int B, int h, int w, int C) {
  PFN_tmapEncodeTiled enc = get_tmap_encoder();
  if (!enc) return -3;
  cuuint64_t gd[4] = {(cuuint64_t)C, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)B};
  cuuint64_t gs[3] = {(cuuint64_t)C * 2, (cuuint64_t)w * C * 2, (cuuint64_t)h * w * C * 2};
  cuuint32_t bx[4] = {64, (cuuint32_t)D3_PW, (cuuint32_t)D3_PH, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(x), gd, gs, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("dwconv3(tma): cuTensorMapEncodeTiled failed (%d) for x (%d,%d,%d,%d)", (int)r, B, h, w, C);
    return -3;
  }
  return 0;
}

}  // namespace

// Returns 1 when the shape is not handled here (the caller falls through to the register-window kernel).
int dwconv3_gelu_tma(const void* x, const float* wT, const float* bias, void* out, int B, int h, int w, int C,
                     cudaStream_t s) {
  if (C % 64 || (reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(out) & 15)) return 1;
  CUtensorMap tm;
  int rc = d3_make_tmap(&tm, x, B, h, w, C);
  if (rc) return rc;
  const int tiles_x = cdiv(w, D3_TW), tiles_y = cdiv(h, D3_TH), cgs = C / 64;
  const int64_t nt = (int64_t)B * tiles_x * tiles_y * cgs;
  if (nt >= (1ll << 31)) return 1;
  const int grid = d3_grid((int)nt, cgs, 2);
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(dwconv3_tma_kernel<MODE_FWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * D3_TILE_BYTES);
    cudaFuncSetAttribute(dwconv3_tma_kernel<MODE_BWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * D3_TILE_BYTES);
    attr = true;
  }
  dwconv3_tma_kernel<MODE_FWD><<<grid, 256, 2 * D3_TILE_BYTES, s>>>(tm, wT, bias, nullptr, out, nullptr, h, w, C, tiles_x,
                                                                   tiles_y, (int)nt);
  return 0;
}

int64_t dwconv3_gelu_bwd_tma_ws_floats() { return (int64_t)512 * 640; }   // per-CTA partials, grid <= 512

// Returns 1 when the shape is not handled here.
int dwconv3_gelu_bwd_tma(const void* x, const float* wT, const float* bias, const float* g, float* du, float* dwT,
                         float* dbias, float* ws, int B, int h, int w, int C, cudaStream_t s) {
  if (!ws || C % 64 || (reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(g) & 15) ||
      (reinterpret_cast<uintptr_t>(du) & 15))
    return 1;
  CUtensorMap tm;
  int rc = d3_make_tmap(&tm, x, B, h, w, C);
  if (rc) return rc;
  const int tiles_x = cdiv(w, D3_TW), tiles_y = cdiv(h, D3_TH), cgs = C / 64;
  const int64_t nt = (int64_t)B * tiles_x * tiles_y * cgs;
  if (nt >= (1ll << 31)) return 1;
  const int grid = d3_grid((int)nt, cgs, 1);
  if ((int64_t)grid * 640 > dwconv3_gelu_bwd_tma_ws_floats()) return 1;
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(dwconv3_tma_kernel<MODE_BWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * D3_TILE_BYTES);
    attr = true;
  }
  dwconv3_tma_kernel<MODE_BWD><<<grid, 256, 2 * D3_TILE_BYTES, s>>>(tm, wT, bias, g, du, ws, h, w, C, tiles_x, tiles_y,
                                                                   (int)nt);
  dwconv3_wgrad_finalize_kernel<<<cdiv(10 * C, 256), 256, 0, s>>>(ws, grid, cgs, C, dwT, dbias);
  return 0;
}

}  // namespace dgtd
