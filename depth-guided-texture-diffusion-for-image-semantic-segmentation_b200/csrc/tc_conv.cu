// tcgen05 implicit-GEMM convolution over NHWC bf16 for the ShapePropDecoder stack
// (cod.py:1216-1222) and the injection-folded last conv (cod.py:1471).
//
// GEMM view: M = output pixels, N = Cout, K = taps x 32 (input channels padded to 32).
// Nothing is materialised: per tap the TMA producer loads the (TH x TW) pixel tile shifted by
// the tap offset straight from the NHWC tensor (4-D tensor map, element strides = conv stride,
// out-of-bounds = zero padding) into a 64B-swizzled K-major smem tile that tcgen05.mma consumes.
// Groups (the 16 decoders of the path) are a grid dimension: group g reads channel slice
// [32g, 32g+32) of x, weight rows [g*w_group_rows, ...) and writes out + g*out_group_stride.
#include "blackwell.cuh"
#include "common.cuh"

namespace dgtd {

int sm_count();

struct ConvParams {
  int B, oh, ow, Cout, ldo;
  int ks, stride, off;
  int TW, TH, tiles_x, tiles_y, tiles_n, groups;
  int w_group_rows;
  int64_t out_group_stride;
  int x5d;        // group-major input: tmX is 5-D {32 ch, W, H, B, group}, a group's pixels are dense 64-byte rows
  int out_split;  // groups == 1, bf16: 32-channel chunk c of the output goes to out + c * out_group_stride (pixel pitch ldo)
  const float* bias;  // [groups * w_group_rows] nullable
  void* out;
};

template <int BN>
struct ConvCfg {
  static constexpr int BM = 128, CP = 32;                 // channels per tap (padded)
  static constexpr int A_BYTES = BM * CP * 2, B_BYTES = BN * CP * 2;
  static constexpr int STAGES = 8;
  static constexpr int TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;
  static constexpr int SMEM_BYTES = STAGES * (A_BYTES + B_BYTES) + 256 + 1024;
};

template <int BN, int ACT, typename OT>
__global__ void __launch_bounds__(256, 1)
tc_conv_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW,
               const ConvParams p) {
  using Cfg = ConvCfg<BN>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ __align__(1024) uint8_t smem[];   // 128B-swizzle atoms need 1024-byte alignment
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * Cfg::A_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * (Cfg::A_BYTES + Cfg::B_BYTES));
  uint64_t* full = bars;
  uint64_t* empty = bars + STAGES;
  uint64_t* tfull = bars + 2 * STAGES;
  uint64_t* tempty = bars + 2 * STAGES + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int taps = p.ks * p.ks;
  const int tiles_img = p.tiles_x * p.tiles_y;
  const int num_tiles = p.groups * p.B * tiles_img * p.tiles_n;
  const uint32_t a_bytes = (uint32_t)(p.TW * p.TH) * Cfg::CP * 2;

  auto decode = [&](int tile, int& g, int& b, int& ty, int& tx, int& nb) {
    nb = tile % p.tiles_n; tile /= p.tiles_n;
    tx = tile % p.tiles_x; tile /= p.tiles_x;
    ty = tile % p.tiles_y; tile /= p.tiles_y;
    b = tile % p.B;
    g = tile / p.B;
  };

  if (warp == 0 && lane == 0) {
    bw::prefetch_tmap(&tmX);
    bw::prefetch_tmap(&tmW);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) {
      bw::mbar_init(&full[i], 1);
      bw::mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      bw::mbar_init(&tfull[i], 1);
      bw::mbar_init(&tempty[i], 128);
    }
    bw::fence_mbar_init();
  }
  if (warp == 2) bw::tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  bw::tc_fence_before();
  __syncthreads();
  bw::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        int g, b, ty, tx, nb;
        decode(tile, g, b, ty, tx, nb);
        const int ix0 = tx * p.TW * p.stride + p.off, iy0 = ty * p.TH * p.stride + p.off;
        for (int t = 0; t < taps; ++t) {
          const int dy = t / p.ks, dx = t - dy * p.ks;
          bw::mbar_wait(&empty[stage], phase ^ 1);
          bw::mbar_arrive_expect_tx(&full[stage], a_bytes + Cfg::B_BYTES);
          if (p.x5d) bw::tma_load_5d(&tmX, &full[stage], sA + stage * Cfg::A_BYTES, 0, ix0 + dx, iy0 + dy, b, g);
          else bw::tma_load_4d(&tmX, &full[stage], sA + stage * Cfg::A_BYTES, g * Cfg::CP, ix0 + dx, iy0 + dy, b);
          bw::tma_load_2d(&tmW, &full[stage], sB + stage * Cfg::B_BYTES, t * Cfg::CP,
                          g * p.w_group_rows + nb * BN);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = bw::umma_idesc_bf16(128, BN);
      int stage = 0, iter = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++iter) {
        const int as = iter & 1;
        const uint32_t aphase = (iter >> 1) & 1;
        bw::mbar_wait(&tempty[as], aphase ^ 1);
        bw::tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int t = 0; t < taps; ++t) {
          bw::mbar_wait(&full[stage], phase);
          bw::tc_fence_after();
          const uint64_t da = bw::umma_smem_desc_kmajor(bw::smem_u32(sA + stage * Cfg::A_BYTES), 64);
          const uint64_t db = bw::umma_smem_desc_kmajor(bw::smem_u32(sB + stage * Cfg::B_BYTES), 64);
#pragma unroll
          for (int k = 0; k < 2; ++k) bw::umma_bf16(d_tmem, da + 2 * k, db + 2 * k, idesc, (t | k) != 0);
          bw::umma_commit(&empty[stage]);
          if (t == taps - 1) bw::umma_commit(&tfull[as]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp >= 4) {
    const int ew = warp - 4;
    int iter = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++iter) {
      int g, b, ty, tx, nb;
      decode(tile, g, b, ty, tx, nb);
      const int as = iter & 1;
      const uint32_t aphase = (iter >> 1) & 1;
      bw::mbar_wait(&tfull[as], aphase);
      bw::tc_fence_after();
      const int r = ew * 32 + lane;                 // row of the tile = (j, i) pixel
      const int j = r / p.TW, i = r - j * p.TW;
      const int oy = ty * p.TH + j, ox = tx * p.TW + i;
      const bool row_ok = (j < p.TH) && oy < p.oh && ox < p.ow;
      OT* orow = reinterpret_cast<OT*>(p.out) + (int64_t)g * p.out_group_stride +
                 (((int64_t)b * p.oh + oy) * p.ow + ox) * p.ldo;
      const float* bias = p.bias ? p.bias + g * p.w_group_rows : nullptr;
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t v[32];
        bw::tmem_ld_32x32(tmem_base + ((uint32_t)(ew * 32) << 16) + as * BN + c0, v);
        bw::tmem_ld_wait();
        const int col0 = nb * BN + c0;
        if (row_ok && col0 < p.Cout) {
#pragma unroll
          for (int q = 0; q < 32; q += 8) {
            if (col0 + q >= p.Cout) break;
            float f[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) f[e] = __uint_as_float(v[q + e]);
            if (bias) {
              float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + col0 + q));
              float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + col0 + q + 4));
              f[0] += b0.x; f[1] += b0.y; f[2] += b0.z; f[3] += b0.w;
              f[4] += b1.x; f[5] += b1.y; f[6] += b1.z; f[7] += b1.w;
            }
            if (ACT == DGTD_ACT_RELU) {
#pragma unroll
              for (int e = 0; e < 8; ++e) f[e] = fmaxf(f[e], 0.f);
            }
            store4(orow + col0 + q, f[0], f[1], f[2], f[3]);
            store4(orow + col0 + q + 4, f[4], f[5], f[6], f[7]);
          }
        }
      }
      bw::tc_fence_before();
      bw::mbar_arrive(&tempty[as]);
    }
  }

  bw::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    bw::tc_fence_after();
    bw::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------------
// Resident-weights form of the per-tap kernel (the injection-folded 4x4 stride-r convs, round 2).  The kernel
// above re-loads the BN x 32 weight tile of every tap for every output tile: as many L2 -> SM bytes as the
// activations, and the three launches of a step ran at 10.5 TB/s of L2 traffic (85 % of the LTS cap) with the
// tensor pipe at 28 %.  Here a CTA owns ONE (group, n-block) key, loads its taps x BN x 32 weights once and
// walks that key's output tiles; only the activation tiles stream.
template <int BN>
struct ConvRwCfg {
  static constexpr int BM = 128, CP = 32, MAX_TAPS = 16;
  static constexpr int A_BYTES = BM * CP * 2;
  static constexpr int W_BYTES = MAX_TAPS * BN * CP * 2;
  static constexpr int STAGES = 8;
  static constexpr int TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;
  static constexpr int NEPI = 8;               // two epilogue warps per TMEM lane quadrant, half of the columns each
  static constexpr int STG_BYTES = NEPI * 2048;   // per epilogue warp: one 32-row x 64-byte staging tile
  static constexpr int SMEM_BYTES = STAGES * A_BYTES + W_BYTES + STG_BYTES + 256 + 1024;
};

template <int BN, int ACT, typename OT>
__global__ void __launch_bounds__(128 + 32 * ConvRwCfg<BN>::NEPI, 1)
tc_conv_resw_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW,
                    const ConvParams p) {
  using Cfg = ConvRwCfg<BN>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sA = smem;
  uint8_t* sW = smem + STAGES * Cfg::A_BYTES;
  uint8_t* sStg = sW + Cfg::W_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sStg + Cfg::STG_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + STAGES;
  uint64_t* tfull = bars + 2 * STAGES;
  uint64_t* tempty = bars + 2 * STAGES + 2;
  uint64_t* wfull = bars + 2 * STAGES + 4;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 5);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int taps = p.ks * p.ks;
  const int tiles_img = p.tiles_x * p.tiles_y;
  const int per_key = p.B * tiles_img;
  const int keys = p.groups * p.tiles_n;                      // <= gridDim.x (checked by the launcher)
  const int nct = (int)gridDim.x / keys;                      // CTAs sharing a key
  const int key = (int)blockIdx.x % keys, ci = (int)blockIdx.x / keys;
  const int g = key / p.tiles_n, nb = key - g * p.tiles_n;
  const bool active = ci < nct;
  const uint32_t a_bytes = (uint32_t)(p.TW * p.TH) * Cfg::CP * 2;

  if (warp == 0 && lane == 0) {
    bw::prefetch_tmap(&tmX);
    bw::prefetch_tmap(&tmW);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) {
      bw::mbar_init(&full[i], 1);
      bw::mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      bw::mbar_init(&tfull[i], 1);
      bw::mbar_init(&tempty[i], 32 * Cfg::NEPI);
    }
    bw::mbar_init(wfull, 1);
    bw::fence_mbar_init();
  }
  if (warp == 2) bw::tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  bw::tc_fence_before();
  __syncthreads();
  bw::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0 && active) {
      bw::mbar_arrive_expect_tx(wfull, (uint32_t)taps * BN * 64);
#pragma unroll 1
      for (int t = 0; t < taps; ++t)
        bw::tma_load_2d(&tmW, wfull, sW + t * BN * 64, t * Cfg::CP, g * p.w_group_rows + nb * BN);
      int stage = 0;
      uint32_t phase = 0;
      for (int pos = ci; pos < per_key; pos += nct) {
        const int b = pos / tiles_img, r = pos - b * tiles_img;
        const int ty = r / p.tiles_x, tx = r - ty * p.tiles_x;
        const int ix0 = tx * p.TW * p.stride + p.off, iy0 = ty * p.TH * p.stride + p.off;
        for (int t = 0; t < taps; ++t) {
          const int dy = t / p.ks, dx = t - dy * p.ks;
          bw::mbar_wait(&empty[stage], phase ^ 1);
          bw::mbar_arrive_expect_tx(&full[stage], a_bytes);
          if (p.x5d) bw::tma_load_5d(&tmX, &full[stage], sA + stage * Cfg::A_BYTES, 0, ix0 + dx, iy0 + dy, b, g);
          else bw::tma_load_4d(&tmX, &full[stage], sA + stage * Cfg::A_BYTES, g * Cfg::CP, ix0 + dx, iy0 + dy, b);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && active) {
      constexpr uint32_t idesc = bw::umma_idesc_bf16(128, BN);
      int stage = 0, iter = 0;
      uint32_t phase = 0;
      bw::mbar_wait(wfull, 0);
      bw::tc_fence_after();
      const uint64_t db_base = bw::umma_smem_desc_kmajor(bw::smem_u32(sW), 64);
      for (int pos = ci; pos < per_key; pos += nct, ++iter) {
        const int as = iter & 1;
        const uint32_t aphase = (iter >> 1) & 1;
        bw::mbar_wait(&tempty[as], aphase ^ 1);
        bw::tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int t = 0; t < taps; ++t) {
          bw::mbar_wait(&full[stage], phase);
          bw::tc_fence_after();
          const uint64_t da = bw::umma_smem_desc_kmajor(bw::smem_u32(sA + stage * Cfg::A_BYTES), 64);
          const uint64_t db = db_base + (uint64_t)((t * BN * 64) >> 4);
#pragma unroll
          for (int k = 0; k < 2; ++k) bw::umma_bf16(d_tmem, da + 2 * k, db + 2 * k, idesc, (t | k) != 0);
          bw::umma_commit(&empty[stage]);
          if (t == taps - 1) bw::umma_commit(&tfull[as]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp >= 4 && active) {
    const int ew = (warp - 4) & 3, part = (warp - 4) >> 2;   // TMEM lane quadrant (= warp % 4), column half
    constexpr int CPW = BN / (Cfg::NEPI / 4);
    int iter = 0;
    const float* bias = p.bias ? p.bias + g * p.w_group_rows : nullptr;
    for (int pos = ci; pos < per_key; pos += nct, ++iter) {
      const int b = pos / tiles_img, rr = pos - b * tiles_img;
      const int ty = rr / p.tiles_x, tx = rr - ty * p.tiles_x;
      const int as = iter & 1;
      const uint32_t aphase = (iter >> 1) & 1;
      bw::mbar_wait(&tfull[as], aphase);
      bw::tc_fence_after();
      const int r = ew * 32 + lane;                 // row of the tile = (j, i) pixel
      const int j = r / p.TW, i = r - j * p.TW;
      const int oy = ty * p.TH + j, ox = tx * p.TW + i;
      const bool row_ok = (j < p.TH) && oy < p.oh && ox < p.ow;
      OT* orow = reinterpret_cast<OT*>(p.out) + (int64_t)g * p.out_group_stride +
                 (((int64_t)b * p.oh + oy) * p.ow + ox) * p.ldo;
      if (sizeof(OT) == 2) {
        // bf16 results: 32 rows x 32 channels are transposed through a swizzled staging tile so that four lanes write
        // the 64 contiguous bytes of a pixel with 16-byte stores (the direct form issued 8-byte stores at a pitch of
        // a whole token row: 32 partially written sectors per instruction, 6x the output bytes in L2 transactions)
        uint8_t* stg = sStg + (warp - 4) * 2048;
        OT* rowp[4];
        bool rowok[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int r2 = ew * 32 + k * 8 + (lane >> 2);
          const int j2 = r2 / p.TW, i2 = r2 - j2 * p.TW;
          const int oy2 = ty * p.TH + j2, ox2 = tx * p.TW + i2;
          rowok[k] = (j2 < p.TH) && oy2 < p.oh && ox2 < p.ow;
          rowp[k] = reinterpret_cast<OT*>(p.out) + (int64_t)g * p.out_group_stride +
                    (((int64_t)b * p.oh + oy2) * p.ow + ox2) * p.ldo;
        }
        const int piece = lane & 3;
#pragma unroll 1
        for (int c0 = part * CPW; c0 < (part + 1) * CPW; c0 += 32) {
          uint32_t v[32];
          bw::tmem_ld_32x32(tmem_base + ((uint32_t)(ew * 32) << 16) + as * BN + c0, v);
          bw::tmem_ld_wait();
          const int col0 = nb * BN + c0;
          if (col0 >= p.Cout) break;                   // warp-uniform
#pragma unroll
          for (int q = 0; q < 32; q += 8) {
            float f[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) f[e] = __uint_as_float(v[q + e]);
            if (bias && col0 + q < p.Cout) {
              float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + col0 + q));
              float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + col0 + q + 4));
              f[0] += b0.x; f[1] += b0.y; f[2] += b0.z; f[3] += b0.w;
              f[4] += b1.x; f[5] += b1.y; f[6] += b1.z; f[7] += b1.w;
            }
            if (ACT == DGTD_ACT_RELU) {
#pragma unroll
              for (int e = 0; e < 8; ++e) f[e] = fmaxf(f[e], 0.f);
            }
            __nv_bfloat162 h0 = __floats2bfloat162_rn(f[0], f[1]), h1 = __floats2bfloat162_rn(f[2], f[3]);
            __nv_bfloat162 h2 = __floats2bfloat162_rn(f[4], f[5]), h3 = __floats2bfloat162_rn(f[6], f[7]);
            uint4 u;
            u.x = *reinterpret_cast<uint32_t*>(&h0); u.y = *reinterpret_cast<uint32_t*>(&h1);
            u.z = *reinterpret_cast<uint32_t*>(&h2); u.w = *reinterpret_cast<uint32_t*>(&h3);
            *reinterpret_cast<uint4*>(stg + lane * 64 + ((((q >> 3) ^ (lane >> 1)) & 3) << 4)) = u;
          }
          __syncwarp();
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int row = k * 8 + (lane >> 2);
            const uint4 u = *reinterpret_cast<const uint4*>(stg + row * 64 + (((piece ^ (row >> 1)) & 3) << 4));
            if (rowok[k] && col0 + piece * 8 < p.Cout) *reinterpret_cast<uint4*>(rowp[k] + col0 + piece * 8) = u;
          }
          __syncwarp();                                // the staging tile is rewritten by the next chunk
        }
      } else {
#pragma unroll 1
      for (int c0 = part * CPW; c0 < (part + 1) * CPW; c0 += 32) {
        uint32_t v[32];
        bw::tmem_ld_32x32(tmem_base + ((uint32_t)(ew * 32) << 16) + as * BN + c0, v);
        bw::tmem_ld_wait();
        const int col0 = nb * BN + c0;
        if (row_ok && col0 < p.Cout) {
#pragma unroll
          for (int q = 0; q < 32; q += 8) {
            if (col0 + q >= p.Cout) break;
            float f[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) f[e] = __uint_as_float(v[q + e]);
            if (bias) {
              float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + col0 + q));
              float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + col0 + q + 4));
              f[0] += b0.x; f[1] += b0.y; f[2] += b0.z; f[3] += b0.w;
              f[4] += b1.x; f[5] += b1.y; f[6] += b1.z; f[7] += b1.w;
            }
            if (ACT == DGTD_ACT_RELU) {
#pragma unroll
              for (int e = 0; e < 8; ++e) f[e] = fmaxf(f[e], 0.f);
            }
            store4(orow + col0 + q, f[0], f[1], f[2], f[3]);
            store4(orow + col0 + q + 4, f[4], f[5], f[6], f[7]);
          }
        }
      }
      }
      bw::tc_fence_before();
      bw::mbar_arrive(&tempty[as]);
    }
  }

  bw::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    bw::tc_fence_after();
    bw::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------------
// 3x3 / stride 1 / pad 1 variant (decoder conv1, conv2 and the identity-grid conv3): ONE halo tile per
// output tile.  The per-tap kernel above re-reads the input nine times from L2 (9 x 8 KB of A per 128
// output pixels); with only 32 output channels per group that makes the grouped decoder convs L2-feed
// bound.  Here the tile is 16 rows x 8 pixels and the producer loads the (16+2) x (8+2) pixel halo once
// (11.25 KB, 64B-swizzled, zero fill = padding).  The A operand of tap (dy,dx) is the SAME shared-memory
// tile read through a descriptor that starts (dy*10 + dx) pixels further and strides 10 pixels (640 B)
// between 8-row groups: the 128 MMA rows (j, i) = (row, pixel) land on halo pixel (j+dy, i+dx).
// The nine weight tiles of a (group, n-block) stay resident (double buffered across group changes);
// tiles are ordered so that a CTA changes (group, n-block) at most groups*tiles_n times.
constexpr int HALO_TW = 8, HALO_TH = 16, HALO_PW = HALO_TW + 2, HALO_PH = HALO_TH + 2;
constexpr int HALO_BYTES = HALO_PH * HALO_PW * 64;          // 11520
constexpr int HALO_STAGE = 12288;                           // 1024-aligned slot

template <int BN>
struct HaloCfg {
  static constexpr int W_BYTES = 9 * BN * 64;               // all taps of one (group, n-block)
  static constexpr int STAGES = BN >= 128 ? 4 : 8;
  static constexpr int TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;
  // epilogue warps: 4 (one per TMEM lane quadrant) for the 32-column tiles, whose single chunk is not worth splitting;
  // 8 (two per quadrant, half of the columns each) from 64 columns up -- with 4 warps the N = 128 conv1 of the decoder
  // bank ran the tensor-core pipe at 38 %: one warp per scheduler, every TMEM load / bias load / store latency exposed
  static constexpr int NEPI = BN >= 64 ? 8 : 4;
  static constexpr int STG_BYTES = NEPI * 2 * 2048;         // per epilogue warp: two 32-row x 64-byte staging tiles
  static constexpr int SMEM_BYTES = STAGES * HALO_STAGE + 2 * W_BYTES + STG_BYTES + 256 + 1024;
};

// K-major 64B-swizzle descriptor with an explicit 8-row-group pitch.  The start address is only 64-byte
// aligned (one pixel), not aligned to the 512-byte swizzle pattern: measured on B200, the MMA unit applies
// the XOR pattern to the absolute shared-memory address bits, i.e. exactly what TMA wrote, so the
// descriptor's base_offset field stays 0 (setting it to (addr >> 7) & 7 gives wrong results).
__device__ __forceinline__ uint64_t halo_desc(uint32_t addr, uint32_t sbo_bytes) {
  return (uint64_t)((addr >> 4) & 0x3FFF) | ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46) | (4ull << 61);
}

template <int BN, int ACT, typename OT>
__global__ void __launch_bounds__(128 + 32 * HaloCfg<BN>::NEPI, 1)
tc_conv_halo_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW,
                    const __grid_constant__ CUtensorMap tmO, const ConvParams p) {
  using Cfg = HaloCfg<BN>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sA = smem;
  uint8_t* sW = smem + STAGES * HALO_STAGE;
  uint8_t* sStg = smem + STAGES * HALO_STAGE + 2 * Cfg::W_BYTES;      // 1024-aligned (all sizes above are)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sStg + Cfg::STG_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + STAGES;
  uint64_t* tfull = bars + 2 * STAGES;
  uint64_t* tempty = bars + 2 * STAGES + 2;
  uint64_t* wfull = bars + 2 * STAGES + 4;
  uint64_t* wempty = bars + 2 * STAGES + 6;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 8);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles_img = p.tiles_x * p.tiles_y;
  const int per_key = p.B * tiles_img;                      // tiles sharing one (group, n-block)
  // Work assignment: a CTA owns ONE (group, n-block) key (its nine weight tiles are loaded once) and walks the
  // images in order together with the CTAs of the other keys, so that the pixel rows of an image -- which
  // interleave the channel slices of all groups -- are consumed by all groups while they are in L2.
  const int keys = p.groups * p.tiles_n;
  const int kmod = keys < (int)gridDim.x ? keys : (int)gridDim.x;    // keys in flight
  const int nct = keys < (int)gridDim.x ? (int)gridDim.x / keys : 1; // CTAs sharing a key
  const int key0 = (int)blockIdx.x % kmod, ci = (int)blockIdx.x / kmod;
  const int per_cta = ci < nct ? (per_key - ci + nct - 1) / nct : 0;   // positions of a key walked by this CTA
  // Division-free walk (the single producer / MMA threads are latency chains: a handful of integer divisions per
  // tile cost more than the eighteen MMAs of a 32-column tile): position pos = ci + tt*nct within a key,
  // (tx, ty, b) advanced incrementally.
  struct Walk {
    int key, g, nb, tt, tx, ty, b;
  };
  auto walk_begin = [&](Walk& wk, int key) {
    wk.key = key; wk.g = key / p.tiles_n; wk.nb = key - wk.g * p.tiles_n; wk.tt = 0;
    wk.tx = ci % p.tiles_x;
    const int r = ci / p.tiles_x;
    wk.ty = r % p.tiles_y; wk.b = r / p.tiles_y;
  };
  auto walk_next = [&](Walk& wk) {
    ++wk.tt;
    wk.tx += nct;
    while (wk.tx >= p.tiles_x) { wk.tx -= p.tiles_x; if (++wk.ty == p.tiles_y) { wk.ty = 0; ++wk.b; } }
  };

  if (warp == 0 && lane == 0) {
    bw::prefetch_tmap(&tmX);
    bw::prefetch_tmap(&tmW);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) {
      bw::mbar_init(&full[i], 1);
      bw::mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      bw::mbar_init(&tfull[i], 1);
      bw::mbar_init(&tempty[i], 32 * Cfg::NEPI);
      bw::mbar_init(&wfull[i], 1);
      bw::mbar_init(&wempty[i], 1);
    }
    bw::fence_mbar_init();
  }
  if (warp == 2) bw::tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  bw::tc_fence_before();
  __syncthreads();
  bw::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0, wcount = 0;
      uint32_t phase = 0;
      Walk wk;
      for (int key = key0; key < keys && per_cta > 0; key += kmod) {
        walk_begin(wk, key);
        {   // the nine weight tiles of this (group, n-block) into the other buffer
          const int buf = wcount & 1;
          bw::mbar_wait(&wempty[buf], ((wcount >> 1) & 1) ^ 1);
          bw::mbar_arrive_expect_tx(&wfull[buf], Cfg::W_BYTES);
#pragma unroll 1
          for (int t = 0; t < 9; ++t)
            bw::tma_load_2d(&tmW, &wfull[buf], sW + buf * Cfg::W_BYTES + t * BN * 64, t * 32,
                            wk.g * p.w_group_rows + wk.nb * BN);
          ++wcount;
        }
        for (; wk.tt < per_cta; walk_next(wk)) {
          bw::mbar_wait(&empty[stage], phase ^ 1);
          bw::mbar_arrive_expect_tx(&full[stage], HALO_BYTES);
          if (p.x5d)
            bw::tma_load_5d(&tmX, &full[stage], sA + stage * HALO_STAGE, 0, wk.tx * HALO_TW - 1, wk.ty * HALO_TH - 1,
                            wk.b, wk.g);
          else
            bw::tma_load_4d(&tmX, &full[stage], sA + stage * HALO_STAGE, wk.g * 32, wk.tx * HALO_TW - 1,
                            wk.ty * HALO_TH - 1, wk.b);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = bw::umma_idesc_bf16(128, BN);
      int stage = 0, iter = 0, wcount = 0, buf = 0;
      uint32_t phase = 0;
      const uint64_t da_base = halo_desc(bw::smem_u32(sA), HALO_PW * 64);
      const uint64_t db_base = bw::umma_smem_desc_kmajor(bw::smem_u32(sW), 64);
      for (int key = key0; key < keys && per_cta > 0; key += kmod) {
        if (wcount > 0) bw::umma_commit(&wempty[buf]);   // previous weights free once their MMAs retire
        buf = wcount & 1;
        bw::mbar_wait(&wfull[buf], (wcount >> 1) & 1);
        ++wcount;
        const uint64_t db0 = db_base + (uint64_t)((buf * Cfg::W_BYTES) >> 4);
        for (int tt = 0; tt < per_cta; ++tt, ++iter) {
          const int as = iter & 1;
          const uint32_t aphase = (iter >> 1) & 1;
          bw::mbar_wait(&tempty[as], aphase ^ 1);
          bw::tc_fence_after();
          const uint32_t d_tmem = tmem_base + as * BN;
          bw::mbar_wait(&full[stage], phase);
          bw::tc_fence_after();
          const uint64_t da0 = da_base + (uint64_t)((stage * HALO_STAGE) >> 4);
#pragma unroll
          for (int t = 0; t < 9; ++t) {
            const int dy = t / 3, dx = t - 3 * dy;
            const uint64_t da = da0 + (uint64_t)(((dy * HALO_PW + dx) * 64) >> 4);   // descriptor address field: 16-byte units
            const uint64_t db = db0 + (uint64_t)((t * BN * 64) >> 4);
#pragma unroll
            for (int k = 0; k < 2; ++k) bw::umma_bf16(d_tmem, da + 2 * k, db + 2 * k, idesc, (t | k) != 0);
          }
          bw::umma_commit(&empty[stage]);
          bw::umma_commit(&tfull[as]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp >= 4) {
    const int ew = (warp - 4) & 3, part = (warp - 4) >> 2;   // TMEM lane quadrant (= warp % 4), column half
    constexpr int CPW = BN / (Cfg::NEPI / 4);                // columns per epilogue warp
    int iter = 0;
    uint32_t sbuf = 0;
    Walk wk;
    for (int key = key0; key < keys && per_cta > 0; key += kmod)
    for (walk_begin(wk, key); wk.tt < per_cta; walk_next(wk), ++iter) {
      const int g = wk.g, b = wk.b, ty = wk.ty, tx = wk.tx, nb = wk.nb;
      const int as = iter & 1;
      const uint32_t aphase = (iter >> 1) & 1;
      bw::mbar_wait(&tfull[as], aphase);
      bw::tc_fence_after();
      const int r = ew * 32 + lane;                 // MMA row = (j, i): image row j, pixel i of the 16 x 8 tile
      const int j = r >> 3, i = r & 7;
      const int oy = ty * HALO_TH + j, ox = tx * HALO_TW + i;
      const bool row_ok = oy < p.oh && ox < p.ow;
      const float* bias = p.bias ? p.bias + g * p.w_group_rows : nullptr;
      if (sizeof(OT) == 2) {
        // bf16 results leave through a 64B-swizzled staging tile (32 rows = 4 image rows x 8 pixels, 64 B each)
        // and ONE 5-D TMA store per 32 channels: full lines instead of 32 scattered 8-byte stores per lane;
        // the tensor map clips tile rows / channels beyond the image.
        uint8_t* stg = sStg + (warp - 4) * 4096;
#pragma unroll 1
        for (int c0 = part * CPW; c0 < (part + 1) * CPW; c0 += 32) {
          uint32_t v[32];
          bw::tmem_ld_32x32(tmem_base + ((uint32_t)(ew * 32) << 16) + as * BN + c0, v);
          bw::tmem_ld_wait();
          const int col0 = nb * BN + c0;
          if (col0 >= p.Cout) break;
          uint8_t* buf = stg + (sbuf & 1) * 2048;
          if (lane == 0) bw::tma_store_wait_read<1>();   // the store that last read this buffer (two commits ago)
          __syncwarp();
#pragma unroll
          for (int q = 0; q < 32; q += 8) {
            float f[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) f[e] = __uint_as_float(v[q + e]);
            if (bias && col0 + q < p.Cout) {
              float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + col0 + q));
              float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + col0 + q + 4));
              f[0] += b0.x; f[1] += b0.y; f[2] += b0.z; f[3] += b0.w;
              f[4] += b1.x; f[5] += b1.y; f[6] += b1.z; f[7] += b1.w;
            }
            if (ACT == DGTD_ACT_RELU) {
#pragma unroll
              for (int e = 0; e < 8; ++e) f[e] = fmaxf(f[e], 0.f);
            }
            __nv_bfloat162 h0 = __floats2bfloat162_rn(f[0], f[1]), h1 = __floats2bfloat162_rn(f[2], f[3]);
            __nv_bfloat162 h2 = __floats2bfloat162_rn(f[4], f[5]), h3 = __floats2bfloat162_rn(f[6], f[7]);
            uint4 u;
            u.x = *reinterpret_cast<uint32_t*>(&h0); u.y = *reinterpret_cast<uint32_t*>(&h1);
            u.z = *reinterpret_cast<uint32_t*>(&h2); u.w = *reinterpret_cast<uint32_t*>(&h3);
            // 16-byte chunk (q/8) of row `lane` lives at chunk (q/8) ^ ((lane >> 1) & 3) of the 64-byte row
            *reinterpret_cast<uint4*>(buf + lane * 64 + ((((q >> 3) ^ (lane >> 1)) & 3) << 4)) = u;
          }
          bw::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (p.out_split) bw::tma_store_5d(&tmO, buf, 0, tx * HALO_TW, ty * HALO_TH + ew * 4, b, col0 >> 5);
            else bw::tma_store_5d(&tmO, buf, col0, tx * HALO_TW, ty * HALO_TH + ew * 4, b, g);
            bw::tma_store_commit();
          }
          ++sbuf;
        }
      } else {
        OT* orow = reinterpret_cast<OT*>(p.out) + (int64_t)g * p.out_group_stride +
                   (((int64_t)b * p.oh + oy) * p.ow + ox) * p.ldo;
#pragma unroll 1
        for (int c0 = part * CPW; c0 < (part + 1) * CPW; c0 += 32) {
          uint32_t v[32];
          bw::tmem_ld_32x32(tmem_base + ((uint32_t)(ew * 32) << 16) + as * BN + c0, v);
          bw::tmem_ld_wait();
          const int col0 = nb * BN + c0;
          if (row_ok && col0 < p.Cout) {
#pragma unroll
            for (int q = 0; q < 32; q += 8) {
              if (col0 + q >= p.Cout) break;
              float f[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) f[e] = __uint_as_float(v[q + e]);
              if (bias) {
                float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + col0 + q));
                float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + col0 + q + 4));
                f[0] += b0.x; f[1] += b0.y; f[2] += b0.z; f[3] += b0.w;
                f[4] += b1.x; f[5] += b1.y; f[6] += b1.z; f[7] += b1.w;
              }
              if (ACT == DGTD_ACT_RELU) {
#pragma unroll
                for (int e = 0; e < 8; ++e) f[e] = fmaxf(f[e], 0.f);
              }
              store4(orow + col0 + q, f[0], f[1], f[2], f[3]);
              store4(orow + col0 + q + 4, f[4], f[5], f[6], f[7]);
            }
          }
        }
      }
      bw::tc_fence_before();
      bw::mbar_arrive(&tempty[as]);
    }
    if (sizeof(OT) == 2 && lane == 0) bw::tma_store_wait_all<0>();   // results are in global memory before exit
  }

  bw::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    bw::tc_fence_after();
    bw::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

template <int BN, int ACT, typename OT>
static int conv_halo_launch(const void* x, int B, int h, int wd, int ldx, int64_t xgs, const __nv_bfloat16* w, int Wrows,
                            ConvParams p, cudaStream_t s) {
  using Cfg = HaloCfg<BN>;
  auto kern = tc_conv_halo_kernel<BN, ACT, OT>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) {
      set_error("tc_conv(halo): cannot opt in to %d B of shared memory: %s", Cfg::SMEM_BYTES, cudaGetErrorString(e));
      return -2;
    }
    configured = true;
  }
  CUtensorMap tmX, tmW;
  {
    uint64_t dims[4] = {(uint64_t)ldx, (uint64_t)wd, (uint64_t)h, (uint64_t)B};
    uint64_t str[3] = {(uint64_t)ldx * 2, (uint64_t)wd * ldx * 2, (uint64_t)h * wd * ldx * 2};
    uint32_t box[4] = {32, HALO_PW, HALO_PH, 1};
    int rc;
    if (p.x5d) {   // group-major: every group is a dense (B, h, w, 32) tensor, xgs elements apart
      uint64_t dims5[5] = {32, (uint64_t)wd, (uint64_t)h, (uint64_t)B, (uint64_t)p.groups};
      uint64_t str5[4] = {(uint64_t)ldx * 2, (uint64_t)wd * ldx * 2, (uint64_t)h * wd * ldx * 2, (uint64_t)xgs * 2};
      uint32_t box5[5] = {32, HALO_PW, HALO_PH, 1, 1};
      rc = make_tmap(&tmX, x, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, dims5, str5, box5, CU_TENSOR_MAP_SWIZZLE_64B);
    } else {
      rc = make_tmap(&tmX, x, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B);
    }
    if (rc) return rc;
  }
  {
    uint64_t dims[2] = {(uint64_t)288, (uint64_t)Wrows}, str[1] = {(uint64_t)288 * 2};
    uint32_t box[2] = {32, (uint32_t)BN};
    int rc = make_tmap(&tmW, w, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B);
    if (rc) return rc;
  }
  CUtensorMap tmO = tmW;
  if (sizeof(OT) == 2) {
    uint64_t dims[5] = {(uint64_t)(p.out_split ? 32 : p.Cout), (uint64_t)p.ow, (uint64_t)p.oh, (uint64_t)p.B,
                        (uint64_t)(p.out_split ? p.Cout / 32 : p.groups)};
    uint64_t str[4] = {(uint64_t)p.ldo * 2, (uint64_t)p.ow * p.ldo * 2, (uint64_t)p.oh * p.ow * p.ldo * 2,
                       (uint64_t)(p.groups > 1 || p.out_split ? p.out_group_stride : (int64_t)p.B * p.oh * p.ow * p.ldo) * 2};
    uint32_t box[5] = {32, HALO_TW, 4, 1, 1};
    int rc = make_tmap(&tmO, p.out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B);
    if (rc) return rc;
  }
  p.TW = HALO_TW; p.TH = HALO_TH;
  p.tiles_x = cdiv(p.ow, HALO_TW);
  p.tiles_y = cdiv(p.oh, HALO_TH);
  p.tiles_n = cdiv(p.Cout, BN);
  const int keys = p.groups * p.tiles_n;
  const int64_t per_key = (int64_t)p.B * p.tiles_x * p.tiles_y;
  int nct = keys < sm_count() ? sm_count() / keys : 1;
  if (nct > per_key) nct = (int)per_key;
  const int grid = keys < sm_count() ? keys * nct : sm_count();
  kern<<<grid, 128 + 32 * Cfg::NEPI, Cfg::SMEM_BYTES, s>>>(tmX, tmW, tmO, p);
  return 0;
}

template <int ACT, typename OT>
static int conv_halo_dispatch_bn(const void* x, int B, int h, int wd, int ldx, int64_t xgs, const __nv_bfloat16* w, int Wrows,
                                 const ConvParams& p, cudaStream_t s) {
  if (p.Cout <= 32) return conv_halo_launch<32, ACT, OT>(x, B, h, wd, ldx, xgs, w, Wrows, p, s);
  if (p.Cout <= 64) return conv_halo_launch<64, ACT, OT>(x, B, h, wd, ldx, xgs, w, Wrows, p, s);
  return conv_halo_launch<128, ACT, OT>(x, B, h, wd, ldx, xgs, w, Wrows, p, s);
}

static void pick_tile(int ow, int oh, int stride, int& TW, int& TH) {
  int lim = 256 / stride;
  if (lim > 32) lim = 32;
  TW = ow < lim ? ow : lim;
  for (int d = TW; d >= 8; --d)
    if (ow % d == 0) { TW = d; break; }
  TH = 128 / TW;
  if (TH > oh) TH = oh;
  if (TH * stride > 256) TH = 256 / stride;
}

template <int BN, int ACT, typename OT>
static int conv_launch(const CUtensorMap& tmX, const __nv_bfloat16* w, int Ktot, int Wrows, ConvParams p,
                       cudaStream_t s) {
  using Cfg = ConvCfg<BN>;
  auto kern = tc_conv_kernel<BN, ACT, OT>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) {
      set_error("tc_conv: cannot opt in to %d B of shared memory: %s", Cfg::SMEM_BYTES, cudaGetErrorString(e));
      return -2;
    }
    configured = true;
  }
  CUtensorMap tmW;
  uint64_t dims[2] = {(uint64_t)Ktot, (uint64_t)Wrows}, str[1] = {(uint64_t)Ktot * 2};
  uint32_t box[2] = {32, (uint32_t)BN};
  int rc = make_tmap(&tmW, w, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_64B);
  if (rc) return rc;
  p.tiles_n = cdiv(p.Cout, BN);
  {   // resident weights: one (group, n-block) key per CTA, when every key gets at least one CTA and all taps fit
    using Rw = ConvRwCfg<BN>;
    const int keys = p.groups * p.tiles_n;
    const int64_t per_key = (int64_t)p.B * p.tiles_x * p.tiles_y;
    if (BN >= 64 && keys <= sm_count() && p.ks * p.ks <= Rw::MAX_TAPS && per_key < (1ll << 31)) {
      auto kern_rw = tc_conv_resw_kernel<BN, ACT, OT>;
      static bool configured_rw = false;
      if (!configured_rw) {
        cudaError_t e = cudaFuncSetAttribute(kern_rw, cudaFuncAttributeMaxDynamicSharedMemorySize, Rw::SMEM_BYTES);
        if (e != cudaSuccess) {
          set_error("tc_conv(resident weights): cannot opt in to %d B of shared memory: %s", Rw::SMEM_BYTES,
                    cudaGetErrorString(e));
          return -2;
        }
        configured_rw = true;
      }
      int nct = sm_count() / keys;
      if (nct > per_key) nct = (int)per_key;
      kern_rw<<<keys * nct, 128 + 32 * Rw::NEPI, Rw::SMEM_BYTES, s>>>(tmX, tmW, p);
      return 0;
    }
  }
  int64_t tiles = (int64_t)p.groups * p.B * p.tiles_x * p.tiles_y * p.tiles_n;
  int grid = tiles < sm_count() ? (int)tiles : sm_count();
  kern<<<grid, 256, Cfg::SMEM_BYTES, s>>>(tmX, tmW, p);
  return 0;
}

template <int ACT, typename OT>
static int conv_dispatch_bn(const CUtensorMap& tmX, const __nv_bfloat16* w, int Ktot, int Wrows,
                            const ConvParams& p, cudaStream_t s) {
  if (p.Cout <= 32) return conv_launch<32, ACT, OT>(tmX, w, Ktot, Wrows, p, s);
  if (p.Cout <= 64) return conv_launch<64, ACT, OT>(tmX, w, Ktot, Wrows, p, s);
  return conv_launch<128, ACT, OT>(tmX, w, Ktot, Wrows, p, s);
}

// x: NHWC bf16, 32-channel slices per group (ldx >= 32*groups... or the caller's channel offset)
int tc_conv_nhwc(const void* x, const void* w, const float* bias, void* out, int B, int h, int wd, int Cin,
                 int ldx, int oh, int ow, int Cout, int ldo, int ks, int stride, int off, int act,
                 int dtype_out, int groups, int64_t x_group_stride, int w_group_rows, int64_t out_group_stride,
                 cudaStream_t s) {
  if (Cin != 32) {
    set_error("conv_nhwc(bf16): Cin must be padded to 32 channels per group (got %d)", Cin);
    return -1;
  }
  if (ldx % 8 || ldo % 8 || Cout % 8 || (reinterpret_cast<uintptr_t>(x) & 15)) {
    set_error("conv_nhwc(bf16): ldx, ldo, Cout must be multiples of 8 and x 16-byte aligned");
    return -1;
  }
  if (stride > 8 || ks > 4) {
    set_error("conv_nhwc(bf16): stride <= 8 and ks <= 4 only");
    return -1;
  }
  ConvParams p{};
  p.B = B; p.oh = oh; p.ow = ow; p.Cout = Cout; p.ldo = ldo; p.ks = ks; p.stride = stride; p.off = off;
  p.groups = groups; p.w_group_rows = w_group_rows; p.out_group_stride = out_group_stride;
  p.bias = bias; p.out = out;
  // group-major operands (round 2): x_group_stride != 32 = every group a dense (B, h, w, ldx) tensor; groups == 1 with
  // an out_group_stride and a pixel pitch ldo < Cout = the 32-channel chunks of the output scattered to dense (B, oh, ow, ldo) tensors
  p.x5d = groups > 1 && x_group_stride != 32;
  p.out_split = groups == 1 && out_group_stride > 0 && ldo < Cout;
  if (p.x5d && (x_group_stride % 8 || ldx < 32)) {
    set_error("conv_nhwc(bf16): x_group_stride must be a multiple of 8 elements");
    return -1;
  }
  const bool halo_ok = ks == 3 && stride == 1 && off == -1 && oh == h && ow == wd;
  if (p.out_split && !(halo_ok && dtype_out == DGTD_BF16 && Cout % 32 == 0)) {
    set_error("conv_nhwc(bf16): the chunk-scattered output needs the 3x3 stride-1 conv, bf16 output and Cout %% 32 == 0");
    return -1;
  }
  if (halo_ok) {
    const int Wrows = groups * w_group_rows;
    const __nv_bfloat16* wp = (const __nv_bfloat16*)w;
    if (dtype_out == DGTD_BF16) {
      if (act == DGTD_ACT_RELU) return conv_halo_dispatch_bn<DGTD_ACT_RELU, __nv_bfloat16>(x, B, h, wd, ldx, x_group_stride, wp, Wrows, p, s);
      return conv_halo_dispatch_bn<DGTD_ACT_NONE, __nv_bfloat16>(x, B, h, wd, ldx, x_group_stride, wp, Wrows, p, s);
    }
    if (act == DGTD_ACT_RELU) return conv_halo_dispatch_bn<DGTD_ACT_RELU, float>(x, B, h, wd, ldx, x_group_stride, wp, Wrows, p, s);
    return conv_halo_dispatch_bn<DGTD_ACT_NONE, float>(x, B, h, wd, ldx, x_group_stride, wp, Wrows, p, s);
  }
  pick_tile(ow, oh, stride, p.TW, p.TH);
  p.tiles_x = cdiv(ow, p.TW);
  p.tiles_y = cdiv(oh, p.TH);
  CUtensorMap tmX;
  {
    // dims innermost first: channels (all groups), W, H, B
    const int rank = p.x5d ? 5 : 4;
    uint64_t dims[5] = {(uint64_t)(p.x5d ? 32 : ldx), (uint64_t)wd, (uint64_t)h, (uint64_t)B, (uint64_t)groups};
    uint64_t str[4] = {(uint64_t)ldx * 2, (uint64_t)wd * ldx * 2, (uint64_t)h * wd * ldx * 2, (uint64_t)x_group_stride * 2};
    uint32_t box[5] = {32, (uint32_t)(p.TW * stride), (uint32_t)(p.TH * stride), 1, 1};
    PFN_tmapEncodeTiled enc = get_tmap_encoder();
    if (!enc) return -3;
    cuuint64_t gd[5], gs[4];
    cuuint32_t bx[5], es[5] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1, 1};
    for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; }
    for (int i = 0; i < rank - 1; ++i) gs[i] = str[i];
    CUresult r = enc(&tmX, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(x), gd, gs, bx, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_error("conv_nhwc(bf16): cuTensorMapEncodeTiled(x) failed (%d): dims=[%d,%d,%d,%d] box=[32,%d,%d,1] stride %d",
                (int)r, ldx, wd, h, B, p.TW * stride, p.TH * stride, stride);
      return -3;
    }
  }
  const int Ktot = ks * ks * 32;
  const int Wrows = groups * w_group_rows;
  const __nv_bfloat16* wp = (const __nv_bfloat16*)w;
  if (dtype_out == DGTD_BF16) {
    if (act == DGTD_ACT_RELU) return conv_dispatch_bn<DGTD_ACT_RELU, __nv_bfloat16>(tmX, wp, Ktot, Wrows, p, s);
    return conv_dispatch_bn<DGTD_ACT_NONE, __nv_bfloat16>(tmX, wp, Ktot, Wrows, p, s);
  }
  if (act == DGTD_ACT_RELU) return conv_dispatch_bn<DGTD_ACT_RELU, float>(tmX, wp, Ktot, Wrows, p, s);
  return conv_dispatch_bn<DGTD_ACT_NONE, float>(tmX, wp, Ktot, Wrows, p, s);
}

}  // namespace dgtd
