// a6 at microbench scale (BASELINE configs[3]: 1024 x 1024 x 256, k = 7), shared weights (wc == 1), on the
// TENSOR pipe: MessagePassing.forward core (cod.py:1190-1205) as a banded GEMM per 8 x 16 pixel tile.
//
//   Y[128 px, C] = A[128 px, 336 halo px] . X[336 halo px, C]
//
// A row p = (py, px) holds the 49 random-walk-normalised weights of pixel p (W / (sum W + eps), cod.py:1201)
// at the columns k = (py + ky) * 24 + (px + kx) of its 7 x 7 neighbourhood inside the tile's 14 x 24 halo window
// (22 wide + 2 so that a halo row is 1.5 MMA K steps and two rows are exactly 3), zero elsewhere.  The
// SIMT formulation of this operator (mp_tiled.cu) is bound by shared-memory broadcast wavefronts at 35 % of the
// FMA roof (DESIGN.md section 9); here the per-pixel weights are written ONCE per tile into the A operand and all
// C channels go through tcgen05.mma: 6.9x the useful FLOPs are executed, at ~30x the rate.
//
// bf16 storage (this file, `mp_tc_kernel`):
//   * X needs no preparation: the channels of a pixel are contiguous in HBM (NHWC), i.e. X is an MN-major B
//     operand.  One 4-D TMA box {64 ch, 24 px, 2 rows} per 64-channel block lands as 48 K rows x 128 B in the
//     SWIZZLE_128B layout tcgen05.mma reads (zero fill outside the map == unfold's zero padding, cod.py:1204).
//   * A is bf16 (kind::f16 wants both operands in ONE 16-bit format: an fp16 A against the bf16 X is an illegal
//     instruction on sm_100a -- measured), K-major SWIZZLE_32B, RESIDENT in shared memory as seven 2-halo-row
//     chunks (7 x 12 KB): the zero pattern of a row never changes, so per tile a builder thread (one per pixel)
//     only overwrites its 49 non-zeros.  Rounding the normalised weights to bf16 adds a zero-mean 2^-9 relative
//     error per tap, i.e. ~2.5e-4 of max|y| after the 49-tap sum -- below the bf16 rounding of the stored result
//     (2^-9 of the element) that bf16 storage implies anyway; stated tolerance 6e-3 of max|ref| per step.
//   * per tile: 7 chunks x 3 MMAs (M 128, N 256, K 16) into one of two 256-column TMEM accumulators; the
//     epilogue of tile i (tcgen05.ld -> bf16 -> swizzled staging -> 4-D TMA store) overlaps the MMAs of tile i+1.
// Warp roles (384 threads, 1 CTA / SM, persistent over tiles): w0 TMA producer, w1 MMA issuer, w2 TMEM
// allocator, w4-7 epilogue (one TMEM lane quadrant = two tile rows each), w8-11 A builders.
// Algorithmic HBM traffic per step: (2 * C * 2 + 49 * 4) * H * W bytes; executed MMA work 2 * 336 * C per pixel.
#include "blackwell.cuh"
#include "common.cuh"

namespace dgtd {
int sm_count();   // tc_gemm.cu

namespace mptc {

constexpr int TH = 8, TW = 16;                 // output tile = 128 pixels = the M of one MMA
constexpr int PW = 24, PH = 14;                // halo window (22 -> 24 columns), K = 336
constexpr int NCHUNK = 7, CK = 48;             // chunk = 2 halo rows = 48 K rows = 3 K steps
constexpr int XBLK = CK * 128;                 // 64-channel block of a chunk: 48 K rows x 128 B
constexpr int NB = 256;                        // channels per pass (N of the MMA)
constexpr int X_STAGE = (NB / 64) * XBLK;      // 24 KB
constexpr int STG = 4 * 4096;                  // 4 epilogue warps x one staging tile (32 px x 128 B)
constexpr int THREADS = 384;

// Shared-memory budget.  The kernel is bound by how many bytes of X it keeps in flight (r2 profile: 72 KB per SM at
// ~2.8 us of loaded TMA latency = 3.8 TB/s of L2->SM traffic, tensor pipe 24 % busy), so every KB not spent elsewhere
// is a KB of X prefetch.  The A (weights) operand is SWIZZLE_32B K-major: one 4 KB block of 128 rows x 32 B (16 K
// columns) per K step, so a chunk takes 12 KB with no padding bytes, which leaves room for 5 X stages.
// RAWTMA (taken when w % 4 == 0, see mp_tc_step_bf16): the 49 raw weights of the tile's pixels arrive as ONE TMA box
// {16 px, 8 rows, 49 taps} (25 KB, warp 3) instead of 49 global loads per builder thread, and the slot costs one X
// stage (4 stages).  fence.proxy.async compiles to MEMBAR.ALL.CTA + FENCE.VIEW.ASYNC and the membar waits for every
// outstanding global load of the thread: with register prefetch the first publish of every tile stalled for a DRAM
// round trip (r2 profile: builder ~7900 cycles per tile against 2688 cycles of MMAs).
constexpr int W_BYTES = 49 * TH * TW * 4, W_SLOT = 25600;
template <bool RAWTMA>
struct Cfg {
  static constexpr int A_CHUNK = 3 * 128 * 32;
  static constexpr int XSTAGES = RAWTMA ? 4 : 5;
  static constexpr int OFF_X = NCHUNK * A_CHUNK;
  static constexpr int OFF_STG = OFF_X + XSTAGES * X_STAGE;
  static constexpr int OFF_W = OFF_STG + STG;
  static constexpr int OFF_BAR = OFF_W + (RAWTMA ? W_SLOT : 0);
  static constexpr int NBARS = 2 * XSTAGES + 2 * NCHUNK + 4 + 2;
  static constexpr int SMEM = OFF_BAR + NBARS * 8 + 16 + 1024;   // + alignment slack
  // byte offset of element (row m, chunk-local column kl) inside a chunk
  static __device__ __forceinline__ uint32_t a_off(uint32_t m, uint32_t kl) {
    return (kl >> 4) * 4096 + m * 32 + (((((kl >> 3) & 1)) ^ ((m >> 2) & 1)) << 4) + ((kl & 7) << 1);
  }
  // descriptor of K step k of chunk j, relative to the descriptor of the ring's first byte
  static __device__ __forceinline__ uint64_t a_desc_off(int j, int k) {
    return (uint64_t)((j * A_CHUNK + 4096 * k) >> 4);
  }
};

__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(bw::smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}

// kind::f16 instruction descriptor: fp32 accumulate, A = bf16 K-major, B = bf16 MN-major, M 128 x N 256.
__host__ __device__ constexpr uint32_t idesc() {
  return (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(NB >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

struct Params {
  const float* weight;   // (n, 49, h, w)
  int n, h, w, C;
  int tiles_x, tiles_y, num_tiles;
  float eps;
};

template <bool RAWTMA>
__global__ void __launch_bounds__(THREADS, 1)
mp_tc_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmOut,
             const __grid_constant__ CUtensorMap tmW, const Params p) {
  using C = Cfg<RAWTMA>;
  constexpr int A_CHUNK = C::A_CHUNK, XSTAGES = C::XSTAGES, OFF_X = C::OFF_X, OFF_STG = C::OFF_STG, OFF_BAR = C::OFF_BAR;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;
  uint8_t* sX = smem + OFF_X;
  uint8_t* sStg = smem + OFF_STG;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint64_t* x_full = bars;
  uint64_t* x_empty = bars + XSTAGES;
  uint64_t* a_full = bars + 2 * XSTAGES;
  uint64_t* a_empty = a_full + NCHUNK;
  uint64_t* t_full = a_empty + NCHUNK;
  uint64_t* t_empty = t_full + 2;
  uint64_t* w_full = t_empty + 2;
  uint64_t* w_empty = w_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w_empty + 1);
  float* sW = reinterpret_cast<float*>(smem + C::OFF_W);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nblk = p.C / NB;

  // the A ring starts as all zeros; only the static non-zero pattern is ever rewritten
  for (int i = threadIdx.x; i < NCHUNK * A_CHUNK / 16; i += THREADS)
    reinterpret_cast<uint4*>(sA)[i] = make_uint4(0u, 0u, 0u, 0u);
  if (warp == 0 && lane == 0) {
    bw::prefetch_tmap(&tmX);
    bw::prefetch_tmap(&tmOut);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < XSTAGES; ++i) {
      bw::mbar_init(&x_full[i], 1);
      bw::mbar_init(&x_empty[i], 1);
    }
    for (int i = 0; i < NCHUNK; ++i) {
      bw::mbar_init(&a_full[i], 128);   // every builder thread arrives once per tile
      bw::mbar_init(&a_empty[i], 1);    // tcgen05.commit of the tile's last pass
    }
    for (int i = 0; i < 2; ++i) {
      bw::mbar_init(&t_full[i], 1);
      bw::mbar_init(&t_empty[i], 128);  // every epilogue thread
    }
    bw::mbar_init(w_full, 1);
    bw::mbar_init(w_empty, 128);        // every builder thread, once it has read its 49 raw weights
    bw::fence_mbar_init();
  }
  if (warp == 2) bw::tmem_alloc(tmem_slot, 512);
  bw::fence_proxy_async_smem();
  bw::tc_fence_before();
  __syncthreads();
  bw::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer: X halo rows, 2 at a time =====================
    // The whole warp walks the loop (warp-uniform control flow: no divergence bookkeeping around the uniform-datapath
    // TMA instructions); one elected lane issues.
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t x_base = bw::smem_u32(sX);
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      int t = tile;
      const int tx = t % p.tiles_x; t /= p.tiles_x;
      const int ty = t % p.tiles_y;
      const int img = t / p.tiles_y;
      const int x0 = tx * TW - 3, y0 = ty * TH - 3;
      for (int nb = 0; nb < nblk; ++nb) {
#pragma unroll 1
        for (int j = 0; j < NCHUNK; ++j) {
          bw::mbar_wait(&x_empty[stage], phase ^ 1);
          if (bw::elect_one()) {
            bw::mbar_arrive_expect_tx(&x_full[stage], X_STAGE);
            uint8_t* dst = sX + stage * X_STAGE;
#pragma unroll
            for (int b = 0; b < NB / 64; ++b)
              bw::tma_load_4d(&tmX, &x_full[stage], dst + b * XBLK, nb * NB + 64 * b, x0, y0 + 2 * j, img);
          }
          __syncwarp();
          if (++stage == XSTAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
    (void)x_base;
  } else if (warp == 3) {
    if (RAWTMA) {
      // ===================== raw weights of the next tile: one TMA box per tile =====================
      uint32_t tcount = 0;
      for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++tcount) {
        int t = tile;
        const int tx = t % p.tiles_x; t /= p.tiles_x;
        const int ty = t % p.tiles_y;
        const int img = t / p.tiles_y;
        bw::mbar_wait(w_empty, (tcount & 1) ^ 1);
        if (bw::elect_one()) {
          bw::mbar_arrive_expect_tx(w_full, W_BYTES);
          bw::tma_load_4d(&tmW, w_full, sW, tx * TW, ty * TH, 0, img);
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp in the loop, one elected lane issues) =====================
    // 21 MMAs of 128 clocks per tile: the loop around them must stay well under 384 clocks per chunk, so the
    // descriptors are precomputed and the chunk loop is unrolled (r2 profile: the first version spent 2/3 of the
    // issuing warp's time on loop overhead and ran the tensor pipe at 24 %).
    constexpr uint32_t IDESC = idesc();
    const uint64_t da0 = bw::umma_smem_desc_kmajor(bw::smem_u32(sA), 32);
    const uint64_t db0 = bw::umma_smem_desc_mnmajor_sw128(bw::smem_u32(sX), XBLK, 1024);
    int stage = 0, iter = 0;
    uint32_t phase = 0, tphase = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, tphase ^= 1) {
      for (int nb = 0; nb < nblk; ++nb, ++iter) {
        const int as = iter & 1;
        bw::mbar_wait(&t_empty[as], ((iter >> 1) & 1) ^ 1);
        const uint32_t d_tmem = tmem_base + as * NB;
        const bool first = nb == 0, last = nb == nblk - 1;
#pragma unroll 1
        for (int j = 0; j < NCHUNK; ++j) {
          bw::mbar_wait(&x_full[stage], phase);
          if (first) bw::mbar_wait(&a_full[j], tphase);
          bw::tc_fence_after();
          if (bw::elect_one()) {
            const uint64_t db = db0 + (uint64_t)(stage * (X_STAGE >> 4));
#pragma unroll
            for (int k = 0; k < CK / 16; ++k)
              bw::umma_bf16(d_tmem, da0 + C::a_desc_off(j, k), db + 128u * k, IDESC, (j | k) != 0);
            bw::umma_commit(&x_empty[stage]);
            if (last) bw::umma_commit(&a_empty[j]);
            if (j == NCHUNK - 1) bw::umma_commit(&t_full[as]);
          }
          __syncwarp();
          if (++stage == XSTAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp >= 4 && warp < 8) {
    // ===================== epilogue: TMEM -> bf16 -> staging -> TMA store =====================
    const int quad = warp & 3;
    uint8_t* tl = sStg + quad * 4096;
    const uint32_t swz = (uint32_t)(lane & 7);
    int iter = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      int t = tile;
      const int tx = t % p.tiles_x; t /= p.tiles_x;
      const int ty = t % p.tiles_y;
      const int img = t / p.tiles_y;
      for (int nb = 0; nb < nblk; ++nb, ++iter) {
        const int as = iter & 1;
        bw::mbar_wait(&t_full[as], (iter >> 1) & 1);
        bw::tc_fence_after();
        const uint32_t t0 = tmem_base + ((uint32_t)(quad * 32) << 16) + as * NB;
#pragma unroll 1
        for (int c = 0; c < NB / 64; ++c) {
          uint32_t v[2][32];
          bw::tmem_ld_32x32(t0 + c * 64, v[0]);
          bw::tmem_ld_32x32(t0 + c * 64 + 32, v[1]);
          bw::tmem_ld_wait();
          if (c == NB / 64 - 1) {   // all TMEM reads of this accumulator have landed: hand it back
            bw::tc_fence_before();
            bw::mbar_arrive(&t_empty[as]);
          }
          if (lane == 0) bw::tma_store_wait_read<0>();   // the store that last read the staging tile is done
          __syncwarp();
#pragma unroll
          for (int hf = 0; hf < 2; ++hf)
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              uint4 u;
              __nv_bfloat162 b0 = __floats2bfloat162_rn(__uint_as_float(v[hf][8 * q + 0]), __uint_as_float(v[hf][8 * q + 1]));
              __nv_bfloat162 b1 = __floats2bfloat162_rn(__uint_as_float(v[hf][8 * q + 2]), __uint_as_float(v[hf][8 * q + 3]));
              __nv_bfloat162 b2 = __floats2bfloat162_rn(__uint_as_float(v[hf][8 * q + 4]), __uint_as_float(v[hf][8 * q + 5]));
              __nv_bfloat162 b3 = __floats2bfloat162_rn(__uint_as_float(v[hf][8 * q + 6]), __uint_as_float(v[hf][8 * q + 7]));
              u.x = *reinterpret_cast<uint32_t*>(&b0); u.y = *reinterpret_cast<uint32_t*>(&b1);
              u.z = *reinterpret_cast<uint32_t*>(&b2); u.w = *reinterpret_cast<uint32_t*>(&b3);
              *reinterpret_cast<uint4*>(tl + lane * 128 + ((((uint32_t)(hf * 4 + q)) ^ swz) << 4)) = u;
            }
          bw::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_4d(&tmOut, tl, nb * NB + c * 64, tx * TW, ty * TH + 2 * quad, img);
            bw::tma_store_commit();
          }
        }
      }
    }
    if (lane == 0) bw::tma_store_wait_all<0>();
  } else if (warp >= 8) {
    // ===================== A builders: one thread per output pixel =====================
    // This role sets the pace of the kernel (r2 profile: the MMA warp spent 1/3 of its time waiting for chunk 0 of
    // the next tile while a builder thread needed ~1500 instructions per tile), so everything that does not change
    // from tile to tile is hoisted: the 14 byte offsets of a pixel's taps inside a chunk (7 per halo-row parity),
    // 32-bit plane offsets for the 49 weight loads, fences only after chunks the thread actually wrote.
    // Builder warp w owns tile rows w and w + 4 (lanes 0-15 / 16-31): rows of the SAME parity cross chunk boundaries at
    // the same tap row ky, so the publish / acquire steps inside the ky loop are warp-uniform.  With rows 2w and 2w + 1
    // in one warp every ky iteration diverged and the warp executed both paths (r2 profile: 1340 instructions per tile,
    // the MMA warp waiting on a_full 44 % of the time).
    const int py = (warp - 8) + 4 * (lane >> 4), px = lane & 15;
    const int m = py * 16 + px;
    const int plane = p.h * p.w;                      // host guarantees 49 * h * w < 2^31
    uint32_t off_e[7], off_o[7];                      // taps kx = 0..6 in an even / odd halo row of a chunk
#pragma unroll
    for (int kx = 0; kx < 7; ++kx) {
      off_e[kx] = C::a_off((uint32_t)m, (uint32_t)(px + kx));
      off_o[kx] = C::a_off((uint32_t)m, (uint32_t)(24 + px + kx));
    }
    const uint32_t sA_u32 = bw::smem_u32(sA);
    float wr[49];
    auto load_raw = [&](int tile) {
      int t = tile;
      const int tx = t % p.tiles_x; t /= p.tiles_x;
      const int ty = t % p.tiles_y;
      const int img = t / p.tiles_y;
      const int gy = ty * TH + py, gx = tx * TW + px;
      const bool ok = gy < p.h && gx < p.w;
      const float* wp = p.weight + ((int64_t)img * 49 * plane + (int64_t)gy * p.w + gx);
      if (ok) {
#pragma unroll
        for (int k = 0; k < 49; ++k) wr[k] = __ldg(wp + k * plane);
      } else {
#pragma unroll
        for (int k = 0; k < 49; ++k) wr[k] = 0.f;
      }
    };
    uint32_t tcount = 0;
    int tile = blockIdx.x;
    if (!RAWTMA && tile < p.num_tiles) load_raw(tile);
    for (; tile < p.num_tiles; tile += gridDim.x, ++tcount) {
      if (RAWTMA) {   // this tile's raw weights: shared memory [49][8][16], filled by TMA (zero outside the map)
        bw::mbar_wait(w_full, tcount & 1);
        const float* wsrc = sW + py * TW + px;
#pragma unroll
        for (int k = 0; k < 49; ++k) wr[k] = wsrc[k * (TH * TW)];
        bw::mbar_arrive(w_empty);   // consumed: warp 3 may fetch the next tile's box
      }
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
      for (int k = 0; k < 48; k += 4) { s0 += wr[k]; s1 += wr[k + 1]; s2 += wr[k + 2]; s3 += wr[k + 3]; }
      const float inv = 1.0f / (((s0 + s1) + (s2 + s3)) + wr[48] + p.eps);
      uint32_t wp2[25];   // normalised weights as bf16 pairs (tap 2i in the low half)
#pragma unroll
      for (int k = 0; k < 25; ++k) {
        const __nv_bfloat162 b = __floats2bfloat162_rn(wr[2 * k] * inv, k < 24 ? wr[2 * k + 1] * inv : 0.f);
        wp2[k] = *reinterpret_cast<const uint32_t*>(&b);
      }
      // prefetch the next tile's weights (measured: issuing these loads only after the last publish of the tile, to keep
      // them out of the way of the membar inside fence.proxy.async, costs 0.249 -> 0.319 ms: the loads are then exposed)
      if (!RAWTMA && tile + (int)gridDim.x < p.num_tiles) load_raw(tile + gridDim.x);
      // Chunks are acquired strictly in order, EVERY chunk by EVERY builder thread (also the chunks a pixel has no
      // taps in): a thread may only arrive on a_full[c] for this tile after a_empty[c] says the previous tile's MMAs
      // are done with chunk c, which in turn needed all 128 arrivals of the previous tile -- so no thread can arrive
      // twice inside one phase of a_full[c] (a thread running a tile ahead would otherwise complete the phase early).
      const uint32_t eparity = (tcount & 1) ^ 1;
      int cur = 0;
      bool wrote = false;
      bw::mbar_wait(&a_empty[0], eparity);
#pragma unroll
      for (int ky = 0; ky < 7; ++ky) {
        const int j = (py + ky) >> 1;
        while (cur < j) {                       // done with chunk `cur`: publish it, acquire the next
          if (wrote) bw::fence_proxy_async_smem();
          wrote = false;
          bw::mbar_arrive(&a_full[cur]);
          ++cur;
          bw::mbar_wait(&a_empty[cur], eparity);
        }
        const uint32_t cbase = sA_u32 + (uint32_t)(j * A_CHUNK);
        // halo row parity r = (py + ky) & 1: for even ky it is py & 1, for odd ky the other one
        const bool odd_row = ((py + ky) & 1) != 0;
#pragma unroll
        for (int kx = 0; kx < 7; ++kx) {
          const int t = ky * 7 + kx;
          const uint32_t v = (t & 1) ? (wp2[t >> 1] >> 16) : wp2[t >> 1];
          const uint32_t addr = cbase + (odd_row ? off_o[kx] : off_e[kx]);
          asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"((unsigned short)v) : "memory");
        }
        wrote = true;
      }
      while (cur < NCHUNK - 1) {
        if (wrote) bw::fence_proxy_async_smem();
        wrote = false;
        bw::mbar_arrive(&a_full[cur]);
        ++cur;
        bw::mbar_wait(&a_empty[cur], eparity);
      }
      if (wrote) bw::fence_proxy_async_smem();
      bw::mbar_arrive(&a_full[NCHUNK - 1]);
    }
  }
  bw::tc_fence_before();
  __syncthreads();
  if (warp == 2) bw::tmem_dealloc(tmem_base, 512);
}

}  // namespace mptc

// One diffusion step on the tensor pipe; 0 on success, 1 when the shape is not handled here.
template <bool RAWTMA>
static int mp_tc_launch(const CUtensorMap& tmX, const CUtensorMap& tmOut, const CUtensorMap& tmW, const mptc::Params& p,
                        int grid, cudaStream_t s) {
  using namespace mptc;
  using Cf = Cfg<RAWTMA>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e1 = cudaFuncSetAttribute(mp_tc_kernel<RAWTMA>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cf::SMEM);
    if (e1 != cudaSuccess) {
      set_error("message_passing_tc: cannot opt in to %d B smem: %s", Cf::SMEM, cudaGetErrorString(e1));
      return -2;
    }
    configured = true;
  }
  mp_tc_kernel<RAWTMA><<<grid, THREADS, Cf::SMEM, s>>>(tmX, tmOut, tmW, p);
  return 0;
}

int mp_tc_step_bf16(const void* x, const float* weight, void* out, int n, int h, int w, int c, float eps, cudaStream_t s) {
  using namespace mptc;
  if (c % NB != 0 || (int64_t)h * w * 49 >= (int64_t)1 << 31) return 1;
  CUtensorMap tmX, tmOut;
  const uint64_t dims[4] = {(uint64_t)c, (uint64_t)w, (uint64_t)h, (uint64_t)n};
  const uint64_t strides[3] = {(uint64_t)c * 2, (uint64_t)w * c * 2, (uint64_t)h * w * c * 2};
  const uint32_t box_in[4] = {64, PW, 2, 1}, box_out[4] = {64, TW, 2, 1};
  int rc = make_tmap(&tmX, x, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, dims, strides, box_in, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  rc = make_tmap(&tmOut, out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, dims, strides, box_out, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  Params p;
  p.weight = weight;
  p.n = n; p.h = h; p.w = w; p.C = c;
  p.tiles_x = cdiv(w, TW);
  p.tiles_y = cdiv(h, TH);
  p.num_tiles = n * p.tiles_x * p.tiles_y;
  p.eps = eps;
  const int grid = p.num_tiles < sm_count() ? p.num_tiles : sm_count();
  CUtensorMap tmW = tmX;   // placeholder when the raw weights are read with plain loads
  const bool rawtma = w % 4 == 0;   // TMA needs 16-byte multiples for the weight planes' row pitch
  if (rawtma) {
    const uint64_t wdims[4] = {(uint64_t)w, (uint64_t)h, 49, (uint64_t)n};
    const uint64_t wstr[3] = {(uint64_t)w * 4, (uint64_t)h * w * 4, (uint64_t)49 * h * w * 4};
    const uint32_t wbox[4] = {TW, TH, 49, 1};
    rc = make_tmap(&tmW, weight, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, wdims, wstr, wbox, CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc) return rc;
  }
  return rawtma ? mp_tc_launch<true>(tmX, tmOut, tmW, p, grid, s) : mp_tc_launch<false>(tmX, tmOut, tmW, p, grid, s);
}

}  // namespace dgtd
