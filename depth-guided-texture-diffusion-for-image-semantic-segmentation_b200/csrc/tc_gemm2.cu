// 2-CTA (cta_group::2) tcgen05 GEMM: a CTA pair on one TPC computes a 256 x BN tile.
//
// Why: a single-CTA 128x256 tile needs 96 B/clk/SM of operand traffic at full MMA rate, more
// than the L2->SM fabric delivers (~43 B/clk/SM measured: profiles/r1_launches_b64_v2.md shows
// the K=2048 GEMM stuck at 36% tensor-pipe).  In a pair each CTA stages its own 128 rows of A
// and only HALF of the B tile; tcgen05.mma.cta_group::2 reads both halves through the pair's
// shared memory, so the per-SM feed drops to 64 B/clk.
//
// Protocol (rank 0 = leader):
//   * both CTAs run a TMA producer (own A rows + own half of B); the transaction bytes of both
//     land on the LEADER's `full` barrier (cp.async.bulk.tensor ... .cta_group::2);
//   * the leader's MMA thread issues M=256 UMMAs; tcgen05.commit multicasts to the `empty` /
//     `tmem_full` barriers of both CTAs;
//   * each CTA's 8 epilogue warps drain their own 128 TMEM lanes and arrive (remotely for
//     rank 1) on the leader's `tmem_empty` barrier.
#include "tc_common.cuh"

namespace dgtd {

namespace bw2 {
__device__ __forceinline__ uint32_t cta_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `p`'s counterpart in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_rank(const void* p, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(bw::smem_u32(p)), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(const CUtensorMap* m, uint32_t leader_bar, void* dst, int c0,
                                                int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(bw::smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(leader_bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(bw::smem_u32(dst_smem)),
               "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the same-offset barrier of both CTAs of the pair when the issued MMAs retire
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(bw::smem_u32(bar)), "h"((uint16_t)3)
      : "memory");
}
}  // namespace bw2

template <int BN>
struct Tc2Cfg {
  static constexpr int BM = 128, BK = 64;                          // per CTA; the pair covers 256 rows
  static constexpr int A_BYTES = BM * BK * 2, B_BYTES = (BN / 2) * BK * 2;   // B: this CTA's half
  static constexpr int STAGES = BN >= 256 ? 5 : 6;
  static constexpr int TMEM_COLS = 2 * BN;
  static constexpr int STG_BYTES = 8 * 2 * 4096;   // 8 epilogue warps x 2 staging tiles of 4 KB
  static constexpr int XCH_BYTES = BN == 128 ? 2 * 8 * 32 * 8 : 0;   // LNROW: (sum, sum of squares) of 2 tile parities x 8 warps
  static constexpr int SMEM_BYTES = STAGES * (A_BYTES + B_BYTES) + STG_BYTES + 512 + XCH_BYTES + 1024;
};

template <int BN, int ACT, typename OT, bool RESIDUAL, int NEPI = 8, bool LNROW = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128 + 32 * NEPI, 1)
tc_gemm2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const __grid_constant__ CUtensorMap tmOut, const __grid_constant__ CUtensorMap tmRes,
                const TcParams p) {
  using Cfg = Tc2Cfg<BN>;
  constexpr int BM = Cfg::BM, BK = Cfg::BK, STAGES = Cfg::STAGES;
  // identical carve-up in both CTAs (the hardware addresses the peer's operands by offset)
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * Cfg::A_BYTES;
  uint8_t* sStg = smem + STAGES * (Cfg::A_BYTES + Cfg::B_BYTES);   // epilogue staging, 1024-aligned
  uint64_t* bars = reinterpret_cast<uint64_t*>(sStg + Cfg::STG_BYTES);
  uint64_t* rbars = bars + 2 * STAGES + 6;   // [8 warps][2] residual-tile barriers
  uint64_t* full = bars;                     // used on the leader only
  uint64_t* empty = bars + STAGES;
  uint64_t* tfull = bars + 2 * STAGES;
  uint64_t* tempty = bars + 2 * STAGES + 2;  // used on the leader only
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = bw2::cta_rank();
  const bool leader = rank == 0;
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
  const int tiles_mn = p.tiles_m * p.tiles_n;    // tiles_m counts 256-row pair tiles
  const int num_tiles = tiles_mn * p.splits;
  const int num_kb = (p.K + BK - 1) / BK;
  const int kbs = p.splits > 1 ? p.kb_per_split : num_kb;

  bw2::cluster_sync();  // both CTAs resident before the pair-wide TMEM allocation
  if (warp == 0 && lane == 0) {
    bw::prefetch_tmap(&tmA);
    bw::prefetch_tmap(&tmB);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) {
      bw::mbar_init(&full[i], 2);     // one arrival per CTA's producer
      bw::mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      bw::mbar_init(&tfull[i], 1);
      bw::mbar_init(&tempty[i], 2 * NEPI * 32);  // epilogue threads of both CTAs
    }
    for (int i = 0; i < 16; ++i) bw::mbar_init(&rbars[i], 1);
    bw::fence_mbar_init();
  }
  if (warp == 2) bw2::tmem_alloc_2sm(tmem_slot, Cfg::TMEM_COLS);
  bw::tc_fence_before();
  bw2::cluster_sync();
  bw::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      // ===================== TMA producer (both CTAs) =====================
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
        const int z = tile / tiles_mn, t2 = tile - z * tiles_mn;
        const int m_blk = t2 / p.tiles_n, n_blk = t2 - m_blk * p.tiles_n;
        const int m0 = m_blk * 256 + (int)rank * BM;
        const int n0 = n_blk * BN + (int)rank * (BN / 2);
        const int kb0 = z * kbs, kb1 = min(num_kb, kb0 + kbs);
        for (int kb = kb0; kb < kb1; ++kb) {
          bw::mbar_wait(&empty[stage], phase ^ 1);
          const uint32_t lbar = bw2::map_to_rank(&full[stage], 0);
          if (p.mn_major) {   // {64 MN, 64 K-row} boxes, one 8 KB block per 64 columns
            bw2::tma_load_2d_2sm(&tmA, lbar, sA + stage * Cfg::A_BYTES, m0, kb * BK);
            bw2::tma_load_2d_2sm(&tmA, lbar, sA + stage * Cfg::A_BYTES + 8192, m0 + 64, kb * BK);
#pragma unroll
            for (int j = 0; j < BN / 128; ++j)
              bw2::tma_load_2d_2sm(&tmB, lbar, sB + stage * Cfg::B_BYTES + j * 8192, n0 + 64 * j, kb * BK);
          } else {
            bw2::tma_load_2d_2sm(&tmA, lbar, sA + stage * Cfg::A_BYTES, kb * BK, m0);
            bw2::tma_load_2d_2sm(&tmB, lbar, sB + stage * Cfg::B_BYTES, kb * BK, n0);
          }
          if (leader) bw::mbar_arrive_expect_tx(&full[stage], 2 * (Cfg::A_BYTES + Cfg::B_BYTES));
          else bw2::mbar_arrive_cluster(lbar);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (leader && lane == 0) {
      // ===================== MMA issuer (leader CTA only) =====================
      const uint32_t idesc = bw::umma_idesc_bf16(256, BN) | (p.mn_major ? (3u << 15) : 0u);
      const uint32_t kstep = p.mn_major ? 128u : 2u;   // 16 K rows x 128 B vs 16 elements x 2 B, in 16-byte units
      int stage = 0, iter = 0;
      uint32_t phase = 0;
      for (int tile = cluster_id; tile < num_tiles; tile += num_clusters, ++iter) {
        const int as = iter & 1;
        const uint32_t aphase = (iter >> 1) & 1;
        bw::mbar_wait(&tempty[as], aphase ^ 1);
        bw::tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        const int z = tile / tiles_mn;
        const int kb0 = z * kbs, kb1 = min(num_kb, kb0 + kbs);
        for (int kb = kb0; kb < kb1; ++kb) {
          bw::mbar_wait(&full[stage], phase);
          bw::tc_fence_after();
          const uint32_t a_addr = bw::smem_u32(sA + stage * Cfg::A_BYTES), b_addr = bw::smem_u32(sB + stage * Cfg::B_BYTES);
          const uint64_t da = p.mn_major ? bw::umma_smem_desc_mnmajor_sw128(a_addr, 8192, 1024)
                                         : bw::umma_smem_desc_kmajor(a_addr, 128);
          const uint64_t db = p.mn_major ? bw::umma_smem_desc_mnmajor_sw128(b_addr, 8192, 1024)
                                         : bw::umma_smem_desc_kmajor(b_addr, 128);
#pragma unroll
          for (int k = 0; k < BK / 16; ++k)
            bw2::umma_bf16_2sm(d_tmem, da + kstep * k, db + kstep * k, idesc, ((kb - kb0) | k) != 0);
          bw2::umma_commit_2sm(&empty[stage]);
          if (kb == kb1 - 1) bw2::umma_commit_2sm(&tfull[as]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (both CTAs, own 128 TMEM lanes) =====================
    const int quad = warp & 3, half = (warp - 4) >> 2;   // half = column part (2 or 4 per quadrant)
    uint8_t* stg = sStg + (warp - 4) * (NEPI == 8 ? 8192 : 4096);
    uint64_t* rbar = rbars + ((warp - 4) & 7) * 2;
    uint32_t sbuf = 0;
    int iter = 0;
    for (int tile = cluster_id; tile < num_tiles; tile += num_clusters, ++iter) {
      const int z = tile / tiles_mn, t2 = tile - z * tiles_mn;
      const int m_blk = t2 / p.tiles_n, n_blk = t2 - m_blk * p.tiles_n;
      const int as = iter & 1;
      const uint32_t aphase = (iter >> 1) & 1;
      bw::mbar_wait(&tfull[as], aphase);
      bw::tc_fence_after();
      const uint32_t rel = bw2::map_to_rank(&tempty[as], 0);
      if constexpr (LNROW) {
        static_assert(!LNROW || (BN == 128 && NEPI == 8 && !RESIDUAL && sizeof(OT) == 4), "row LayerNorm: one 128-column fp32 tile");
        tc_epilogue_tile_tma_ln128(p, &tmOut, tmem_base + as * BN, quad, half, lane, m_blk * 256 + (int)rank * BM + quad * 32, stg,
                                   reinterpret_cast<float2*>(sStg + Cfg::STG_BYTES + 512), iter & 1, sbuf,
                                   [rel] { bw2::mbar_arrive_cluster(rel); });
      } else {
        tc_epilogue_tile_tma<BN, ACT, OT, RESIDUAL, NEPI / 4>(p, &tmOut, &tmRes, tmem_base + as * BN, quad, half, lane,
                                                    z * p.split_rows + m_blk * 256 + (int)rank * BM + quad * 32, n_blk, stg, rbar,
                                                    sbuf, [rel] { bw2::mbar_arrive_cluster(rel); });
      }
    }
    if (lane == 0) bw::tma_store_wait_all<0>();   // all results are in global memory before exit
  }

  // nobody leaves (or frees TMEM) while the peer may still signal our barriers / read our smem
  bw::tc_fence_before();
  bw2::cluster_sync();
  if (warp == 2) {
    bw::tc_fence_after();
    bw2::tmem_dealloc_2sm(tmem_base, Cfg::TMEM_COLS);
  }
}

template <int BN, int ACT, typename OT, bool RESIDUAL, int NEPI = 8, bool LNROW = false>
static int tc2_launch(const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* B, int64_t ldb, TcParams p,
                      cudaStream_t s) {
  using Cfg = Tc2Cfg<BN>;
  auto kern = tc_gemm2_kernel<BN, ACT, OT, RESIDUAL, NEPI, LNROW>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) {
      set_error("tc_gemm2: cannot opt in to %d B of shared memory: %s", Cfg::SMEM_BYTES, cudaGetErrorString(e));
      return -2;
    }
    configured = true;
  }
  CUtensorMap tmA, tmB;
  if (p.mn_major) {   // A: (K rows) x M, B: (K rows) x N, row-major with pitches lda / ldb
    uint64_t dimsA[2] = {(uint64_t)p.M, (uint64_t)p.K}, strA[1] = {(uint64_t)lda * 2};
    uint64_t dimsB[2] = {(uint64_t)p.N, (uint64_t)p.K}, strB[1] = {(uint64_t)ldb * 2};
    uint32_t box[2] = {64, 64};
    int rc = make_tmap(&tmA, A, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dimsA, strA, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    rc = make_tmap(&tmB, B, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dimsB, strB, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  } else {
    {
      uint64_t dims[2] = {(uint64_t)p.K, (uint64_t)p.M}, str[1] = {(uint64_t)lda * 2};
      uint32_t box[2] = {64, 128};
      int rc = make_tmap(&tmA, A, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
      if (rc) return rc;
    }
    {
      uint64_t dims[2] = {(uint64_t)p.K, (uint64_t)p.N}, str[1] = {(uint64_t)ldb * 2};
      uint32_t box[2] = {64, (uint32_t)(BN / 2)};
      int rc = make_tmap(&tmB, B, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
      if (rc) return rc;
    }
  }
  CUtensorMap tmOut, tmRes;
  {
    constexpr bool BF = sizeof(OT) == 2;
    const uint64_t out_rows = p.splits > 1 || p.split_rows > p.M ? (uint64_t)p.split_rows * p.splits : (uint64_t)p.M;
    uint64_t dims[2] = {(uint64_t)p.N, out_rows}, str[1] = {(uint64_t)p.ldo * sizeof(OT)};
    uint32_t box[2] = {BF ? 64u : 32u, 32u};
    int rc = make_tmap(&tmOut, p.out, BF ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                       dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
    tmRes = tmOut;
    if (RESIDUAL) {
      rc = make_tmap(&tmRes, p.residual, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, dims, str, box,
                     CU_TENSOR_MAP_SWIZZLE_128B);
      if (rc) return rc;
    }
  }
  p.tiles_m = cdiv(p.M, 256);
  p.tiles_n = cdiv(p.N, BN);
  int tiles = p.tiles_m * p.tiles_n * p.splits;
  int pairs = sm_count() / 2;
  int clusters = tiles < pairs ? tiles : pairs;
  kern<<<2 * clusters, 128 + 32 * NEPI, Cfg::SMEM_BYTES, s>>>(tmA, tmB, tmOut, tmRes, p);
  return 0;
}

template <int BN>
static int tc2_dispatch(const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* B, int64_t ldb,
                        const TcParams& p, int act, int dtype_out, bool residual, cudaStream_t s) {
  if (residual) return tc2_launch<BN, DGTD_ACT_NONE, float, true>(A, lda, B, ldb, p, s);
  if (dtype_out == DGTD_BF16) {
    if (act == DGTD_ACT_GELU) {   // pwconv1: the GELU epilogue is issue-latency bound -> 16 epilogue warps at BN = 256
      // (K >= 1024, stage 3: the main loop of a tile is long enough to hide the 8-warp epilogue, which measures 65 vs 69 us)
      if (BN == 256 && p.K < 1024) return tc2_launch<BN, DGTD_ACT_GELU, __nv_bfloat16, false, BN == 256 ? 16 : 8>(A, lda, B, ldb, p, s);
      return tc2_launch<BN, DGTD_ACT_GELU, __nv_bfloat16, false>(A, lda, B, ldb, p, s);
    }
    if (act == DGTD_ACT_RELU) return tc2_launch<BN, DGTD_ACT_RELU, __nv_bfloat16, false>(A, lda, B, ldb, p, s);
    return tc2_launch<BN, DGTD_ACT_NONE, __nv_bfloat16, false>(A, lda, B, ldb, p, s);
  }
  if (act == DGTD_ACT_GELU) return tc2_launch<BN, DGTD_ACT_GELU, float, false>(A, lda, B, ldb, p, s);
  if (act == DGTD_ACT_RELU) return tc2_launch<BN, DGTD_ACT_RELU, float, false>(A, lda, B, ldb, p, s);
  return tc2_launch<BN, DGTD_ACT_NONE, float, false>(A, lda, B, ldb, p, s);
}

// Returns 0 launched, <0 error, 1 = shape not handled here (caller uses the 1-CTA kernel).
int tc_gemm2_launch(const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* B, int64_t ldb, TcParams p,
                    int act, int dtype_out, bool residual, cudaStream_t s) {
  if (p.N < 128 || p.M < 256) return 1;
  const size_t esz = dtype_out == DGTD_BF16 ? 2 : 4;
  if ((p.ldo * esz) % 16 || (reinterpret_cast<uintptr_t>(p.out) & 15) ||
      (residual && (reinterpret_cast<uintptr_t>(p.residual) & 15)))
    return 1;   // TMA store needs 16-byte aligned rows
  const int64_t pair_tiles_256 = (int64_t)cdiv(p.M, 256) * cdiv(p.N, 256);
  if (p.N % 256 == 0 && pair_tiles_256 >= sm_count() / 2)
    return tc2_dispatch<256>(A, lda, B, ldb, p, act, dtype_out, residual, s);
  return tc2_dispatch<128>(A, lda, B, ldb, p, act, dtype_out, residual, s);
}

// out (M x 128 fp32) = LayerNorm_rows(A . B^T + bias) * ln_w + ln_b, the LayerNorm fused in the epilogue (p.ln_w / p.ln_b / p.ln_eps set).
// Returns 1 when the shape is not handled here.
int tc_gemm2_ln_launch(const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* B, int64_t ldb, TcParams p, cudaStream_t s) {
  if (p.N != 128 || p.M < 256 || p.ldo != 128 || (reinterpret_cast<uintptr_t>(p.out) & 15)) return 1;
  return tc2_launch<128, DGTD_ACT_NONE, float, false, 8, true>(A, lda, B, ldb, p, s);
}

// Split-K partial products for weight gradients: partial[z] (M x N fp32) = A[:, Kz] . B[:, Kz]^T
// partial: splits x roundup(M, 256) x N floats.  A is (K x M), B is (K x N) row-major, read as MN-major operands.
int tc_gemm2_splitk(const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* B, int64_t ldb, float* partial, int M,
                    int N, int K, int splits, cudaStream_t s) {
  TcParams p{};
  p.M = M; p.N = N; p.K = K; p.out = partial; p.ldo = N; p.rows_per_sample = 1;
  p.splits = splits;
  p.split_rows = cdiv(M, 256) * 256;
  p.mn_major = 1;
  const int num_kb = cdiv(K, 64);
  p.kb_per_split = cdiv(num_kb, splits);
  if ((int64_t)(splits - 1) * p.kb_per_split >= num_kb) {   // every split must own at least one k-block
    p.splits = cdiv(num_kb, p.kb_per_split);
  }
  if (p.splits != splits) {
    set_error("tc_gemm2_splitk: %d splits leave an empty split for K=%d", splits, K);
    return -1;
  }
  if (N % 256 == 0) return tc2_launch<256, DGTD_ACT_NONE, float, false>(A, lda, B, ldb, p, s);
  return tc2_launch<128, DGTD_ACT_NONE, float, false>(A, lda, B, ldb, p, s);
}

}  // namespace dgtd
