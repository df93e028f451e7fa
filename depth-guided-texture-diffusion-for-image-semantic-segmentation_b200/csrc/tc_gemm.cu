// Dense contractions of the path on the 5th-gen tensor cores (tcgen05 + TMEM + TMA):
//   C[M,N] = A[M,K] . B[N,K]^T   bf16 operands (K-major), fp32 accumulation in TMEM,
// with the epilogues of convnext_Block (cod.py:1109-1116), the down-sample convs (:1134) and
// the head / decoder convs fused on the accumulator read-back.
//
// One persistent CTA per SM, 256 threads, warp-specialised:
//   warp 0 (one lane)  TMA producer: 128xBK A tile + BNxBK B tile per stage, 128B swizzle
//   warp 1 (one lane)  tcgen05.mma issuer: 128 x BN x 16 UMMAs, accumulator in TMEM
//   warp 2             TMEM allocation / release
//   warps 4-11         epilogue: tcgen05.ld (32 lanes x 32 columns, double buffered; two warps per
//                      TMEM lane quadrant split the columns) -> registers -> bias / GELU (packed
//                      fp32x2) / gamma / DropPath scale / residual -> 16-byte global stores
// Two TMEM accumulator stages let the epilogue of tile i overlap the main loop of tile i+1.
#include <mutex>

#include "simt_gemm.cuh"
#include "tc_common.cuh"

namespace dgtd {

// ---------------------------------------------------------------- tensor-map plumbing
PFN_tmapEncodeTiled get_tmap_encoder() {
  static PFN_tmapEncodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q);
    if (e == cudaSuccess && q == cudaDriverEntryPointSuccess) fn = (PFN_tmapEncodeTiled)p;
  });
  if (!fn) set_error("cuTensorMapEncodeTiled is not available from this driver");
  return fn;
}

int make_tmap(CUtensorMap* out, const void* base, CUtensorMapDataType dt, int rank,
              const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box,
              CUtensorMapSwizzle swz) {
  PFN_tmapEncodeTiled enc = get_tmap_encoder();
  if (!enc) return -3;
  cuuint64_t gd[5], gs[5];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gd[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
    if (i > 0) gs[i - 1] = strides_bytes[i - 1];
  }
  CUresult r = enc(out, dt, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (CUresult %d) rank=%d dims=[%llu,%llu] box=[%u,%u]", (int)r,
              rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0), box[0],
              rank > 1 ? box[1] : 0);
    return -3;
  }
  return 0;
}

int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

template <int BN>
struct TcCfg {
  static constexpr int BM = 128, BK = 64;
  static constexpr int A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2;
  static constexpr int STAGES = BN >= 256 ? 4 : 6;
  static constexpr int TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;
  static constexpr int BAR_BYTES = 256;
  static constexpr int SMEM_BYTES = STAGES * (A_BYTES + B_BYTES) + BAR_BYTES + 1024;  // +align slack
};

// TF32: fp32 operands read as they are (kind::tf32, 10-bit mantissas): a k-block is still 128 bytes per row = 32 elements,
// one instruction covers K = 8.  Used where an fp32 activation would otherwise be cast to bf16 by a separate pass.
template <int BN, int ACT, typename OT, bool RESIDUAL, bool CONV3 = false, bool TF32 = false>
__global__ void __launch_bounds__(384, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const TcParams p) {
  using Cfg = TcCfg<BN>;
  constexpr int BM = Cfg::BM, BK = TF32 ? Cfg::BK / 2 : Cfg::BK, STAGES = Cfg::STAGES;   // elements per 128-byte k-block row
  extern __shared__ __align__(1024) uint8_t smem[];   // 128B-swizzle atoms need 1024-byte alignment
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * Cfg::A_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * (Cfg::A_BYTES + Cfg::B_BYTES));
  uint64_t* full = bars;                    // [STAGES]
  uint64_t* empty = bars + STAGES;          // [STAGES]
  uint64_t* tfull = bars + 2 * STAGES;      // [2]
  uint64_t* tempty = bars + 2 * STAGES + 2; // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_tiles = p.tiles_m * p.tiles_n;
  const int num_kb = CONV3 ? 9 * p.cv_chunks : (p.K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    bw::prefetch_tmap(&tmA);
    bw::prefetch_tmap(&tmB);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) {
      bw::mbar_init(&full[i], 1);
      bw::mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      bw::mbar_init(&tfull[i], 1);
      bw::mbar_init(&tempty[i], 256);
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
      // ===================== TMA producer =====================
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int m_blk = tile / p.tiles_n, n_blk = tile - m_blk * p.tiles_n;
        int img = 0, oy0 = 0, ox0 = 0;
        if (CONV3) {   // m_blk = (image, patch row, patch column)
          const int px = m_blk % p.cv_tiles_x, t = m_blk / p.cv_tiles_x;
          ox0 = px * 16; oy0 = (t % p.cv_tiles_y) * 8; img = t / p.cv_tiles_y;
        }
        int tap = 0, chunk = 0;
        for (int kb = 0; kb < num_kb; ++kb) {
          bw::mbar_wait(&empty[stage], phase ^ 1);
          bw::mbar_arrive_expect_tx(&full[stage], Cfg::A_BYTES + Cfg::B_BYTES);
          if (CONV3) {
            const int dy = tap / 3, dx = tap - dy * 3;
            bw::tma_load_4d(&tmA, &full[stage], sA + stage * Cfg::A_BYTES, chunk * BK, ox0 + dx - 1, oy0 + dy - 1, img);
            if (++chunk == p.cv_chunks) { chunk = 0; ++tap; }
          } else {
            bw::tma_load_2d(&tmA, &full[stage], sA + stage * Cfg::A_BYTES, kb * BK, m_blk * BM);
          }
          bw::tma_load_2d(&tmB, &full[stage], sB + stage * Cfg::B_BYTES, kb * BK, n_blk * BN);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      // ===================== MMA issuer =====================
      constexpr uint32_t idesc = TF32 ? bw::umma_idesc_tf32(BM, BN) : bw::umma_idesc_bf16(BM, BN);
      int stage = 0;
      uint32_t phase = 0;
      int iter = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++iter) {
        const int as = iter & 1;
        const uint32_t aphase = (iter >> 1) & 1;
        bw::mbar_wait(&tempty[as], aphase ^ 1);  // epilogue has drained this accumulator
        bw::tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          bw::mbar_wait(&full[stage], phase);
          bw::tc_fence_after();
          const uint64_t da = bw::umma_smem_desc_kmajor(bw::smem_u32(sA + stage * Cfg::A_BYTES), 128);
          const uint64_t db = bw::umma_smem_desc_kmajor(bw::smem_u32(sB + stage * Cfg::B_BYTES), 128);
#pragma unroll
          for (int k = 0; k < 4; ++k) {  // +32 B per K step (16 bf16 / 8 tf32) inside the 128B swizzle atom
            if (TF32) bw::umma_tf32(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
            else bw::umma_bf16(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
          }
          bw::umma_commit(&empty[stage]);            // smem slot free once these MMAs retire
          if (kb == num_kb - 1) bw::umma_commit(&tfull[as]);  // accumulator complete
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (8 warps) =====================
    // warp w may read TMEM lanes [32*(w%4), +32); the two warps of a quadrant split the columns.
    const int quad = warp & 3, half = (warp - 4) >> 2;
    int iter = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++iter) {
      const int m_blk = tile / p.tiles_n, n_blk = tile - m_blk * p.tiles_n;
      const int as = iter & 1;
      const uint32_t aphase = (iter >> 1) & 1;
      bw::mbar_wait(&tfull[as], aphase);
      bw::tc_fence_after();
      uint64_t* rel = &tempty[as];
      int row = m_blk * BM + quad * 32 + lane;
      if (CONV3) {   // accumulator row r = pixel (r / 16, r % 16) of the patch -> NHWC pixel index, or masked
        const int px = m_blk % p.cv_tiles_x, t = m_blk / p.cv_tiles_x;
        const int r = quad * 32 + lane;
        const int oy = (t % p.cv_tiles_y) * 8 + (r >> 4), ox = px * 16 + (r & 15);
        row = (oy < p.cv_h && ox < p.cv_w) ? ((t / p.cv_tiles_y) * p.cv_h + oy) * p.cv_w + ox : p.M;
      }
      tc_epilogue_tile<BN, ACT, OT, RESIDUAL>(p, tmem_base + as * BN, quad, half, lane, row, n_blk,
                                              [rel] { bw::mbar_arrive(rel); });
    }
  }

  bw::tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    bw::tc_fence_after();
    bw::tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

template <int BN, int ACT, typename OT, bool RESIDUAL>
static int tc_launch(const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* B, int64_t ldb,
                     TcParams p, cudaStream_t s) {
  using Cfg = TcCfg<BN>;
  auto kern = tc_gemm_kernel<BN, ACT, OT, RESIDUAL>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) {
      set_error("tc_gemm: cannot opt in to %d B of shared memory: %s", Cfg::SMEM_BYTES, cudaGetErrorString(e));
      return -2;
    }
    configured = true;
  }
  CUtensorMap tmA, tmB;
  {
    uint64_t dims[2] = {(uint64_t)p.K, (uint64_t)p.M}, str[1] = {(uint64_t)lda * 2};
    uint32_t box[2] = {64, 128};
    int rc = make_tmap(&tmA, A, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  }
  {
    uint64_t dims[2] = {(uint64_t)p.K, (uint64_t)p.N}, str[1] = {(uint64_t)ldb * 2};
    uint32_t box[2] = {64, (uint32_t)BN};
    int rc = make_tmap(&tmB, B, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  }
  p.tiles_m = cdiv(p.M, 128);
  p.tiles_n = cdiv(p.N, BN);
  int tiles = p.tiles_m * p.tiles_n;
  int grid = tiles < sm_count() ? tiles : sm_count();
  kern<<<grid, 384, Cfg::SMEM_BYTES, s>>>(tmA, tmB, p);
  return 0;
}

// fp32 operands on kind::tf32 (N <= 64): out fp32 = A[M,K] . B[N,K]^T + bias
template <int BN>
static int tc_launch_tf32(const float* A, const float* B, TcParams p, cudaStream_t s) {
  using Cfg = TcCfg<BN>;
  auto kern = tc_gemm_kernel<BN, DGTD_ACT_NONE, float, false, false, true>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) {
      set_error("tc_gemm(tf32): cannot opt in to %d B of shared memory: %s", Cfg::SMEM_BYTES, cudaGetErrorString(e));
      return -2;
    }
    configured = true;
  }
  CUtensorMap tmA, tmB;
  {
    uint64_t dims[2] = {(uint64_t)p.K, (uint64_t)p.M}, str[1] = {(uint64_t)p.K * 4};
    uint32_t box[2] = {32, 128};
    int rc = make_tmap(&tmA, A, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  }
  {
    uint64_t dims[2] = {(uint64_t)p.K, (uint64_t)p.N}, str[1] = {(uint64_t)p.K * 4};
    uint32_t box[2] = {32, (uint32_t)BN};
    int rc = make_tmap(&tmB, B, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  }
  p.tiles_m = cdiv(p.M, 128);
  p.tiles_n = cdiv(p.N, BN);
  const int tiles = p.tiles_m * p.tiles_n;
  const int grid = tiles < sm_count() ? tiles : sm_count();
  kern<<<grid, 384, Cfg::SMEM_BYTES, s>>>(tmA, tmB, p);
  return 0;
}

template <int ACT, typename OT, bool RESIDUAL>
static int tc_dispatch_bn(const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* B, int64_t ldb,
                          const TcParams& p, cudaStream_t s) {
  // widest tile that divides the work sensibly; N <= 32 keeps a single narrow tile
  if (p.N <= 32) return tc_launch<32, ACT, OT, RESIDUAL>(A, lda, B, ldb, p, s);
  if (p.N <= 64) return tc_launch<64, ACT, OT, RESIDUAL>(A, lda, B, ldb, p, s);
  if (p.N % 256 == 0 && (int64_t)cdiv(p.M, 128) * (p.N / 256) >= sm_count())
    return tc_launch<256, ACT, OT, RESIDUAL>(A, lda, B, ldb, p, s);
  return tc_launch<128, ACT, OT, RESIDUAL>(A, lda, B, ldb, p, s);
}

// 3x3 / stride 1 / pad 1 convolution as an implicit GEMM: x (B, h, w, Cp) bf16 with Cp a multiple of 64,
// weights (Cout, 9 * Cp) bf16 tap-major, out (B*h*w, ldo) fp32 = conv + bias.
template <int BN>
static int tc_conv3_launch(const __nv_bfloat16* x, const __nv_bfloat16* w, TcParams p, int B, int Cp, cudaStream_t s) {
  using Cfg = TcCfg<BN>;
  auto kern = tc_gemm_kernel<BN, DGTD_ACT_NONE, float, false, true>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) {
      set_error("tc_conv3: cannot opt in to %d B of shared memory: %s", Cfg::SMEM_BYTES, cudaGetErrorString(e));
      return -2;
    }
    configured = true;
  }
  CUtensorMap tmA, tmB;
  {
    uint64_t dims[4] = {(uint64_t)Cp, (uint64_t)p.cv_w, (uint64_t)p.cv_h, (uint64_t)B};
    uint64_t str[3] = {(uint64_t)Cp * 2, (uint64_t)p.cv_w * Cp * 2, (uint64_t)p.cv_h * p.cv_w * Cp * 2};
    uint32_t box[4] = {64, 16, 8, 1};
    int rc = make_tmap(&tmA, x, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  }
  {
    uint64_t dims[2] = {(uint64_t)p.K, (uint64_t)p.N}, str[1] = {(uint64_t)p.K * 2};
    uint32_t box[2] = {64, (uint32_t)BN};
    int rc = make_tmap(&tmB, w, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dims, str, box, CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  }
  p.tiles_m = B * p.cv_tiles_y * p.cv_tiles_x;
  p.tiles_n = cdiv(p.N, BN);
  const int tiles = p.tiles_m * p.tiles_n;
  const int grid = tiles < sm_count() ? tiles : sm_count();
  kern<<<grid, 384, Cfg::SMEM_BYTES, s>>>(tmA, tmB, p);
  return 0;
}

int tc_conv3(const __nv_bfloat16* x, const __nv_bfloat16* w, const float* bias, float* out, int B, int h, int wd,
             int Cp, int Cout, int64_t ldo, cudaStream_t s) {
  TcParams p{};
  p.M = B * h * wd; p.N = Cout; p.K = 9 * Cp; p.bias = bias; p.out = out; p.ldo = ldo; p.rows_per_sample = 1;
  p.cv_h = h; p.cv_w = wd; p.cv_chunks = Cp / 64; p.cv_tiles_x = cdiv(wd, 16); p.cv_tiles_y = cdiv(h, 8);
  if (Cout <= 32) return tc_conv3_launch<32>(x, w, p, B, Cp, s);
  if (Cout <= 64) return tc_conv3_launch<64>(x, w, p, B, Cp, s);
  return tc_conv3_launch<128>(x, w, p, B, Cp, s);
}

int tc_linear(const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* B, int64_t ldb, const float* bias,
              void* out, int M, int N, int K, int64_t ldo, int dtype_out, int act, cudaStream_t s,
              const float2* row_stats = nullptr, const float* col_s = nullptr) {
  TcParams p{};
  p.M = M; p.N = N; p.K = K; p.bias = bias; p.out = out; p.ldo = ldo; p.rows_per_sample = 1;
  p.row_stats = row_stats; p.col_s = col_s;
  {
    int rc2 = tc_gemm2_launch(A, lda, B, ldb, p, act, dtype_out, false, s);
    if (rc2 <= 0) return rc2;
  }
  if (dtype_out == DGTD_BF16) {
    if (act == DGTD_ACT_GELU) return tc_dispatch_bn<DGTD_ACT_GELU, __nv_bfloat16, false>(A, lda, B, ldb, p, s);
    if (act == DGTD_ACT_RELU) return tc_dispatch_bn<DGTD_ACT_RELU, __nv_bfloat16, false>(A, lda, B, ldb, p, s);
    return tc_dispatch_bn<DGTD_ACT_NONE, __nv_bfloat16, false>(A, lda, B, ldb, p, s);
  }
  if (act == DGTD_ACT_GELU) return tc_dispatch_bn<DGTD_ACT_GELU, float, false>(A, lda, B, ldb, p, s);
  if (act == DGTD_ACT_RELU) return tc_dispatch_bn<DGTD_ACT_RELU, float, false>(A, lda, B, ldb, p, s);
  return tc_dispatch_bn<DGTD_ACT_NONE, float, false>(A, lda, B, ldb, p, s);
}

int tc_linear_residual(const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* B, int64_t ldb,
                       const float* bias, const float* gamma, const float* keep, int rows_per_sample,
                       const float* residual, float* out, int M, int N, int K, cudaStream_t s) {
  TcParams p{};
  p.M = M; p.N = N; p.K = K; p.bias = bias; p.gamma = gamma; p.keep = keep;
  p.rows_per_sample = rows_per_sample > 0 ? rows_per_sample : 1;
  p.residual = residual; p.out = out; p.ldo = N;
  {
    int rc2 = tc_gemm2_launch(A, lda, B, ldb, p, DGTD_ACT_NONE, DGTD_F32, true, s);
    if (rc2 <= 0) return rc2;
  }
  return tc_dispatch_bn<DGTD_ACT_NONE, float, true>(A, lda, B, ldb, p, s);
}

}  // namespace dgtd

using namespace dgtd;

extern "C" {

int dgtd_linear_fwd(const void* a, const void* w, const float* bias, void* out, int M, int N, int K,
                    int ldo, int dtype_in, int dtype_out, int act, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(a && w && out, "linear: null pointer");
  DGTD_CHECK_ARG(M > 0 && N > 0 && K > 0 && ldo >= N, "linear: bad shape M=%d N=%d K=%d ldo=%d", M, N, K, ldo);
  DGTD_CHECK_ARG(act >= 0 && act <= 2, "linear: bad activation %d", act);
  cudaStream_t s = (cudaStream_t)stream;
  if (dtype_in == DGTD_BF16) {
    DGTD_CHECK_ARG(K % 8 == 0 && N % 8 == 0 && ldo % 8 == 0, "linear(bf16): K, N, ldo must be multiples of 8");
    int rc = tc_linear((const __nv_bfloat16*)a, K, (const __nv_bfloat16*)w, K, bias, out, M, N, K, ldo,
                       dtype_out, act, s);
    if (rc) return rc;
    DGTD_LAUNCH_CHECK("linear(tcgen05)");
    return 0;
  }
  DGTD_CHECK_ARG(dtype_in == DGTD_F32, "linear: bad dtype_in %d", dtype_in);
  DGTD_CHECK_ARG(K % 4 == 0 && N % 4 == 0 && ldo % 4 == 0, "linear(fp32): K, N, ldo must be multiples of 4");
  RowMajorLoader al{(const float*)a, K, 0, M, K};
  RowMajorLoader bl{(const float*)w, K, 0, N, K};
#define DGTD_SIMT_LIN(OT, ACT)                                        \
  {                                                                   \
    EpiBiasAct<OT, ACT> ep{(OT*)out, bias, ldo};                      \
    launch_simt_gemm<true, true>(al, bl, ep, M, N, K, 1, s);          \
  }
  if (dtype_out == DGTD_F32) {
    if (act == DGTD_ACT_GELU) DGTD_SIMT_LIN(float, DGTD_ACT_GELU)
    else if (act == DGTD_ACT_RELU) DGTD_SIMT_LIN(float, DGTD_ACT_RELU)
    else DGTD_SIMT_LIN(float, DGTD_ACT_NONE)
  } else {
    if (act == DGTD_ACT_GELU) DGTD_SIMT_LIN(__nv_bfloat16, DGTD_ACT_GELU)
    else if (act == DGTD_ACT_RELU) DGTD_SIMT_LIN(__nv_bfloat16, DGTD_ACT_RELU)
    else DGTD_SIMT_LIN(__nv_bfloat16, DGTD_ACT_NONE)
  }
#undef DGTD_SIMT_LIN
  DGTD_LAUNCH_CHECK("linear(fp32)");
  return 0;
}

int dgtd_linear_ln_fwd(const void* a, const void* w, const float* bias, const float* ln_w, const float* ln_b, float eps,
                       float* out, int M, int N, int K, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(a && w && ln_w && ln_b && out, "linear_ln: null pointer");
  DGTD_CHECK_ARG(M >= 256 && N == 128 && K > 0 && K % 8 == 0, "linear_ln: needs N == 128, M >= 256, K %% 8 == 0 (M=%d N=%d K=%d)", M, N, K);
  DGTD_CHECK_ARG((reinterpret_cast<uintptr_t>(ln_w) & 15) == 0 && (reinterpret_cast<uintptr_t>(ln_b) & 15) == 0 &&
                     (!bias || (reinterpret_cast<uintptr_t>(bias) & 15) == 0) && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
                 "linear_ln: bias / ln_w / ln_b / out must be 16-byte aligned");
  TcParams p{};
  p.M = M; p.N = N; p.K = K; p.bias = bias; p.out = out; p.ldo = N; p.rows_per_sample = 1;
  p.ln_w = ln_w; p.ln_b = ln_b; p.ln_eps = eps;
  const int rc = tc_gemm2_ln_launch((const __nv_bfloat16*)a, K, (const __nv_bfloat16*)w, K, p, (cudaStream_t)stream);
  if (rc > 0) {
    set_error("linear_ln: shape not handled by the 2-CTA kernel");
    return -1;
  }
  if (rc) return rc;
  DGTD_LAUNCH_CHECK("linear_ln(tcgen05)");
  return 0;
}

int dgtd_linear_tf32_fwd(const float* a, const float* w, const float* bias, float* out, int M, int N, int K, int ldo,
                         dgtd_stream_t stream) {
  DGTD_CHECK_ARG(a && w && out, "linear_tf32: null pointer");
  DGTD_CHECK_ARG(M > 0 && N > 0 && N <= 64 && K > 0 && ldo >= N, "linear_tf32: bad shape M=%d N=%d K=%d ldo=%d (N <= 64)", M, N, K,
                 ldo);
  DGTD_CHECK_ARG(K % 4 == 0 && N % 8 == 0 && ldo % 4 == 0, "linear_tf32: K, ldo must be multiples of 4, N of 8");
  DGTD_CHECK_ARG((reinterpret_cast<uintptr_t>(a) & 15) == 0 && (reinterpret_cast<uintptr_t>(w) & 15) == 0 &&
                     (reinterpret_cast<uintptr_t>(out) & 15) == 0,
                 "linear_tf32: operands must be 16-byte aligned");
  TcParams p{};
  p.M = M; p.N = N; p.K = K; p.bias = bias; p.out = out; p.ldo = ldo; p.rows_per_sample = 1;
  const int rc = N <= 32 ? tc_launch_tf32<32>(a, w, p, (cudaStream_t)stream) : tc_launch_tf32<64>(a, w, p, (cudaStream_t)stream);
  if (rc) return rc;
  DGTD_LAUNCH_CHECK("linear_tf32(tcgen05)");
  return 0;
}

int dgtd_linear_lnfold_fwd(const void* a, const void* w, const float* bias, const float* col_s, const float* row_stats,
                           void* out, int M, int N, int K, int ldo, int dtype_out, int act, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(a && w && bias && col_s && row_stats && out, "linear_lnfold: null pointer");
  DGTD_CHECK_ARG(M > 0 && N > 0 && K > 0 && ldo >= N, "linear_lnfold: bad shape M=%d N=%d K=%d ldo=%d", M, N, K, ldo);
  DGTD_CHECK_ARG(act >= 0 && act <= 2, "linear_lnfold: bad activation %d", act);
  DGTD_CHECK_ARG(K % 8 == 0 && N % 8 == 0 && ldo % 8 == 0, "linear_lnfold: K, N, ldo must be multiples of 8");
  DGTD_CHECK_ARG((reinterpret_cast<uintptr_t>(row_stats) & 7) == 0 && (reinterpret_cast<uintptr_t>(col_s) & 15) == 0,
                 "linear_lnfold: row_stats must be 8-byte, col_s 16-byte aligned");
  int rc = tc_linear((const __nv_bfloat16*)a, K, (const __nv_bfloat16*)w, K, bias, out, M, N, K, ldo, dtype_out, act,
                     (cudaStream_t)stream, (const float2*)row_stats, col_s);
  if (rc) return rc;
  DGTD_LAUNCH_CHECK("linear_lnfold(tcgen05)");
  return 0;
}

int dgtd_conv3x3_tc_fwd(const void* x, const void* w, const float* bias, float* out, int B, int h, int wd, int Cp,
                        int Cout, int ldo, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(x && w && out, "conv3x3_tc: null pointer");
  DGTD_CHECK_ARG(B > 0 && h > 0 && wd > 0 && Cp > 0 && Cp % 64 == 0 && Cout > 0 && Cout % 8 == 0 && Cout <= 128 &&
                     ldo >= Cout && ldo % 4 == 0,
                 "conv3x3_tc: Cp must be a multiple of 64, Cout a multiple of 8 and <= 128 (B=%d h=%d w=%d Cp=%d Cout=%d)",
                 B, h, wd, Cp, Cout);
  DGTD_CHECK_ARG((int64_t)B * h * wd < (1ll << 31), "conv3x3_tc: too many pixels");
  DGTD_CHECK_ARG((reinterpret_cast<uintptr_t>(x) & 127) == 0 && (reinterpret_cast<uintptr_t>(w) & 15) == 0 &&
                     (reinterpret_cast<uintptr_t>(out) & 15) == 0,
                 "conv3x3_tc: x must be 128-byte aligned, w / out 16-byte aligned");
  int rc = tc_conv3((const __nv_bfloat16*)x, (const __nv_bfloat16*)w, bias, out, B, h, wd, Cp, Cout, ldo,
                    (cudaStream_t)stream);
  if (rc) return rc;
  DGTD_LAUNCH_CHECK("conv3x3_tc");
  return 0;
}

int dgtd_linear_residual_fwd(const void* a, const void* w, const float* bias, const float* gamma,
                             const float* keep, int rows_per_sample, const float* residual,
                             float* out, int M, int N, int K, int dtype_in, dgtd_stream_t stream) {
  DGTD_CHECK_ARG(a && w && bias && residual && out, "linear_residual: null pointer");
  DGTD_CHECK_ARG(M > 0 && N > 0 && K > 0, "linear_residual: bad shape");
  DGTD_CHECK_ARG(!keep || rows_per_sample > 0, "linear_residual: rows_per_sample required with keep");
  cudaStream_t s = (cudaStream_t)stream;
  if (dtype_in == DGTD_BF16) {
    DGTD_CHECK_ARG(K % 8 == 0 && N % 8 == 0, "linear_residual(bf16): K, N must be multiples of 8");
    int rc = tc_linear_residual((const __nv_bfloat16*)a, K, (const __nv_bfloat16*)w, K, bias, gamma, keep,
                                rows_per_sample, residual, out, M, N, K, s);
    if (rc) return rc;
    DGTD_LAUNCH_CHECK("linear_residual(tcgen05)");
    return 0;
  }
  DGTD_CHECK_ARG(dtype_in == DGTD_F32, "linear_residual: bad dtype_in %d", dtype_in);
  DGTD_CHECK_ARG(K % 4 == 0 && N % 4 == 0, "linear_residual(fp32): K, N must be multiples of 4");
  RowMajorLoader al{(const float*)a, K, 0, M, K};
  RowMajorLoader bl{(const float*)w, K, 0, N, K};
  EpiResidual ep{out, bias, gamma, keep, residual, rows_per_sample > 0 ? rows_per_sample : 1, N};
  launch_simt_gemm<true, true>(al, bl, ep, M, N, K, 1, s);
  DGTD_LAUNCH_CHECK("linear_residual(fp32)");
  return 0;
}

}  // extern "C"
