// TF32 tensor-core (tcgen05 / TMEM) product for the MIXED-PRECISION trailing update of BASELINE config 5:
//     C[m x n] (FP64) = beta * C + alpha * sum_p A_p^T B_p        A_p: k x m, B_p: k x n  (FP32 copies of FP64 operands, col-major)
//
// EXPERIMENTAL -- OFF BY DEFAULT (capital_set_trailing_precision).  Written after the round's GPU budget was spent: it assembles for
// sm_100a (SASS: UTCHMMA / UTMALDG / LDTM, profiles/r02_sass_tf32.md) but its first execution is whoever runs
// tests/test_gpu_zz_late.py.  The default FP64 path never touches this file's kernels.
//
// Why it exists: the reference has no float BLAS path (src/blas/interface.hpp:43-97 is double only); the FP64 trailing update
// (summa::syrk, summa.hpp:143-145) is the one place of the hot path whose arithmetic a user may trade for speed, and the one place
// where Blackwell's 5th-generation tensor cores apply (tcgen05 has no kind::f64).  The panel / base case, R12 and the inverse stay FP64.
//
// B200 design.  Both operands are K-contiguous ("K-major" for UMMA), so a (128 rows x 32 k) FP32 tile is 128 rows of 128 bytes:
// one TMA box per operand per stage (SWIZZLE_128B), consumed in place by tcgen05.mma.kind::tf32 (M = 128, N = 128, K = 8 per
// instruction, four per stage) through shared-memory matrix descriptors; the 128 x 128 FP32 accumulator lives in TMEM (128 lanes x
// 128 columns).  Warp roles: warp 0 lane 0 drives TMA, warp 1 lane 0 issues the MMAs and commits them to the stage's "empty"
// mbarrier, warp 2 owns the TMEM allocation; afterwards all four warps read their 32 lanes with tcgen05.ld (32x32b.x16: thread =
// accumulator row, 16 consecutive columns) and store FP64 -- for a fixed column the 32 lanes of a warp write 32 consecutive rows,
// i.e. coalesced 256-byte segments of the column-major C.
// passes = 3: every operand is split as x = hi + lo (both TF32-representable) and the product accumulates hi*hi + hi*lo + lo*hi in
// the same TMEM tile: FP32-class accuracy at three times the tensor work (still an order of magnitude under the DMMA time).
// Every mbarrier wait is bounded (2 s of %globaltimer): a protocol error ends the kernel with info = -3 instead of hanging the GPU.
#include "common.cuh"
#include <algorithm>

namespace {

constexpr int TBM = 128, TBN = 128, TBK = 32;  // tile; TBK floats = one 128-byte swizzle row
constexpr int TSTAGES = 6;
constexpr int T_A_BYTES = TBM * 128, T_B_BYTES = TBN * 128, T_STAGE_BYTES = T_A_BYTES + T_B_BYTES;
constexpr int T_SMEM = TSTAGES * T_STAGE_BYTES + (2 * TSTAGES + 1) * 8 + 16 + 1024;
constexpr int T_PAIRS_MAX = 6;  // operand classes (<= 2) x passes (<= 3)
constexpr uint32_t T_TMEM_COLS = 128;
// instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 = 1 @ [4,6), a_format / b_format TF32 = 2 @ [7,10) / [10,13),
// a_major = b_major = K (0) @ 15 / 16, N >> 3 @ [17,23), M >> 4 @ [24,29)
constexpr uint32_t T_IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(TBN >> 3) << 17) | ((uint32_t)(TBM >> 4) << 24);
static_assert(T_IDESC == 0x08200910u, "instruction descriptor of tcgen05.mma.kind::tf32 128x128, K-major A and B");

struct Tf32Maps {
  CUtensorMap a[T_PAIRS_MAX];
  CUtensorMap b[T_PAIRS_MAX];
};
struct Tf32Params {
  int M, N, K;
  int npair;
  int flags, noff;
  int gm, gn;
  double alpha, beta;
  double* C;
  long long ldc;
  int* err;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
// false = gave up (2 s): the caller leaves its loop, the kernel ends, the host sees info = -3
__device__ __forceinline__ bool mbar_wait_bounded(uint32_t bar, uint32_t parity, int* err) {
  unsigned long long t0 = 0;
  for (unsigned spin = 0;; spin++) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (ok) return true;
    if ((spin & 1023u) == 1023u) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      if (t0 == 0) t0 = t;
      else if (t - t0 > 2000000000ull || *(volatile int*)err == -3) { atomicExch(err, -3); return false; }
    }
  }
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor), K-major operand, 128-byte swizzle: start address >> 4 @ [0,14),
// leading byte offset @ [16,30) (not used by the hardware for a swizzled K-major operand with one atom along K; 1 as
// cute::UMMA::make_umma_desc<Major::K> sets it), stride byte offset = 8 rows x 128 B = 1024 (>> 4) @ [32,46), version 1 @ 46,
// layout SWIZZLE_128B = 2 @ [61,64).  Tiles are 1024-byte aligned (base_offset 0).
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | (1ull << 16) | ((uint64_t)(1024u >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the mbarrier once every tcgen05.mma issued so far by this thread has completed (implies fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

__global__ void __launch_bounds__(128, 1) gemm_tn_tf32_kernel(const __grid_constant__ Tf32Maps maps, const Tf32Params p) {
  extern __shared__ uint8_t smem_raw[];
  const int tm = blockIdx.x, tn = blockIdx.y;
  const int m0 = tm * TBM, n0 = tn * TBN;
  if ((p.flags & CAPITAL_GEMM_C_UPPER) && m0 > n0 + p.noff + TBN - 1) return;  // tile strictly below the diagonal (whole CTA)
  // an earlier CTA's watchdog fired: the launch is lost, do not spend 2 s per remaining tile (block-uniform decision)
  if (__syncthreads_or(*(volatile int*)p.err == -3)) return;
  const int nk = (p.K + TBK - 1) / TBK;
  const int niter = nk * p.npair;

  const uint32_t raw_u32 = smem_u32(smem_raw);
  const uint32_t smem_base = (raw_u32 + 1023u) & ~1023u;
  const uint32_t full0 = smem_base + TSTAGES * T_STAGE_BYTES;
  const uint32_t empty0 = full0 + TSTAGES * 8;
  const uint32_t tfull = empty0 + TSTAGES * 8;
  const uint32_t tmem_slot = tfull + 8;
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - raw_u32));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < TSTAGES; s++) {
      mbar_init(full0 + s * 8, 1);
      mbar_init(empty0 + s * 8, 1);
    }
    mbar_init(tfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 2) {  // one warp allocates the accumulator's TMEM columns and lets other CTAs of the SM allocate too
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"(T_TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0 && lane == 0) {
    // ---------------- TMA producer ----------------
    int it = 0;
    bool alive = true;
    for (int pr = 0; pr < p.npair && alive; pr++) {
      const CUtensorMap* ma = &maps.a[pr];
      const CUtensorMap* mb = &maps.b[pr];
      for (int j = 0; j < nk; j++, it++) {
        const int s = it % TSTAGES;
        const uint32_t ph = (it / TSTAGES) & 1;
        if (!mbar_wait_bounded(empty0 + s * 8, ph ^ 1, p.err)) { alive = false; break; }
        mbar_expect_tx(full0 + s * 8, T_STAGE_BYTES);
        tma_load_2d(smem_base + s * T_STAGE_BYTES, ma, full0 + s * 8, j * TBK, m0);
        tma_load_2d(smem_base + s * T_STAGE_BYTES + T_A_BYTES, mb, full0 + s * 8, j * TBK, n0);
      }
    }
  } else if (warp == 1 && lane == 0) {
    // ---------------- MMA issuer: one thread on behalf of the CTA ----------------
    for (int it = 0; it < niter; it++) {
      const int s = it % TSTAGES;
      const uint32_t ph = (it / TSTAGES) & 1;
      if (!mbar_wait_bounded(full0 + s * 8, ph, p.err)) break;
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint64_t da = umma_desc_k_sw128(smem_base + s * T_STAGE_BYTES);
      const uint64_t db = umma_desc_k_sw128(smem_base + s * T_STAGE_BYTES + T_A_BYTES);
#pragma unroll
      for (int k8 = 0; k8 < TBK / 8; k8++)  // 8 floats = 32 bytes further along K inside the swizzle row: start address + 2 (>> 4)
        umma_tf32(tmem_base, da + (uint64_t)(2 * k8), db + (uint64_t)(2 * k8), T_IDESC, (it > 0 || k8 > 0) ? 1u : 0u);
      umma_commit(empty0 + s * 8);  // the stage is free again once these MMAs have read it
    }
    umma_commit(tfull);  // the accumulator is complete once everything issued above has retired
  }
  __syncwarp();

  // ---------------- epilogue: all four warps, warp w reads TMEM lanes [32 w, 32 w + 32) ----------------
  const bool have = mbar_wait_bounded(tfull, 0, p.err);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  __syncwarp();
  const int row = m0 + warp * 32 + lane;
  const double alpha = p.alpha, beta = p.beta;
  const bool upper_only = p.flags & CAPITAL_GEMM_C_UPPER;
#pragma unroll 1
  for (int c0 = 0; c0 < TBN; c0 += 16) {
    if (n0 + c0 >= p.N) break;  // uniform over the CTA
    __syncwarp();               // tcgen05.ld is .sync.aligned: the lanes that skipped the stores below rejoin here
    uint32_t v[16];
    const uint32_t taddr = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0;
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    if (!have || row >= p.M) continue;
#pragma unroll
    for (int j = 0; j < 16; j++) {
      const int col = n0 + c0 + j;
      if (col >= p.N || (upper_only && row > col + p.noff)) continue;
      double* cc = p.C + (long long)col * p.ldc + row;
      double r = alpha * (double)__uint_as_float(v[j]);
      if (beta != 0.0) r += beta * *cc;
      *cc = r;
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(T_TMEM_COLS) : "memory");
}

// FP64 window (k x cols, ld) -> FP32 copies rounded to TF32 (cvt.rna): hi, and optionally lo = tf32(x - hi)
__global__ void to_tf32_kernel(long long k, long long cols, const double* src, long long ld, float* hi, float* lo, long long ldf) {
  const long long total = k * cols;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const long long c = idx / k, r = idx - c * k;
    const double x = src[c * ld + r];
    uint32_t h;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"((float)x));
    const float hf = __uint_as_float(h);
    hi[c * ldf + r] = hf;
    if (lo) {
      uint32_t l;
      asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(l) : "f"((float)(x - (double)hf)));
      lo[c * ldf + r] = __uint_as_float(l);
    }
  }
}

capital_status_t make_map_f32(capital_ctx* ctx, CUtensorMap* map, const float* base, int64_t k, int64_t cols, int64_t ldf, int box_cols) {
  cuuint64_t dims[2] = {(cuuint64_t)k, (cuuint64_t)cols};
  cuuint64_t strides[1] = {(cuuint64_t)ldf * 4};
  cuuint32_t box[2] = {(cuuint32_t)TBK, (cuuint32_t)box_cols};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = ctx->encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    ctx->set_error("cuTensorMapEncodeTiled (f32) failed: CUresult " + std::to_string((int)r));
    return CAPITAL_ERR_CUDA;
  }
  return CAPITAL_OK;
}

}  // namespace

capital_status_t gemm_tf32_init(capital_ctx* ctx) {
  CAP_CUDA(cudaFuncSetAttribute(gemm_tn_tf32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, T_SMEM));
  return CAPITAL_OK;
}

// C = beta C + alpha sum over classes A_c^T B_c, operands given in FP64 and converted here (workspaces are per stream: a product on the
// deferred stream must not reuse the buffers of one in flight on the chain).  passes = 1 (TF32) or 3 (split operands).
capital_status_t gemm_tn_tf32_x(capital_ctx* ctx, cudaStream_t st, int64_t m, int64_t n, int64_t k, double alpha, const GemmOperands& ops,
                                double beta, double* C, int64_t ldc, int flags, int noff, int passes) {
  if (m <= 0 || n <= 0 || k <= 0) return CAPITAL_OK;
  if ((passes != 1 && passes != 3) || ops.ncls < 1 || ops.ncls > GEMM_NCLS_MAX || ops.lda < k || ops.ldb < k || ldc < m ||
      (flags & ~CAPITAL_GEMM_C_UPPER) || m >= (1LL << 31) - 256 || n >= (1LL << 31) - 256 || k >= (1LL << 31) - 256) {
    ctx->set_error("gemm_tn_tf32: unsupported arguments (passes 1 or 3, only the C_UPPER structure flag)");
    return CAPITAL_ERR_INVALID;
  }
  if (!ctx->tf32_ready) {
    CAP_TRY(gemm_tf32_init(ctx));
    ctx->tf32_ready = true;
  }
  const std::string tag = stream_tag(ctx, st);
  const int64_t ldf = round_up(k, 4);  // 16-byte rows for TMA
  Tf32Maps maps;
  memset(&maps, 0, sizeof(maps));
  Tf32Params p{};
  int np = 0;
  for (int c = 0; c < ops.ncls; c++) {
    const bool same = ops.A[c] == ops.B[c] && ops.lda == ops.ldb && m == n;
    float *ahi, *alo = nullptr, *bhi, *blo = nullptr;
    const std::string sfx = tag + std::to_string(c);
    CAP_TRY(ctx->workspace("tf32_ahi" + sfx, (size_t)ldf * m * 4, (void**)&ahi));
    if (passes == 3) CAP_TRY(ctx->workspace("tf32_alo" + sfx, (size_t)ldf * m * 4, (void**)&alo));
    const int gr = (int)std::min<long long>(((long long)k * std::max(m, n) + 255) / 256, (long long)ctx->num_sms * 8);
    to_tf32_kernel<<<gr, 256, 0, st>>>(k, m, ops.A[c], ops.lda, ahi, alo, ldf);
    ctx->counters.kernel_launches++;
    if (same) { bhi = ahi; blo = alo; }
    else {
      CAP_TRY(ctx->workspace("tf32_bhi" + sfx, (size_t)ldf * n * 4, (void**)&bhi));
      if (passes == 3) CAP_TRY(ctx->workspace("tf32_blo" + sfx, (size_t)ldf * n * 4, (void**)&blo));
      to_tf32_kernel<<<gr, 256, 0, st>>>(k, n, ops.B[c], ops.ldb, bhi, blo, ldf);
      ctx->counters.kernel_launches++;
    }
    CAP_CUDA(cudaGetLastError());
    const float* pa[3] = {ahi, ahi, alo};
    const float* pb[3] = {bhi, blo, bhi};
    for (int q = 0; q < passes; q++, np++) {
      CAP_TRY(make_map_f32(ctx, &maps.a[np], pa[q], k, m, ldf, TBM));
      CAP_TRY(make_map_f32(ctx, &maps.b[np], pb[q], k, n, ldf, TBN));
    }
  }
  p.M = (int)m; p.N = (int)n; p.K = (int)k; p.npair = np; p.flags = flags; p.noff = noff;
  p.gm = (int)ceil_div(m, TBM); p.gn = (int)ceil_div(n, TBN);
  p.alpha = alpha; p.beta = beta; p.C = C; p.ldc = ldc; p.err = ctx->d_info;
  dim3 grid((unsigned)p.gm, (unsigned)p.gn, 1);
  const int tli = ctx->tl_begin(st, 9, (double)m, (double)n, (double)k);
  gemm_tn_tf32_kernel<<<grid, 128, T_SMEM, st>>>(maps, p);
  ctx->tl_end(st, tli);
  CAP_CUDA(cudaGetLastError());
  ctx->counters.kernel_launches++;
  ctx->tf32_launches++;
  ctx->tf32_flops += 2.0 * (double)m * (double)n * (double)k * ops.ncls * passes * ((flags & CAPITAL_GEMM_C_UPPER) ? 0.5 : 1.0);
  return CAPITAL_OK;
}

capital_status_t gemm_tn_tf32(capital_ctx* ctx, cudaStream_t st, int64_t m, int64_t n, int64_t k, double alpha, const double* A, int64_t lda,
                              const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int flags, int passes) {
  GemmOperands ops;
  ops.A[0] = A; ops.B[0] = B; ops.lda = lda; ops.ldb = ldb;
  return gemm_tn_tf32_x(ctx, st, m, n, k, alpha, ops, beta, C, ldc, flags, 0, passes);
}
