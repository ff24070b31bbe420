// FP64 tensor-core GEMM for sm_100a:  C[m x n] = alpha * A^T B + beta * C   (A: k x m, B: k x n, col-major)
//
// This is the kernel behind every trailing update of the CholInv schedule -- the reference's
// cblas_dgemm(T,N) in summa::syrk_internal (summa.hpp:143-145), cblas_dtrmm in summa::invoke
// (summa.hpp:64,71) and the Gram products of cacqr (cacqr.hpp:15,95) -- with the triangular
// structure the reference throws away (summa.hpp:115-116) turned into skipped k-tiles / output tiles.
//
// B200 design.  FP64 has no tcgen05 path (ptxas: "Unknown modifier .kind::f64"); the FP64 tensor pipe
// is reached through mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4; measured 37.2 TFLOP/s = 64 FMA/clk/SM, see
// profiles/r01_fp64_pipe_ceilings.log).  Both operands are K-contiguous, so a (rows x 16 k) tile is one
// 128-byte row per matrix column: TMA (cp.async.bulk.tensor.2d, SWIZZLE_128B) stages it with one
// instruction per operand per stage from a dedicated producer warp; consumers wait on mbarriers (no
// __syncthreads in the main loop).  Inside a 16-wide k tile the four DMMAs use the k permutation
// {4q+j}: lane q then owns 32 contiguous bytes of every row, read as two conflict-free LDS.128
// (the 128B swizzle XORs the 16B chunk index with row%8, so the 8 lanes of a quarter-warp -- two rows x
// four q -- hit 8 distinct chunks).  Out-of-range rows/columns are zero-filled by TMA, so ragged M/N/K
// need no predicates in the main loop.
#include "common.cuh"
#include <algorithm>

namespace {

struct GemmParams {
  int M, N, K;
  int rowoffA, rowoffB;  // element offset of the operand's first row inside its (16B-aligned) tensor map
  int flags;
  int noff;    // column index of this window of B / C inside the full operand (column-chunked launches)
  int koff;    // row index of this window inside the full operand (k-chunked launches keep the triangular k ranges right)
  int ksplit;  // gridDim.z chunks of the k range; > 1 => epilogue accumulates with atomics (C pre-initialised, beta ignored)
  int ncls;    // operand classes: the contraction runs over ncls (A_i, B_i) pairs with identical shapes (SUMMA k-slices, summa.hpp:185-193)
  int gm, gn;  // tile grid
  double alpha, beta;
  double* C;
  long long ldc;
  double* Ct;       // optional second output: the TRANSPOSE of the result, Ct[row * ldct + col] (tall-skinny apply of CholeskyQR2)
  long long ldct;
  double* kpart;    // split-k: partial tiles of chunk z go to kpart + z * kstride (deterministic two-stage reduction) instead of atomics
  long long kstride, ldk;
  int no_c;         // skip the store to C (only Ct is wanted)
  GemmXDev x;  // depth exchange fused into the epilogue (XMODE != 0)
};

struct GemmMaps {
  CUtensorMap a[GEMM_NCLS_MAX];
  CUtensorMap b[GEMM_NCLS_MAX];
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!ok);
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
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
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

constexpr int BK = 16;  // doubles per k tile = one 128-byte swizzle row

// Warp roles: NCW consumer warps (whole warpgroups) + one producer warpgroup of which a single lane drives TMA.
// Registers are allocated per warpgroup on sm_100, so a 9th warp would be charged as four anyway; with RC > 0 the
// producer group hands its registers to the consumers (setmaxnreg), which is what lets a 64x32 warp tile
// (128 accumulator registers) live without spills.
// XMODE: 0 = plain product; 1 / 2 = depth exchange fused into the epilogue (GemmXDev in common.cuh).
template <int BM, int BN, int WM, int WN, int STAGES, int MINB, int RC, int RP, int XMODE>
__global__ void __launch_bounds__(((BM / WM) * (BN / WN) + 4) * 32, MINB)
    gemm_tn_kernel(const __grid_constant__ GemmMaps maps, const GemmParams p) {
  constexpr int NWM = BM / WM, NWN = BN / WN, NCW = NWM * NWN;
  constexpr int FM = WM / 8, FN = WN / 8;
  constexpr int A_BYTES = BM * 128, B_BYTES = BN * 128, STAGE_BYTES = A_BYTES + B_BYTES;

  extern __shared__ uint8_t smem_raw[];
  const int flags = p.flags;
  const int gm = p.gm, gn = p.gn;
  const int lin = (int)(blockIdx.x + gridDim.x * blockIdx.y);
  // Longest-tile-first over the WHOLE grid: with a triangular operand the k extent depends on one tile coordinate only, so the
  // linear CTA id is mapped to tiles in order of decreasing k extent (row-major over the other coordinate).  The first wave then
  // holds the longest tiles and second residents / the tail get the short ones (a per-column reversal alone interleaves long and
  // short tiles and lets two long tiles share an SM).
  int tm, tn;
  if (flags & CAPITAL_GEMM_A_UPPER) { tm = gm - 1 - lin / gn; tn = lin % gn; }
  else if (flags & CAPITAL_GEMM_B_UPPER) { tn = gn - 1 - lin / gm; tm = lin % gm; }
  else if (flags & CAPITAL_GEMM_A_LOWER) { tm = lin / gn; tn = lin % gn; }
  else if (flags & CAPITAL_GEMM_B_LOWER) { tn = lin / gm; tm = lin % gm; }
  else { tm = lin % gm; tn = lin / gm; }
  if (XMODE == 2 && (tn % p.x.c) != p.x.z) return;  // another layer computes this tile column and stores it here
  const int m0 = tm * BM, n0 = tn * BN;
  const int n0g = n0 + p.noff;  // column position used by the structure tests
  if ((flags & CAPITAL_GEMM_C_UPPER) && m0 > n0g + BN - 1) return;  // tile strictly below the diagonal

  int kb = 0, ke = p.K;
  if (flags & CAPITAL_GEMM_A_UPPER) ke = min(ke, m0 + BM - p.koff);
  if (flags & CAPITAL_GEMM_A_LOWER) kb = max(kb, m0 - p.koff);
  if (flags & CAPITAL_GEMM_B_UPPER) ke = min(ke, n0g + BN - p.koff);
  if (flags & CAPITAL_GEMM_B_LOWER) kb = max(kb, n0g - p.koff);
  kb &= ~(BK - 1);
  int nk = ke > kb ? (ke - kb + BK - 1) / BK : 0;
  if (nk == 0 && p.beta == 1.0 && p.ksplit <= 1) return;  // nothing to add (k-chunk entirely outside the operand's triangle); same on every layer
  if (p.ksplit > 1) {  // this CTA's contiguous chunk of k tiles
    const int per = (nk + p.ksplit - 1) / p.ksplit;
    const int t0 = min(nk, (int)blockIdx.z * per), t1 = min(nk, t0 + per);
    kb += t0 * BK;
    nk = t1 - t0;
    // An empty chunk has nothing to add to C (atomics), but the two-stage reduction reads every chunk's slice of kpart: it stores
    // its zeros there, or the reduction would add whatever an earlier product left in the workspace.
    if (nk == 0 && !p.kpart) return;
  }
  const int niter = nk * p.ncls;  // the k tiles of every operand class, one after the other

  // 1024-byte alignment for the 128B swizzle, computed as an OFFSET into the shared array so that the pointer keeps its
  // shared address space (fragment loads then compile to LDS.128 instead of generic LD.E.128)
  const uint32_t raw_u32 = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw_u32 + 1023u) & ~1023u) - raw_u32);
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t full0 = smem_base + STAGES * STAGE_BYTES;
  const uint32_t empty0 = full0 + STAGES * 8;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; s++) {
      mbar_init(full0 + s * 8, 1);
      mbar_init(empty0 + s * 8, NCW);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();

  if (warp >= NCW) {
    // ---------------- TMA producer warpgroup ----------------
    if (RC > 0) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(RP));
    if (warp == NCW && lane == 0) {
      int it = 0;
      for (int cls = 0; cls < p.ncls; cls++) {
        const CUtensorMap* ma = cls ? &maps.a[1] : &maps.a[0];
        const CUtensorMap* mb = cls ? &maps.b[1] : &maps.b[0];
        for (int j = 0; j < nk; j++, it++) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1;
          mbar_wait(empty0 + s * 8, ph ^ 1);
          mbar_expect_tx(full0 + s * 8, STAGE_BYTES);
          const int kk = kb + j * BK;
          tma_load_2d(smem_base + s * STAGE_BYTES, ma, full0 + s * 8, p.rowoffA + kk, m0);
          tma_load_2d(smem_base + s * STAGE_BYTES + A_BYTES, mb, full0 + s * 8, p.rowoffB + kk, n0);
        }
      }
    }
    return;
  }

  // ---------------- DMMA consumers ----------------
  if (RC > 0) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(RC));
  const int wm = warp % NWM, wn = warp / NWM;
  const int g = lane >> 2, q = lane & 3;
  double acc[FM][FN][2];
#pragma unroll
  for (int i = 0; i < FM; i++)
#pragma unroll
    for (int j = 0; j < FN; j++) acc[i][j][0] = acc[i][j][1] = 0.0;

  const int a_row_off = (wm * WM + g) * 128;
  const int b_row_off = A_BYTES + (wn * WN + g) * 128;
  const int swz[2] = {((2 * q) ^ g) * 16, ((2 * q + 1) ^ g) * 16};

  for (int it = 0; it < niter; it++) {
    const int s = it % STAGES;
    const uint32_t ph = (it / STAGES) & 1;
    mbar_wait(full0 + s * 8, ph);
    const uint8_t* st = smem + s * STAGE_BYTES;
#pragma unroll
    for (int h = 0; h < 2; h++) {
      double2 af[FM], bf[FN];
#pragma unroll
      for (int i = 0; i < FM; i++) af[i] = *reinterpret_cast<const double2*>(st + a_row_off + i * 1024 + swz[h]);
#pragma unroll
      for (int j = 0; j < FN; j++) bf[j] = *reinterpret_cast<const double2*>(st + b_row_off + j * 1024 + swz[h]);
#pragma unroll
      for (int i = 0; i < FM; i++)
#pragma unroll
        for (int j = 0; j < FN; j++) dmma884(acc[i][j][0], acc[i][j][1], af[i].x, bf[j].x);
#pragma unroll
      for (int i = 0; i < FM; i++)
#pragma unroll
        for (int j = 0; j < FN; j++) dmma884(acc[i][j][0], acc[i][j][1], af[i].y, bf[j].y);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(empty0 + s * 8);
  }

  const int nother = (XMODE != 0) ? p.x.c - 1 : 0;

  // ---------------- epilogue: C = alpha * acc + beta * C (to every replica when the exchange is on) ----------------
  const double alpha = p.alpha, beta = p.beta;
  const bool upper_only = flags & CAPITAL_GEMM_C_UPPER;
#pragma unroll
  for (int j = 0; j < FN; j++) {
#pragma unroll
    for (int e = 0; e < 2; e++) {
      const int col = n0 + wn * WN + j * 8 + 2 * q + e;
      if (col >= p.N) continue;
      const long long coff = (long long)col * p.ldc;
      double* cc = p.C + coff;
#pragma unroll
      for (int i = 0; i < FM; i++) {
        const int row = m0 + wm * WM + i * 8 + g;
        if (row >= p.M || (upper_only && row > col + p.noff)) continue;
        double v = alpha * acc[i][j][e];
        if (XMODE == 0 && p.ksplit > 1) {
          if (p.kpart) p.kpart[(long long)blockIdx.z * p.kstride + (long long)col * p.ldk + row] = v;
          else atomicAdd(cc + row, v);
          continue;
        }
        if (beta != 0.0) v += beta * cc[row];
        if (XMODE != 0 || !p.no_c) cc[row] = v;
        if (XMODE == 0 && p.Ct) p.Ct[(long long)row * p.ldct + col] = v;
        if (XMODE != 0) {  // mode 1: the partner's receive buffer for my partial; mode 2: the partner's replica of C
          for (int oi = 0; oi < nother; oi++) p.x.Cpeer[oi][coff + row] = v;
        }
      }
    }
  }
  if (XMODE != 0) __threadfence_system();  // the replicas' stores are performed before the kernel retires (the done flag follows on the stream)
}

template <int BM_, int BN_, int WM, int WN, int STAGES, int MINB, int RC, int RP>
struct GemmCfg {
  static_assert(((BM_ / WM) * (BN_ / WN)) % 4 == 0, "consumer warps must form whole warpgroups");
  static constexpr int BM = BM_, BN = BN_;
  static constexpr int threads = ((BM / WM) * (BN / WN) + 4) * 32;
  static constexpr int smem = STAGES * (BM + BN) * 128 + 2 * STAGES * 8 + 1024;
  template <int XMODE>
  static constexpr auto kernel() { return gemm_tn_kernel<BM, BN, WM, WN, STAGES, MINB, RC, RP, XMODE>; }
};
using CfgBig = GemmCfg<128, 128, 64, 32, 5, 1, 232, 40>;   // 8 consumer warps + producer group, 1 CTA / SM
using CfgSmall = GemmCfg<64, 64, 32, 32, 6, 2, 0, 0>;       // 4 consumer warps + producer group, 2 CTAs / SM

capital_status_t make_map(capital_ctx* ctx, CUtensorMap* map, const double* base, int64_t rows, int64_t cols, int64_t ld,
                          int box_rows_k, int box_cols) {
  cuuint64_t dims[2] = {(cuuint64_t)rows, (cuuint64_t)cols};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 8};
  cuuint32_t box[2] = {(cuuint32_t)box_rows_k, (cuuint32_t)box_cols};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = ctx->encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, (void*)base, dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    ctx->set_error("cuTensorMapEncodeTiled failed: CUresult " + std::to_string((int)r) + " rows=" + std::to_string(rows) +
                   " cols=" + std::to_string(cols) + " ld=" + std::to_string(ld));
    return CAPITAL_ERR_CUDA;
  }
  return CAPITAL_OK;
}

struct GemmExtra {
  double* Ct = nullptr; int64_t ldct = 0; int no_c = 0;
  double* kpart = nullptr; int64_t kstride = 0, ldk = 0;
};
template <class Cfg>
capital_status_t launch(capital_ctx* ctx, cudaStream_t st, int64_t m, int64_t n, int64_t k, double alpha, GemmOperands ops, double beta, double* C,
                        int64_t ldc, int flags, int ksplit, int koff, int noff, const GemmXDev* x, const GemmExtra* ex = nullptr) {
  constexpr int BM = Cfg::BM, BN = Cfg::BN;
  GemmParams p{};
  if (ex) { p.Ct = ex->Ct; p.ldct = ex->ldct; p.no_c = ex->no_c; p.kpart = ex->kpart; p.kstride = ex->kstride; p.ldk = ex->ldk; }
  p.M = (int)m; p.N = (int)n; p.K = (int)k; p.flags = flags; p.alpha = alpha; p.beta = beta; p.C = C; p.ldc = ldc; p.ksplit = ksplit; p.koff = koff; p.noff = noff;
  p.ncls = ops.ncls;
  // TMA fetches 16-byte granules: a window that starts on an odd row (8-byte aligned only) cannot be addressed by
  // box coordinates, so it is first copied to an aligned scratch (O(k m) bytes against O(k m n) flops; only odd
  // split points of non-power-of-two sizes ever take this path).  One scratch per stream: a product on another stream may still be
  // reading its own copy.
  const int sid = ctx->stream_id(st);
  int64_t la[GEMM_NCLS_MAX], lb[GEMM_NCLS_MAX];
  for (int c = 0; c < ops.ncls; c++) {
    la[c] = ops.lda; lb[c] = ops.ldb;
    const bool same = (ops.A[c] == ops.B[c] && ops.lda == ops.ldb && m == n);
    const int64_t lds = round_up(k, 2);
    if ((uintptr_t)ops.A[c] & 15) {
      double* sc;
      CAP_TRY(ctx->workspace("gemm_align" + std::to_string(gemm_align_slot(sid, 0, c)), (size_t)lds * m * 8, (void**)&sc));
      CAP_TRY(copy_block(ctx, st, k, m, ops.A[c], ops.lda, sc, lds));
      if (same) { ops.B[c] = sc; lb[c] = lds; }
      ops.A[c] = sc; la[c] = lds;
    }
    if ((uintptr_t)ops.B[c] & 15) {
      double* sc;
      CAP_TRY(ctx->workspace("gemm_align" + std::to_string(gemm_align_slot(sid, 1, c)), (size_t)lds * n * 8, (void**)&sc));
      CAP_TRY(copy_block(ctx, st, k, n, ops.B[c], ops.ldb, sc, lds));
      ops.B[c] = sc; lb[c] = lds;
    }
  }
  p.rowoffA = 0;
  p.rowoffB = 0;
  GemmMaps maps;
  memset(&maps, 0, sizeof(maps));
  for (int c = 0; c < ops.ncls; c++) {
    CAP_TRY(make_map(ctx, &maps.a[c], ops.A[c], k, m, la[c], BK, BM));
    CAP_TRY(make_map(ctx, &maps.b[c], ops.B[c], k, n, lb[c], BK, BN));
  }
  p.gm = (int)ceil_div(m, BM); p.gn = (int)ceil_div(n, BN);
  const int xmode = x ? x->mode : 0;
  if (xmode) p.x = *x;
  if (xmode == 1) {
    dim3 grid((unsigned)p.gm, (unsigned)p.gn, 1);
    Cfg::template kernel<1>()<<<grid, Cfg::threads, Cfg::smem, st>>>(maps, p);
  } else if (xmode == 2) {
    dim3 grid((unsigned)p.gm, (unsigned)p.gn, 1);
    Cfg::template kernel<2>()<<<grid, Cfg::threads, Cfg::smem, st>>>(maps, p);
  } else {
    dim3 grid((unsigned)p.gm, (unsigned)p.gn, (unsigned)ksplit);
    Cfg::template kernel<0>()<<<grid, Cfg::threads, Cfg::smem, st>>>(maps, p);
  }
  CAP_CUDA(cudaGetLastError());
  return CAPITAL_OK;
}

}  // namespace

// ---- FP64 tensor-pipe ceiling, measured in place ------------------------------------------------------------------
// Register-resident DMMA.8x8x4 loop (8 independent accumulator pairs per warp, 8 warps per SM): what the tensor pipe delivers with
// no memory traffic at all.  bench.py runs it next to the timed steps so that `roofline.peak` is a number of THIS device at THIS
// clock, not a constant from a file.
__global__ void __launch_bounds__(256) dmma_peak_kernel(double* out, int iters, double s) {
  double c[8][2];
#pragma unroll
  for (int i = 0; i < 8; i++) { c[i][0] = 0.0; c[i][1] = 0.0; }
  const double a = s + threadIdx.x * 1e-6, b = 1.0 - s;
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < 8; i++)
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c[i][0]), "+d"(c[i][1]) : "d"(a), "d"(b));
  }
  double r = 0.0;
#pragma unroll
  for (int i = 0; i < 8; i++) r += c[i][0] + c[i][1];
  if (r == 123.456) out[0] = r;
}
capital_status_t gemm_probe_dmma(capital_ctx* ctx, double* tflops, double* ms_out) {
  const int iters = 100000, blocks = ctx->num_sms;
  cudaStream_t st = ctx->stream;
  dmma_peak_kernel<<<blocks, 256, 0, st>>>(ctx->d_scalars + 8, iters / 10, 0.5);  // warm-up
  CAP_CUDA(cudaEventRecord(ctx->ev_start, st));
  dmma_peak_kernel<<<blocks, 256, 0, st>>>(ctx->d_scalars + 8, iters, 0.5);
  CAP_CUDA(cudaEventRecord(ctx->ev_stop, st));
  CAP_CUDA(cudaStreamSynchronize(st));
  float ms = 0;
  CAP_CUDA(cudaEventElapsedTime(&ms, ctx->ev_start, ctx->ev_stop));
  const double flops = 2.0 * 256.0 * 8.0 * (double)iters * 8.0 * (double)blocks;  // 8x8x4 MACs x 8 accumulators x 8 warps x blocks
  *tflops = flops / (ms * 1e-3) / 1e12;
  *ms_out = ms;
  return CAPITAL_OK;
}

// Per-device kernel attributes (the >48 KB dynamic shared memory opt-in is a per-device property): called from capital_create
// after cudaSetDevice, so that every context's device is prepared whatever the process did before.
capital_status_t gemm_tn_init(capital_ctx* ctx) {
  CAP_CUDA(cudaFuncSetAttribute(CfgBig::kernel<0>(), cudaFuncAttributeMaxDynamicSharedMemorySize, CfgBig::smem));
  CAP_CUDA(cudaFuncSetAttribute(CfgBig::kernel<1>(), cudaFuncAttributeMaxDynamicSharedMemorySize, CfgBig::smem));
  CAP_CUDA(cudaFuncSetAttribute(CfgBig::kernel<2>(), cudaFuncAttributeMaxDynamicSharedMemorySize, CfgBig::smem));
  CAP_CUDA(cudaFuncSetAttribute(CfgSmall::kernel<0>(), cudaFuncAttributeMaxDynamicSharedMemorySize, CfgSmall::smem));
  CAP_CUDA(cudaFuncSetAttribute(CfgSmall::kernel<1>(), cudaFuncAttributeMaxDynamicSharedMemorySize, CfgSmall::smem));
  CAP_CUDA(cudaFuncSetAttribute(CfgSmall::kernel<2>(), cudaFuncAttributeMaxDynamicSharedMemorySize, CfgSmall::smem));
  return CAPITAL_OK;
}

// which tile configuration a product of this output shape runs with
static inline bool gemm_uses_big(const capital_ctx* ctx, int64_t m, int64_t n) { return ceil_div(m, 128) * ceil_div(n, 128) >= ctx->num_sms; }

// second stage of the deterministic split-k: C = sum over the chunks, in chunk order
__global__ void splitk_reduce_kernel(long long rows, long long cols, const double* part, long long kstride, long long ldk, int nchunk, double* C,
                                     long long ldc, int upper_only) {
  const long long total = rows * cols;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const long long c = idx / rows, r = idx - c * rows;
    if (upper_only && r > c) continue;
    double s = 0.0;
    for (int z = 0; z < nchunk; z++) s += part[(long long)z * kstride + c * ldk + r];
    C[c * ldc + r] = s;
  }
}

// Split-K variant for short-and-fat products (the tall-skinny Gram matrix, cacqr.hpp:15): C = alpha A^T B with the k range cut
// into chunks, one CTA per (tile, chunk); the partial tiles go to a workspace and are added up in chunk order by a second kernel
// (deterministic: the same bits on every run and on every rank).  128 x 128 tiles when the output has them: 3 upper tiles x 49
// chunks fill the 148 SMs for a 256 x 256 Gram matrix.
capital_status_t gemm_tn_splitk(capital_ctx* ctx, cudaStream_t st, int64_t m, int64_t n, int64_t k, double alpha, const double* A,
                                int64_t lda, const double* B, int64_t ldb, double* C, int64_t ldc, int flags) {
  if (m <= 0 || n <= 0 || k <= 0) return CAPITAL_OK;
  if (lda < k || ldb < k || ldc < m || (lda & 1) || (ldb & 1)) return CAPITAL_ERR_INVALID;
  const bool big = m >= 128 && n >= 128;
  const int64_t t = big ? 128 : 64;
  const int64_t gm = ceil_div(m, t), gn = ceil_div(n, t);
  int64_t tiles = gm * gn;
  if ((flags & CAPITAL_GEMM_C_UPPER) && gm == gn) tiles = gm * (gm + 1) / 2;  // tiles below the diagonal return at once
  int64_t ks = ceil_div((int64_t)ctx->num_sms * (big ? 1 : 2), tiles);
  const int64_t max_ks = ceil_div(k, 16 * 32);  // at least 32 k-tiles per chunk
  if (ks > max_ks) ks = max_ks;
  if (ks < 1) ks = 1;
  ctx->counters.kernel_launches += 2;
  ctx->counters.gemm_launches++;
  ctx->counters.gemm_flops += 2.0 * (double)m * (double)n * (double)k * ((flags & CAPITAL_GEMM_C_UPPER) ? 0.5 : 1.0);
  GemmOperands ops;
  ops.A[0] = A; ops.B[0] = B; ops.lda = lda; ops.ldb = ldb;
  if (ks == 1) {  // one chunk: the tile is stored straight into C
    ctx->counters.kernel_launches--;
    if (big) return launch<CfgBig>(ctx, st, m, n, k, alpha, ops, 0.0, C, ldc, flags, 1, 0, 0, nullptr);
    return launch<CfgSmall>(ctx, st, m, n, k, alpha, ops, 0.0, C, ldc, flags, 1, 0, 0, nullptr);
  }
  GemmExtra ex;
  ex.ldk = round_up(m, 2); ex.kstride = ex.ldk * n;
  CAP_TRY(ctx->workspace("splitk_part", (size_t)ks * ex.kstride * 8, (void**)&ex.kpart));
  const int tli = ctx->tl_begin(st, big ? 1 : 2, (double)m, (double)n, (double)k);
  if (big) CAP_TRY((launch<CfgBig>(ctx, st, m, n, k, alpha, ops, 0.0, C, ldc, flags, (int)ks, 0, 0, nullptr, &ex)));
  else CAP_TRY((launch<CfgSmall>(ctx, st, m, n, k, alpha, ops, 0.0, C, ldc, flags, (int)ks, 0, 0, nullptr, &ex)));
  ctx->tl_end(st, tli);
  const long long total = m * n;
  const int gr = (int)std::min<long long>((total + 255) / 256, (long long)ctx->num_sms * 4);
  splitk_reduce_kernel<<<gr, 256, 0, st>>>(m, n, ex.kpart, ex.kstride, ex.ldk, (int)ks, C, ldc, (flags & CAPITAL_GEMM_C_UPPER) ? 1 : 0);
  CAP_CUDA(cudaGetLastError());
  return CAPITAL_OK;
}

// C = alpha A^T B with the result ALSO (or only, C == nullptr) stored transposed into Ct (ldct).  The tall-skinny apply of
// CholeskyQR2, Q <- Q Rinv, is computed as (Q Rinv)^T = Rinv^T Q^T with K-contiguous operands; the transposed store writes Q back in
// its column-major layout from the epilogue (no separate transpose pass), the plain store keeps Q^T for the next sweep.
capital_status_t gemm_tn_t(capital_ctx* ctx, cudaStream_t st, int64_t m, int64_t n, int64_t k, double alpha, const double* A, int64_t lda,
                           const double* B, int64_t ldb, double* C, int64_t ldc, double* Ct, int64_t ldct, int flags) {
  if (m <= 0 || n <= 0 || k <= 0) return CAPITAL_OK;
  if (lda < k || ldb < k || (C && ldc < m) || !Ct || ldct < n || (lda & 1) || (ldb & 1)) return CAPITAL_ERR_INVALID;
  ctx->counters.kernel_launches++;
  ctx->counters.gemm_launches++;
  const bool atri = flags & (CAPITAL_GEMM_A_UPPER | CAPITAL_GEMM_A_LOWER);
  ctx->counters.gemm_flops += atri ? (double)n * (double)m * (double)(m + 1) : 2.0 * (double)m * (double)n * (double)k;
  GemmOperands ops;
  ops.A[0] = A; ops.B[0] = B; ops.lda = lda; ops.ldb = ldb;
  GemmExtra ex;
  ex.Ct = Ct; ex.ldct = ldct; ex.no_c = C ? 0 : 1;
  const bool big = gemm_uses_big(ctx, m, n);
  const int tli = ctx->tl_begin(st, big ? 1 : 2, (double)m, (double)n, (double)k);
  capital_status_t rs;
  if (big) rs = launch<CfgBig>(ctx, st, m, n, k, alpha, ops, 0.0, C ? C : Ct, C ? ldc : m, flags, 1, 0, 0, nullptr, &ex);
  else rs = launch<CfgSmall>(ctx, st, m, n, k, alpha, ops, 0.0, C ? C : Ct, C ? ldc : m, flags, 1, 0, 0, nullptr, &ex);
  ctx->tl_end(st, tli);
  return rs;
}

// Same product issued as a sequence of k-chunked launches (C accumulates).  Used for deferred work on the low-priority
// stream: a 128x128 tile with k = 8192 occupies its SM for ~1 ms, which would make the latency-critical kernels of the
// high-priority stream wait that long for an SM; chunks of `kc` bound the wait to kc/16 k-tiles.
capital_status_t gemm_tn_chunked(capital_ctx* ctx, cudaStream_t st, int64_t m, int64_t n, int64_t k, double alpha, const double* A,
                                 int64_t lda, const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int flags, int64_t kc) {
  if (kc <= 0 || k <= kc + kc / 2) return gemm_tn(ctx, st, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, flags);
  for (int64_t k0 = 0; k0 < k; k0 += kc) {
    const int64_t kk = (k - k0 < kc + kc / 2) ? k - k0 : kc;
    CAP_TRY(gemm_tn_off(ctx, st, m, n, kk, alpha, A + k0, lda, B + k0, ldb, k0 == 0 ? beta : 1.0, C, ldc, flags, (int)k0, 0));
    if (kk != kc) break;
  }
  return CAPITAL_OK;
}

capital_status_t gemm_tn(capital_ctx* ctx, cudaStream_t st, int64_t m, int64_t n, int64_t k, double alpha, const double* A,
                         int64_t lda, const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int flags) {
  return gemm_tn_off(ctx, st, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc, flags, 0, 0);
}

capital_status_t gemm_tn_off(capital_ctx* ctx, cudaStream_t st, int64_t m, int64_t n, int64_t k, double alpha, const double* A,
                             int64_t lda, const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int flags, int koff, int noff) {
  GemmOperands ops;
  ops.A[0] = A; ops.B[0] = B; ops.lda = lda; ops.ldb = ldb;
  return gemm_tn_x(ctx, st, m, n, k, alpha, ops, beta, C, ldc, flags, koff, noff, nullptr);
}

// General form: `ops.ncls` operand classes, optional fused depth exchange (see GemmXDev).  With an exchange every layer must call
// this with the same shapes and flags (the tile grid and the tile ownership are functions of them only).
capital_status_t gemm_tn_x(capital_ctx* ctx, cudaStream_t st, int64_t m, int64_t n, int64_t k, double alpha, const GemmOperands& ops,
                           double beta, double* C, int64_t ldc, int flags, int koff, int noff, const GemmXDev* x) {
  if (m <= 0 || n <= 0) return CAPITAL_OK;
  bool bad = k < 0 || ops.lda < k || ops.ldb < k || ldc < m || (ops.lda & 1) || (ops.ldb & 1) || ops.ncls < 1 || ops.ncls > GEMM_NCLS_MAX;
  for (int c = 0; !bad && c < ops.ncls; c++) bad = !ops.A[c] || !ops.B[c] || ((uintptr_t)ops.A[c] & 7) || ((uintptr_t)ops.B[c] & 7);
  if (bad) {
    ctx->set_error("gemm_tn: invalid/unsupported leading dimensions (lda, ldb must be even and >= k)");
    return CAPITAL_ERR_INVALID;
  }
  if (k == 0) { ctx->set_error("gemm_tn: k must be positive"); return CAPITAL_ERR_INVALID; }
  if (m >= (1LL << 31) || n >= (1LL << 31) || k >= (1LL << 31) - 16) return CAPITAL_ERR_INVALID;
  if (x && x->mode && (x->c < 2 || x->c - 1 > GEMM_XPEERS_MAX)) { ctx->set_error("gemm_tn: exchange over more than 4 layers"); return CAPITAL_ERR_UNSUPPORTED; }
  if (x && x->mode == 1 && beta != 0.0) { ctx->set_error("gemm_tn: a partial product (mode 1) cannot accumulate"); return CAPITAL_ERR_INVALID; }
  ctx->counters.kernel_launches++;
  ctx->counters.gemm_launches++;
  // algorithmic flops of this product on THIS device (structure exploited exactly, not tile-rounded)
  double f = 2.0 * (double)m * (double)n * (double)k;
  const bool atri = flags & (CAPITAL_GEMM_A_UPPER | CAPITAL_GEMM_A_LOWER), btri = flags & (CAPITAL_GEMM_B_UPPER | CAPITAL_GEMM_B_LOWER);
  if (atri && btri) f = 2.0 * (double)m * (double)n * (double)k / 3.0;
  else if (atri) f = (double)n * (double)m * (double)(m + 1);
  else if (btri && (flags & CAPITAL_GEMM_B_UPPER) && noff > 0 && koff == 0 && k >= noff + n) f = (double)m * (double)n * (double)(2 * (int64_t)noff + n + 1);
  else if (btri) f = (double)m * (double)n * (double)(n + 1);
  else if (flags & CAPITAL_GEMM_C_UPPER) f = (double)k * (double)m * (double)(m + 1);
  f *= ops.ncls;
  if (x && x->mode == 2) f /= x->c;  // this layer computes every c-th tile column
  ctx->counters.gemm_flops += f;
  if (gemm_uses_big(ctx, m, n)) {
    // dominant kernel: optionally bracketed by events on its own stream (capital_profile_begin/end)
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (ctx->profiling) {
      CAP_TRY(ctx->prof_event(&e0)); CAP_TRY(ctx->prof_event(&e1));
      CAP_CUDA(cudaEventRecord(e0, st));
    }
    const int tli = ctx->tl_begin(st, 1, (double)m, (double)n, (double)k * ops.ncls);
    CAP_TRY((launch<CfgBig>(ctx, st, m, n, k, alpha, ops, beta, C, ldc, flags, 1, koff, noff, x)));
    ctx->tl_end(st, tli);
    if (ctx->profiling) {
      CAP_CUDA(cudaEventRecord(e1, st));
      ctx->prof_recs.push_back({e0, e1, f});
    }
    return CAPITAL_OK;
  }
  const int tli = ctx->tl_begin(st, 2, (double)m, (double)n, (double)k * ops.ncls);
  const capital_status_t rs = launch<CfgSmall>(ctx, st, m, n, k, alpha, ops, beta, C, ldc, flags, 1, koff, noff, x);
  ctx->tl_end(st, tli);
  return rs;
}
