// capital_b200 -- shared declarations for the CUDA translation units (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>
#include <map>
#include "../../include/capital_b200.h"

#define CAP_CUDA(call)                                                                                    \
  do {                                                                                                     \
    cudaError_t e__ = (call);                                                                              \
    if (e__ != cudaSuccess) {                                                                              \
      ctx->set_error(std::string(#call) + ": " + cudaGetErrorString(e__) + " (" + __FILE__ + ":" +         \
                     std::to_string(__LINE__) + ")");                                                      \
      return CAPITAL_ERR_CUDA;                                                                             \
    }                                                                                                      \
  } while (0)

#define CAP_TRY(call)                                  \
  do {                                                 \
    capital_status_t s__ = (call);                     \
    if (s__ != CAPITAL_OK) return s__;                 \
  } while (0)

typedef CUresult (*cuTensorMapEncodeTiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                              const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                              CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                              CUtensorMapFloatOOBfill);

struct DeviceBuf {
  void* p = nullptr;
  size_t bytes = 0;
};

struct capital_ctx {
  capital_grid_t grid{};
  int device = 0;
  int num_sms = 148;
  cudaStream_t stream = nullptr;   // main stream (caller's or owned)
  cudaStream_t side = nullptr;     // low-priority stream: deferred ("far") trailing updates, T^T products; lives in a green context
  void* green = nullptr;           // (CUgreenCtx) SM partition of the deferred stream, see make_green_side_stream (api.cu)
  int side_sms = 0;                // SMs of that partition (0: no partition)
  cudaStream_t side_deep[2] = {nullptr, nullptr};  // deferred streams of recursion depths 1 and 2 (multi-GPU schedule), same partition, rising priority
  cudaStream_t hi = nullptr;       // high-priority stream: the critical chain of the recursion
  cudaStream_t copy_in = nullptr, copy_out = nullptr;  // H2D / D2H streams of the host-pointer path
  // EXPERIMENTAL, off by default [env CAPITAL_ZC_OUT=1]: host outputs leave block by block through a kernel that stores straight
  // into the pinned packed arrays (partial columns can leave as soon as they are final; see profiles/r01f_e2e_notes.md)
  cudaStream_t zc_out = nullptr;
  int zc_mode = 0, zc_ctas = 8, zc_depth = 3;  // [env CAPITAL_ZC_CTAS, CAPITAL_ZC_DEPTH]
  std::vector<cudaEvent_t> dep_pool;  // dependency events (timing disabled), recycled per factor call
  size_t dep_used = 0;
  std::vector<cudaEvent_t> io_pool;   // events of the host-pointer streaming path
  size_t io_used = 0;
  bool own_stream = false;
  cudaEvent_t ev_start = nullptr, ev_stop = nullptr, ev_fork = nullptr, ev_join = nullptr;
  cuTensorMapEncodeTiled_fn encode = nullptr;
  capital_counters_t counters{};
  std::string err;
  int* d_info = nullptr;           // device flag: first non-SPD pivot (0 = ok)
  double* d_scalars = nullptr;     // device scratch for reductions (16 doubles)
  std::map<std::string, DeviceBuf> pool;  // named, grow-only workspace (the reference's `info` tables, cholinv.h:35-40)
  // pinned staging for host-pointer callers
  void* pinned = nullptr;
  size_t pinned_bytes = 0;
  // multi-GPU: peer layer (peer.cuh) -- IPC-mapped arenas and flags; NCCL (dlopen'ed) only bootstraps the handle exchange
  void* comm_world = nullptr;          // ncclComm_t, when capital_comm_init was used
  void* peer = nullptr;                // Peer*
  std::vector<cudaEvent_t> comm_pool;  // dependency events of the distributed schedules, recycled per call
  size_t comm_used = 0;
  std::string arena_signature;         // which layout the peer arena currently holds (a new layout starts from zeros)

  // per-launch timing of the dominant kernel (gemm_tn 128x128), off by default
  struct ProfRec { cudaEvent_t e0, e1; double flops; };
  bool profiling = false;
  int64_t kchunk = 0;       // k-chunking of deferred GEMMs (env CAPITAL_KCHUNK); measured r01: 0 (off) is fastest, see profiles/r01c_notes.md
  int64_t far_min = 2048;   // trailing updates at least this large are split into near (critical) / far (deferred)   [env CAPITAL_FAR_MIN]
  int64_t side_min = 1024;  // nodes whose left part is at least this large defer T^T to the low-priority stream      [env CAPITAL_SIDE_MIN]; swept in r01: 256 -> 68.9 ms, 1024 -> 67.0 ms
  bool no_overlap = false;  // debug / measurement: run the recursion on one stream
  // EXPERIMENTAL, off by default (capital_set_trailing_precision): trailing updates A22 -= R12^T R12 on the TF32 tensor cores
  // (gemm_tf32.cu); 0 = FP64 DMMA, 1 = TF32, 3 = 3 x TF32 with split operands.  Products with k below tf32_min_k stay FP64.
  int trailing_mode = 0;
  bool tf32_ready = false;  // the TF32 kernel's attributes are set at its first use, never by the default FP64 path
  int64_t tf32_min_k = 256;
  int64_t tf32_launches = 0;
  double tf32_flops = 0.0;
  std::vector<cudaEvent_t> prof_pool;
  size_t prof_used = 0;
  std::vector<ProfRec> prof_recs;
  capital_status_t prof_event(cudaEvent_t* out) {
    if (prof_used == prof_pool.size()) {
      cudaEvent_t e;
      if (cudaEventCreate(&e) != cudaSuccess) { err = "cudaEventCreate failed"; return CAPITAL_ERR_CUDA; }
      prof_pool.push_back(e);
    }
    *out = prof_pool[prof_used++];
    return CAPITAL_OK;
  }

  // timeline (debug / profiling): CUDA events around every launch of the schedule, read back by capital_timeline_end
  struct TlRec { cudaEvent_t e0, e1; int sid, kind; double a, b, c; };
  bool timeline = false;
  std::vector<TlRec> tl;
  std::vector<cudaEvent_t> tl_pool;
  size_t tl_used = 0;
  int stream_id(cudaStream_t st) const;  // 0 caller, 1 chain, 2-4 deferred (depth 0-2), 5-9 push streams, 10 copy-in, 11 copy-out
  int tl_begin(cudaStream_t st, int kind, double a = 0, double b = 0, double c = 0);
  void tl_end(cudaStream_t st, int idx);

  void set_error(const std::string& s) { err = s; }
  capital_status_t workspace(const std::string& name, size_t bytes, void** out);
  capital_status_t pinned_buf(size_t bytes, void** out);
};

// ---- gemm_tn.cu -------------------------------------------------------------------------------
capital_status_t gemm_tn_init(capital_ctx* ctx);  // per-device kernel attributes
capital_status_t leaf_init(capital_ctx* ctx);
capital_status_t gemm_probe_dmma(capital_ctx* ctx, double* tflops, double* ms);

// Multi-GPU form of the product (dist.cu).  (1) The contraction may run over several operand CLASSES -- the k-slices owned by
// different process rows (summa.hpp:185-193), resident in local mirrors -- inside one launch, accumulators staying in
// registers.  (2) The first half of the reference's depth reduction (MPI_Allreduce over the c layers, summa.hpp:236) is fused
// into the epilogue over peer-mapped memory: every stored value also goes, over NVLink, into buffers of the other layers.
//   mode 1 (k split over layers, c == d): C is this layer's PARTIAL-product buffer and Cpeer[i] the receive buffer that the i-th
//          other layer keeps for this layer: when the kernel has retired on every layer (one flag handshake), each layer holds all
//          c partials and adds them up in layer order with one streaming pass (dist.cu: reduce_partials) -- identical bits in
//          every replica, no collective call, no in-kernel waiting.
//   mode 2 (n split, d == 1): layer tn mod c computes tile column tn with the full k range and stores the FINAL values into its own
//          C and into the C replica of every other layer (Cpeer[i]).
constexpr int GEMM_NCLS_MAX = 2;
constexpr int GEMM_XPEERS_MAX = 3;
struct GemmXDev {
  int mode, c, z;
  double* Cpeer[GEMM_XPEERS_MAX];  // same window as C inside the i-th OTHER layer's buffer
};
struct GemmOperands {
  int ncls = 1;
  const double* A[GEMM_NCLS_MAX] = {nullptr, nullptr};
  const double* B[GEMM_NCLS_MAX] = {nullptr, nullptr};
  int64_t lda = 0, ldb = 0;
};
// Work enqueued on different streams of a context may run at the same time, so a workspace that a kernel reads after the host call
// has returned is kept per stream (capital_ctx::stream_id; the distributed schedule numbers its streams the same way).
static inline std::string stream_tag(const capital_ctx* ctx, cudaStream_t st) {
  const int s = ctx->stream_id(st);
  return s ? "_s" + std::to_string(s) : std::string();
}
// The scratch that gemm_tn copies an operand starting on an odd row into (operand 0 = A, 1 = B; operand class cls), on stream
// `stream_id`.  The dry run of the distributed schedule records its uses under the same number.
static inline int gemm_align_slot(int stream_id, int operand, int cls) { return (stream_id * 2 + operand) * GEMM_NCLS_MAX + cls; }
capital_status_t gemm_tn_x(capital_ctx* ctx, cudaStream_t st, int64_t m, int64_t n, int64_t k, double alpha, const GemmOperands& ops,
                           double beta, double* C, int64_t ldc, int flags, int koff, int noff, const GemmXDev* x);
capital_status_t gemm_tn(capital_ctx* ctx, cudaStream_t st, int64_t m, int64_t n, int64_t k, double alpha, const double* A,
                         int64_t lda, const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int flags);

capital_status_t gemm_tn_off(capital_ctx* ctx, cudaStream_t st, int64_t m, int64_t n, int64_t k, double alpha, const double* A,
                             int64_t lda, const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int flags, int koff, int noff = 0);
capital_status_t gemm_tn_chunked(capital_ctx* ctx, cudaStream_t st, int64_t m, int64_t n, int64_t k, double alpha, const double* A,
                                 int64_t lda, const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int flags, int64_t kc);
capital_status_t gemm_tn_splitk(capital_ctx* ctx, cudaStream_t st, int64_t m, int64_t n, int64_t k, double alpha, const double* A,
                                int64_t lda, const double* B, int64_t ldb, double* C, int64_t ldc, int flags);
capital_status_t gemm_tn_t(capital_ctx* ctx, cudaStream_t st, int64_t m, int64_t n, int64_t k, double alpha, const double* A, int64_t lda,
                           const double* B, int64_t ldb, double* C, int64_t ldc, double* Ct, int64_t ldct, int flags);

// ---- gemm_tf32.cu (experimental mixed-precision trailing update, BASELINE config 5) ----------------------------
capital_status_t gemm_tf32_init(capital_ctx* ctx);
capital_status_t gemm_tn_tf32(capital_ctx* ctx, cudaStream_t st, int64_t m, int64_t n, int64_t k, double alpha, const double* A, int64_t lda,
                              const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int flags, int passes);
capital_status_t gemm_tn_tf32_x(capital_ctx* ctx, cudaStream_t st, int64_t m, int64_t n, int64_t k, double alpha, const GemmOperands& ops,
                                double beta, double* C, int64_t ldc, int flags, int noff, int passes);
// the trailing update of one node: FP64 DMMA by default, TF32 when the context asks for it and the contraction is long enough
static inline bool trailing_uses_tf32(const capital_ctx* ctx, int64_t k) { return ctx->trailing_mode != 0 && k >= ctx->tf32_min_k; }

// ---- layout.cu --------------------------------------------------------------------------------
capital_status_t transpose_block(capital_ctx* ctx, cudaStream_t st, int64_t rows, int64_t cols, const double* src,
                                 int64_t lds, double* dst, int64_t ldd, double scale);
capital_status_t copy_block(capital_ctx* ctx, cudaStream_t st, int64_t rows, int64_t cols, const double* src, int64_t lds,
                            double* dst, int64_t ldd);
capital_status_t zero_block(capital_ctx* ctx, cudaStream_t st, int64_t rows, int64_t cols, double* dst, int64_t ldd);
capital_status_t zero_band(capital_ctx* ctx, cudaStream_t st, int64_t n, double* a, int64_t ld);
capital_status_t pack_upper(capital_ctx* ctx, cudaStream_t st, int64_t n, const double* src, int64_t lds, double* packed,
                            int zero_diag, int64_t col_begin = 0, int64_t col_end = -1);
capital_status_t emit_block_packed(capital_ctx* ctx, cudaStream_t st, const double* src, int64_t lds, double* packed, int64_t r0, int64_t r1,
                                   int64_t c0, int64_t c1, int ctas);
capital_status_t unpack_upper(capital_ctx* ctx, cudaStream_t st, int64_t n, const double* packed, double* dst, int64_t ldd);
capital_status_t triu_copy(capital_ctx* ctx, cudaStream_t st, int64_t n, const double* src, int64_t lds, double* dst,
                           int64_t ldd, int zero_diag);
capital_status_t gen_symmetric(capital_ctx* ctx, cudaStream_t st, double* A, int64_t ld, int64_t lrows, int64_t lcols,
                               int64_t n_global, int x, int y, int d, int diag_dom);
capital_status_t gen_random(capital_ctx* ctx, cudaStream_t st, double* A, int64_t ld, int64_t lrows, int64_t lcols,
                            int64_t pad_rows, int64_t pad_cols, int64_t key);
// sum of squares over the (global-)upper part (or everything) of a local block; accumulates into out[0]
capital_status_t sumsq_block(capital_ctx* ctx, cudaStream_t st, int64_t rows, int64_t cols, const double* a, int64_t ld,
                             int upper_mode, int x, int y, int d, double* out);
capital_status_t sub_identity_local(capital_ctx* ctx, cudaStream_t st, int64_t n, double* a, int64_t ld);

// ---- leaf.cu ----------------------------------------------------------------------------------
// potrf('U') + trtri('U','N') of one nb x nb block (nb <= LEAF_MAX) in shared memory.
constexpr int LEAF_MAX = 64;
constexpr int BASECASE_MAX = 512;  // largest block handled by the one-launch cluster kernel (multiple of 64)
capital_status_t basecase_cholinv(capital_ctx* ctx, cudaStream_t st, int nb, double* W, int64_t ldw, double* R, int64_t ldr,
                                  double* Ri, int64_t ldri, double* RiT, int64_t ldrit);
capital_status_t leaf_cholinv(capital_ctx* ctx, cudaStream_t st, int nb, const double* W, int64_t ldw, double* R, int64_t ldr,
                              double* Ri, int64_t ldri, double* RiT, int64_t ldrit);

// ---- cholinv.cu -------------------------------------------------------------------------------
// local (single-GPU) recursive CholInv on dense n x n blocks; W is destroyed (Schur complements).
// Optional callbacks of the top-level call (host-pointer path): `need_cols` makes `st` wait until columns [0, col_end)
// of W have arrived from the host; `left_done` fires after each left child on the right spine (depth <= 3), when columns
// [0, col_end) of R are final
// and Rinv are final.
struct CholinvHooks {
  void* user;
  capital_status_t (*need_cols)(void* user, cudaStream_t st, int64_t col_end);
  capital_status_t (*left_done)(void* user, cudaStream_t st, int64_t col_end, int depth);
  // optional (host-pointer callers).  `cols_waited`: how many leading columns the chain already waited for -- while it is short of a
  // node's extent, the node's R12 product is issued in column chunks, each behind the arrival of its own columns only.
  // `right_done`: the top-level right child has returned, all of R is final.  `inv_cols`: the top-level inverse block is issued in
  // column chunks; columns [0, col_end) of Rinv are final.
  int64_t (*cols_waited)(void* user);
  capital_status_t (*right_done)(void* user, cudaStream_t st);
  capital_status_t (*inv_cols)(void* user, cudaStream_t st, int64_t col_end);
  // optional, exclusive with left_done / right_done / inv_cols: rows [r0, r1) x columns [c0, c1) (clipped to the upper triangle) of
  // R (which = 0) or Rinv (which = 1) are final on stream `st`.  Fired for the off-diagonal block of every node above depth
  // ctx->zc_depth and for the diagonal triangle of the nodes at that depth (or leaves above it): together they tile the triangle.
  capital_status_t (*block_done)(void* user, cudaStream_t st, int which, int64_t r0, int64_t r1, int64_t c0, int64_t c1);
};
// allow_side = false keeps everything on `st` (the distributed base case runs on the critical chain and must not queue behind
// the deferred stream's GEMMs).
capital_status_t cholinv_local(capital_ctx* ctx, cudaStream_t st, int64_t n, double* W, int64_t ldw, double* R, int64_t ldr,
                               double* Ri, int64_t ldri, double* RiT, int64_t ldrit, bool complete_top, int64_t bc, int split,
                               const CholinvHooks* hooks = nullptr, bool allow_side = true);

static inline int64_t round_up(int64_t a, int64_t b) { return (a + b - 1) / b * b; }
// Does cholinv::invoke split a node of (global = local, single GPU) size n, or is it the reference's base case (potrf + trtri of the
// whole block, cholinv.hpp:93)?  Decides whether complete_inv == 0 skips an inverse block at all: a top-level base case always
// returns the full inverse.
static inline bool cholinv_node_splits(int64_t n, int64_t bc, int split) { return n > bc && (n >> split) >= split && (n >> split) > 0; }
static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
