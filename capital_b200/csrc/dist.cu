// Multi-GPU schedules: one process per GPU, peer memory over NVLink / NVSwitch in place of the reference's MPI (peer.cuh).
//
//  * CholInv on a c x d x d grid.  Every SUMMA of cholinv::invoke (summa.hpp:46-161) is ONE fused kernel launch per rank:
//      operands    the X block owned by (y, kb, z) and the Y block owned by (x, kb, z) for the k classes kb of layer z
//                  [util::transpose + row / column MPI_Bcast, summa.hpp:185,193] are not fetched on demand: every block of
//                  R / R^-1 / (R^-1)^T / A is DMA-pushed into its consumers' MIRROR buffers by the copy engines the moment it
//                  is final (push()), so by the time a product is issued most of its operands have been resident for a long
//                  time, and the rest travels while something else computes;
//      product     local DMMA over the k classes of this layer [cblas_dgemm / dtrmm, summa.hpp:64,143];
//      collect     the depth reduction [MPI_Allreduce over depth, summa.hpp:236] happens inside the GEMM epilogue over
//                  peer-mapped memory (gemm_tn.cu, GemmXDev): partial tiles go straight to the tile's owner layer, which stores
//                  the final tile into every replica.  No collective call, no extra pass over C.
//    The recursion keeps the two-stream shape of the single-GPU schedule (cholinv_local.cu): base cases, R12 and the leading
//    part of the trailing update form the critical CHAIN; the rest of the trailing update and T^T are DEFERRED to a second
//    stream with its own exchange buffers, flags and push stream.
//    Base case = the replicate-everything policy (cholinv/policy.h:160-224): the d^2 local blocks of the slice are pushed to every
//    slice member, each rank factors the dense block, keeps its own cyclic part (zeros below the global diagonal -- the slots the
//    reference's benchmarked NoReplication policy leaves stale at P > 1).
//  * Grids: c == d (the reference's, k split over layers), c = 1 (several k classes per product, no depth exchange) and
//    d = 1 (c replicas: output tile columns split over the layers, results stored to every replica).
//  * CholeskyQR2 1D (c == 1 rect grid): local Gram, one small all-reduce (peer_allreduce_sum), replicated potrf+trtri, local apply
//    (cacqr.hpp:5-29,172-193; cacqr/policy.h:78-85); 3D (c == d): SUMMA Gram + CholInv + SUMMA apply (cacqr.hpp:75-120,195-215).
//
// Synchronisation is by monotonically increasing 64-bit flags (peer.cuh).  Every rank runs the same program, so every rank
// counts the same logical push events; a consumer therefore knows the id of the last push destined to it without any message.
// With `dry` set the schedule is only RECORDED (tests/test_dist_protocol.py replays the traces of all ranks and checks that the
// flag protocol cannot deadlock) -- no CUDA call is made.
#include "dist.cuh"
#include "peer.cuh"
#include <math.h>
#include <stdlib.h>
#include <algorithm>

namespace {

inline int rank_of(const capital_grid_t& g, int x, int y, int z) { return y * g.c * g.d + x * g.c + z; }  // topology.h:81-83 inverted

// ---- small kernels used only by the distributed schedules ---------------------------------------------------
// gathered[(x' + d y')] = local block (s x s, ld lds) of slice rank x' + d y'  ->  dense (s d) x (s d) block, upper part
// (util::block_to_cyclic_*, util.hpp:56-133)
__global__ void blocks_to_dense_kernel(int s, int d, const double* gathered, long long lds, double* dense,
                                       long long ldd) {
  const long long b = (long long)s * d, total = b * b;
  const long long blk = lds * s;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const long long gx = idx / b, gy = idx - gx * b;  // col, row
    double v = 0.0;
    if (gy <= gx) {
      const int xo = (int)(gx % d), yo = (int)(gy % d);
      v = __ldcg(gathered + (xo + (long long)d * yo) * blk + (gx / d) * lds + (gy / d));  // L2 only: written by the slice members' DMA
    }
    dense[gx * ldd + gy] = v;
  }
}
// own cyclic part of three dense blocks at once: loc(j, i) = dense(y + d j, x + d i)   (util::cyclic_to_local, util.hpp:135-164)
__global__ void dense_to_local3_kernel(int s, int d, int x, int y, const double* d0, const double* d1,
                                       const double* d2, long long ldd, double* l0, double* l1,
                                       double* l2, long long ldl) {
  const long long total = (long long)s * s;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const long long i = idx / s, j = idx - i * s;
    const long long src = (x + (long long)d * i) * ldd + (y + (long long)d * j);
    l0[i * ldl + j] = d0[src];
    l1[i * ldl + j] = d1[src];
    l2[i * ldl + j] = d2[src];
  }
}

// Second half of the depth reduction (summa.hpp:236): C = beta * C + sum over the layers' partial products, added in LAYER ORDER on
// every layer (identical bits in every replica).  One streaming pass: every partial is read once, C is read (beta != 0) and written
// once.  upper_only: entries with row > col0 + col are left alone (the producing GEMM only computed the upper tiles).
struct PartialSrc { const double* p[GEMM_XPEERS_MAX + 1]; int n; };
__device__ __forceinline__ double2 ld_sys(const double* p) {
  double2 v;
  asm volatile("ld.relaxed.sys.global.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p) : "memory");
  return v;
}
__global__ void __launch_bounds__(256) reduce_partials_kernel(long long rows, long long cols, PartialSrc src, long long ldp, double beta,
                                                              double* C, long long ldc, int upper_only, long long col0) {
  const long long r2 = (rows + 1) / 2;  // row pairs: every buffer is 16-byte aligned with an even leading dimension
  for (long long c = blockIdx.y; c < cols; c += gridDim.y) {
    const long long rmax = upper_only ? min(rows, c + col0 + 1) : rows;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < r2; i += (long long)gridDim.x * blockDim.x) {
      const long long r = 2 * i;
      if (r >= rmax) break;
      // system-scope loads: all but one of the partials were stored by OTHER GPUs' epilogues over NVLink
      double2 v = ld_sys(src.p[0] + c * ldp + r);
      for (int l = 1; l < src.n; l++) {
        const double2 w = ld_sys(src.p[l] + c * ldp + r);
        v.x += w.x; v.y += w.y;
      }
      double* cc = C + c * ldc + r;
      if (r + 1 < rmax && ((ldc | (long long)(((uintptr_t)C) >> 3)) & 1) == 0) {
        double2* c2 = reinterpret_cast<double2*>(cc);
        if (beta != 0.0) { const double2 o = *c2; v.x += beta * o.x; v.y += beta * o.y; }
        *c2 = v;
      } else {
        cc[0] = beta != 0.0 ? beta * cc[0] + v.x : v.x;
        if (r + 1 < rmax) cc[1] = beta != 0.0 ? beta * cc[1] + v.y : v.y;
      }
    }
  }
}

// One system-scope load from every partner buffer the preceding GEMM stored into, issued between that GEMM and the flag that
// announces it.  A read over NVLink cannot pass the posted writes of the same source to the same destination, so when it returns
// the epilogue's remote stores have been delivered -- the flag itself travels from the stream's front end, not from the SMs, and
// must not get there first.  (Belt and braces on top of the membar.sys every storing thread executes.)
struct PeerTouch { const double* p[GEMM_XPEERS_MAX]; int n; };
__global__ void flush_posted_writes_kernel(PeerTouch t, double* sink) {
  if (threadIdx.x < t.n) {
    double v;
    asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(t.p[threadIdx.x]) : "memory");
    if (v == 1.2345678e300) sink[0] = v;  // keep the load alive
  }
  __threadfence_system();
}

inline int grid_for(const capital_ctx* ctx, long long total) {
  long long b = (total + 255) / 256;
  const long long cap = (long long)ctx->num_sms * 8;
  return (int)(b > cap ? cap : (b < 1 ? 1 : b));
}
inline int64_t packed_ld(int64_t rows) { return round_up(rows, 2); }

// ---- the distributed machinery --------------------------------------------------------------------------------
enum { ROLE_X = 1, ROLE_Y = 2, ROLE_T = 4, ROLE_G = 8 };
// internal product flag (never reaches a kernel): this product is a trailing update A22 -= R12^T R12 -- the one product the
// experimental mixed-precision mode may run on the TF32 tensor cores (gemm_tf32.cu; grids without a depth exchange only)
constexpr int GEMM_TRAILING = 1 << 16;
enum { Q_CHAIN = 0, Q_FAR0 = 1, Q_BULK = PEER_QC };  // deferred classes Q_FAR0 + depth, depth < PEER_NFAR
enum { S_USER = 0, S_CHAIN = 1, S_FAR0 = 2, S_PUSH0 = S_FAR0 + PEER_NFAR, S_COPYIN = S_PUSH0 + PEER_Q, S_COPYOUT = S_COPYIN + 1, S_COUNT = S_COPYOUT + 1 };
constexpr int NK_MAX = GEMM_NCLS_MAX;

// A matrix that lives in the arena together with its mirror slots: xs[j] / ys[j] receive the blocks of the class-j X / Y source,
// ts the blocks of the transpose partner.  All slots share the leading dimension of `own`, so a window has the same offset in each.
struct DMat {
  double* own = nullptr;
  int64_t ld = 0, cols = 0;
  double* xs[NK_MAX] = {nullptr, nullptr};
  double* ys[NK_MAX] = {nullptr, nullptr};
  double* ts = nullptr;
  bool xy_same = false;  // every block pushed in the Y role is also pushed in the X role: one copy serves a consumer that is both
};
struct Win {
  const DMat* M;
  int64_t r0, c0;
};
struct Token {  // a logical push event: class, id, roles it was pushed in
  int q = 0;
  unsigned long long id = 0;
  int roles = 0;
};
struct Flag {
  int rank;     // whose control block
  size_t word;  // which flag
  unsigned long long v;
};
// trace of a dry run: flat int64 records of 8 values (kind, stream, a .. f).  T_READ / T_WRITE describe the arena windows the NEXT
// operation of the stream touches (byte offset from the arena base, leading dimension, rows, cols), T_MAT the slots of the layout.
enum { T_WAIT = 1, T_SIGNAL = 2, T_PRODUCT = 3, T_EVREC = 4, T_EVWAIT = 5, T_DMA = 6, T_KERNEL = 7, T_READ = 8, T_WRITE = 9, T_MAT = 10 };
constexpr int TREC = 8;

struct Dist {
  capital_ctx* ctx = nullptr;
  Peer* P = nullptr;
  capital_grid_t g{};
  int c = 1, d = 1, me = 0;
  int nk = 1;     // k classes this layer multiplies per product
  int xmode = 0;  // depth exchange mode of the fused product (GemmXDev): 0 (c == 1), 1 (k split), 2 (n split, d == 1)
  int srcX[NK_MAX], srcY[NK_MAX], y_in_x[NK_MAX], tpartner = 0;
  int cons_roles[PEER_MAX_RANKS], cons_jx[PEER_MAX_RANKS], cons_jy[PEER_MAX_RANKS];  // what rank t consumes from ME, and in which slot
  int src_roles[PEER_MAX_RANKS];                                                     // what I consume from rank s
  unsigned long long expect[PEER_MAX_RANKS][PEER_Q];  // id of the latest push of class q that rank s sends to me (program order so far)
  // dry run
  bool dry = false;
  std::vector<int64_t>* trace = nullptr;
  int dry_events = 0;
  std::vector<int> dry_evgen;
  // cholinv state
  int64_t L = 0, ld = 0, bc_local = 0;
  int split = 1;
  DMat W, R, Ri, RiT;
  // partial products of the k-split exchange, per stream class: my own partial, and two alternating sets of receive buffers (one
  // per other layer) that the partners' GEMM epilogues store into
  double* pown[PEER_QC][3] = {};
  double* precv[PEER_QC][3] = {};
  int nsets[PEER_QC] = {};            // rotating buffer sets of the class (3 on the chain: chunked products are software-pipelined)
  size_t precv_stride[PEER_QC] = {};  // doubles per partial buffer of the class
  double* gath[2] = {nullptr, nullptr};
  int64_t gath_blk = 0;
  int64_t bc_max = 0;  // widest base-case window of the recursion: what the gather buffers and the dense base-case block hold
  unsigned long long bc_count = 0;
  double *bcW = nullptr, *bcR = nullptr, *bcRi = nullptr, *bcRiT = nullptr;
  bool two_stream = true;
  int64_t far_min = 1024, side_min = 512;
  int64_t chunk_min = 4096;  // R12 / Rinv12 blocks at least this wide are produced and pushed in `chunks` column chunks [env CAPITAL_DIST_CHUNK_MIN]
  int chunks = 4;            // [env CAPITAL_DIST_CHUNKS]
  bool bulk_class = true;    // node-entry pushes of A12 travel on their own push stream [env CAPITAL_DIST_BULK]
  bool flush_reads = true;   // read back from the partners between a storing GEMM and its flag [env CAPITAL_DIST_FLUSH_READS]
  bool pipeline = false;     // chunked products issue chunk j + 1 before adding up chunk j (hides the layers' skew) [env CAPITAL_DIST_PIPELINE];
                             // protocol-checked, but off until it has a clean multi-GPU soak (profiles/r02c_coherence_bug_notes.md)
  // host-pointer callers: A arrives by column chunks on the copy-in stream; finished column ranges are packed and copied out while
  // the rest of the factorization runs
  std::vector<std::pair<int64_t, int>> in_chunks;  // (col_end, event)
  int64_t waited_cols[S_COUNT];
  bool stream_out = false, rinv_streams = false;
  double *dR = nullptr, *dRinv = nullptr, *hR = nullptr, *hRinv = nullptr;
  int64_t cols_out = 0, rinv_cols_out = 0;
  int e_out = -1;

  // ---------------------------------------------------------------------------------------------------------
  cudaStream_t strm(int sid) const {
    if (dry) return (cudaStream_t)(uintptr_t)(sid + 1);
    switch (sid) {
      case S_USER: return ctx->stream;
      case S_CHAIN: return ctx->hi;
      case S_FAR0: return ctx->side;
      case S_FAR0 + 1: return ctx->side_deep[0];
      case S_FAR0 + 2: return ctx->side_deep[1];
      case S_COPYIN: return ctx->copy_in;
      case S_COPYOUT: return ctx->copy_out;
      default: return P->push[sid - S_PUSH0];
    }
  }
  int cstream(int q) const { return q == Q_CHAIN ? S_CHAIN : S_FAR0 + (q - Q_FAR0); }
  void rec(int kind, int sid, int64_t a = 0, int64_t b = 0, int64_t c_ = 0, int64_t d_ = 0, int64_t e_ = 0, int64_t f_ = 0) {
    const int64_t r[TREC] = {kind, sid, a, b, c_, d_, e_, f_};
    trace->insert(trace->end(), r, r + TREC);
  }
  // dry runs only: the next operation of stream `sid` reads / writes this window of rank `rank`'s arena (`group` != 0: one of the
  // cooperating writers of a fused product, which own disjoint tiles of the window)
  void rd(int sid, const double* p, int64_t ldp, int64_t rows, int64_t cols) {
    if (dry && p) rec(T_READ, sid, me, (const char*)p - P->arena, ldp, rows, cols);
  }
  void wr(int sid, int rank, const double* p, int64_t ldp, int64_t rows, int64_t cols, int64_t group = 0) {
    if (dry && p) rec(T_WRITE, sid, rank, (const char*)p - P->arena, ldp, rows, cols, group);
  }
  // dry runs only: the product of stream `sid` first copies each operand that starts on an odd row into the context's alignment
  // scratch (gemm_tn.cu, launch), recorded as a write to scratch slot `gemm_align_slot` at the negative offset -1 - slot
  void wr_align_scratch(int sid, const GemmOperands& ops, int64_t m, int64_t n, int64_t k) {
    if (!dry) return;
    for (int j = 0; j < ops.ncls; j++) {
      const bool same = ops.A[j] == ops.B[j] && ops.lda == ops.ldb && m == n;  // B then reuses A's copy
      if ((uintptr_t)ops.A[j] & 15) rec(T_WRITE, sid, me, -1 - gemm_align_slot(sid, 0, j), 0, k, m);
      if (((uintptr_t)ops.B[j] & 15) && !same) rec(T_WRITE, sid, me, -1 - gemm_align_slot(sid, 1, j), 0, k, n);
    }
  }
  capital_status_t wait_flags(int sid, const std::vector<Flag>& fl) {
    FlagList L_;
    for (size_t i = 0; i < fl.size(); i++) {
      if (fl[i].v == 0) continue;
      if (dry) { rec(T_WAIT, sid, (int64_t)fl[i].word, (int64_t)fl[i].v); continue; }
      L_.add(P->ctrl + fl[i].word, fl[i].v);
      if (L_.n == 24) { CAP_TRY(peer_wait(ctx, strm(sid), L_)); L_.n = 0; }
    }
    if (!dry) CAP_TRY(peer_wait(ctx, strm(sid), L_));
    return CAPITAL_OK;
  }
  capital_status_t signal_flags(int sid, const std::vector<Flag>& fl) {
    FlagList L_;
    for (size_t i = 0; i < fl.size(); i++) {
      if (dry) { rec(T_SIGNAL, sid, fl[i].rank, (int64_t)fl[i].word, (int64_t)fl[i].v); continue; }
      L_.add(ctrl_ptr(P, fl[i].rank, fl[i].word), fl[i].v);
      if (L_.n == 24) { CAP_TRY(peer_signal(ctx, strm(sid), L_)); L_.n = 0; }
    }
    if (!dry) CAP_TRY(peer_signal(ctx, strm(sid), L_));
    return CAPITAL_OK;
  }
  capital_status_t ev_record(int sid, int* ev) {
    if (dry) {
      *ev = dry_events++;
      dry_evgen.push_back(1);
      rec(T_EVREC, sid, *ev);
      return CAPITAL_OK;
    }
    if (ctx->comm_used == ctx->comm_pool.size()) {
      cudaEvent_t e;
      CAP_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      ctx->comm_pool.push_back(e);
    }
    *ev = (int)ctx->comm_used++;
    CAP_CUDA(cudaEventRecord(ctx->comm_pool[*ev], strm(sid)));
    return CAPITAL_OK;
  }
  capital_status_t ev_wait(int sid, int ev) {
    if (ev < 0) return CAPITAL_OK;
    if (dry) { rec(T_EVWAIT, sid, ev); return CAPITAL_OK; }
    CAP_CUDA(cudaStreamWaitEvent(strm(sid), ctx->comm_pool[ev], 0));
    return CAPITAL_OK;
  }
  // rows x cols window (column-major) from my memory into rank `dst_rank`'s arena, by the copy engines
  capital_status_t dma2d(int sid, int dst_rank, double* dst, int64_t ldd, const double* src, int64_t lds, int64_t rows, int64_t cols) {
    if (dry) {
      rd(sid, src, lds, rows, cols);
      wr(sid, dst_rank, dst, ldd, rows, cols);
      rec(T_DMA, sid, dst_rank);
      return CAPITAL_OK;
    }
    const int tli = ctx->tl_begin(strm(sid), 7, (double)rows, (double)cols, (double)dst_rank);
    // in pieces of at most 512 MiB (whole columns): a single peer copy of exactly 2 GiB -- the L x L operand of the n = 32768
    // validator on the 2 x 2 x 2 grid -- was observed to let the flag that follows it overtake the tail of the data
    // (profiles/r02c_coherence_bug_notes.md); smaller pieces also let several copy engines work on one push
    const int64_t cpp = std::max<int64_t>(1, ((int64_t)512 << 20) / (rows * 8));
    for (int64_t c0 = 0; c0 < cols; c0 += cpp) {
      const int64_t nc = std::min(cpp, cols - c0);
      double* dp = dst + c0 * ldd;
      const double* sp = src + c0 * lds;
      if (rows == lds && rows == ldd) CAP_CUDA(cudaMemcpyAsync(dp, sp, (size_t)rows * nc * 8, cudaMemcpyDefault, strm(sid)));
      else CAP_CUDA(cudaMemcpy2DAsync(dp, (size_t)ldd * 8, sp, (size_t)lds * 8, (size_t)rows * 8, (size_t)nc, cudaMemcpyDefault, strm(sid)));
    }
    ctx->tl_end(strm(sid), tli);
    return CAPITAL_OK;
  }
};

// run a device-side helper of another translation unit on stream `sid` (recorded as an opaque kernel in a dry run)
#define DO(D, sid, call)                                 \
  do {                                                   \
    if ((D).dry) (D).rec(T_KERNEL, (sid));               \
    else CAP_TRY(call);                                  \
  } while (0)
#define DO_CUDA(D, sid, call)                            \
  do {                                                   \
    capital_ctx* ctx = (D).ctx;                          \
    if ((D).dry) (D).rec(T_KERNEL, (sid));               \
    else CAP_CUDA(call);                                 \
  } while (0)

// ---- topology tables ----------------------------------------------------------------------------------------------
// k classes of layer z: kb_j = z + j c for c <= d (the reference has c == d: one class per layer, summa.hpp:185-193); a single
// class 0 when d == 1.
inline int nclasses(const capital_grid_t& g) { return g.d == 1 ? 1 : g.d / g.c; }
inline int kclass(const capital_grid_t& g, int z, int j) { return g.d == 1 ? 0 : z + j * g.c; }
inline void coords(const capital_grid_t& g, int r, int* x, int* y, int* z) { *z = r % g.c; *y = r / (g.d * g.c); *x = (r % (g.d * g.c)) / g.c; }

capital_status_t dist_setup(Dist& D, capital_ctx* ctx, bool dry) {
  if (!ctx->peer && ctx->grid.size == 1) {  // degenerate grid: the same code runs with an empty peer table
    Peer* P1 = new Peer();
    P1->size = 1; P1->rank = 0;
    ctx->peer = P1;
  }
  D.ctx = ctx; D.P = peer_of(ctx); D.g = ctx->grid; D.dry = dry;
  const capital_grid_t& g = D.g;
  D.c = g.c; D.d = g.d; D.me = g.rank;
  const bool ok = (g.d == 1) || (g.c >= 1 && g.d % g.c == 0 && g.d / g.c <= NK_MAX);
  if (!ok || g.c - 1 > GEMM_XPEERS_MAX || g.size > PEER_MAX_RANKS) {
    ctx->set_error("distributed schedules need a c x d x d grid with c | d (d / c <= 2) or d == 1, c <= 4, at most 16 ranks");
    return CAPITAL_ERR_UNSUPPORTED;
  }
  D.nk = nclasses(g);
  D.xmode = g.c == 1 ? 0 : (g.d == 1 ? 2 : 1);
  for (int j = 0; j < D.nk; j++) {
    D.srcX[j] = rank_of(g, g.y, kclass(g, g.z, j), g.z);  // owner of X rows = kb, cols = y
    D.srcY[j] = rank_of(g, g.x, kclass(g, g.z, j), g.z);  // owner of Y rows = kb, cols = x
  }
  for (int j = 0; j < D.nk; j++) {
    D.y_in_x[j] = -1;
    for (int jj = 0; jj < D.nk; jj++) if (D.srcX[jj] == D.srcY[j]) D.y_in_x[j] = jj;
  }
  D.tpartner = rank_of(g, g.y, g.x, g.z);
  for (int t = 0; t < g.size; t++) {
    int tx, ty, tz;
    coords(g, t, &tx, &ty, &tz);
    D.cons_roles[t] = 0; D.cons_jx[t] = D.cons_jy[t] = -1; D.src_roles[t] = 0;
    if (t == D.me) continue;
    for (int j = 0; j < D.nk; j++) {
      if (rank_of(g, ty, kclass(g, tz, j), tz) == D.me) { D.cons_roles[t] |= ROLE_X; D.cons_jx[t] = j; }
      if (rank_of(g, tx, kclass(g, tz, j), tz) == D.me) { D.cons_roles[t] |= ROLE_Y; D.cons_jy[t] = j; }
      if (D.srcX[j] == t) D.src_roles[t] |= ROLE_X;
      if (D.srcY[j] == t) D.src_roles[t] |= ROLE_Y;
    }
    if (rank_of(g, ty, tx, tz) == D.me) D.cons_roles[t] |= ROLE_T;  // the transpose partnership is symmetric
    if (D.tpartner == t) D.src_roles[t] |= ROLE_T;
    if (tz == g.z && g.d > 1) { D.cons_roles[t] |= ROLE_G; D.src_roles[t] |= ROLE_G; }  // base-case gather: every slice member
  }
  memset(D.expect, 0, sizeof(D.expect));
  for (int i = 0; i < S_COUNT; i++) D.waited_cols[i] = 0;
  if (const char* e = getenv("CAPITAL_DIST_TWO_STREAM")) D.two_stream = atoi(e) != 0;
  if (const char* e = getenv("CAPITAL_DIST_FAR_MIN")) D.far_min = atoll(e);
  if (const char* e = getenv("CAPITAL_DIST_SIDE_MIN")) D.side_min = atoll(e);
  if (const char* e = getenv("CAPITAL_DIST_CHUNK_MIN")) D.chunk_min = atoll(e);
  if (const char* e = getenv("CAPITAL_DIST_CHUNKS")) D.chunks = atoi(e);
  if (const char* e = getenv("CAPITAL_DIST_BULK")) D.bulk_class = atoi(e) != 0;
  if (const char* e = getenv("CAPITAL_DIST_PIPELINE")) D.pipeline = atoi(e) != 0;
  if (const char* e = getenv("CAPITAL_DIST_FLUSH_READS")) D.flush_reads = atoi(e) != 0;
  if (ctx->no_overlap) D.two_stream = false;
  return CAPITAL_OK;
}

// ---- arena layout ---------------------------------------------------------------------------------------------------
struct Layout {
  char* base;
  size_t off = 0;
  explicit Layout(char* b) : base(b) {}
  double* take(size_t doubles) {
    const size_t o = off;
    off = (size_t)round_up((int64_t)(off + doubles * 8), 1024);
    return (double*)(base + o);
  }
};
// a matrix with the mirror slots of the given roles (every rank allocates every slot: symmetric offsets)
void layout_mat(Layout& lay, const Dist& D, DMat& M, int64_t ld, int64_t cols, int roles, bool xy_same) {
  M.ld = ld; M.cols = cols; M.xy_same = xy_same;
  const size_t n = (size_t)ld * cols;
  M.own = lay.take(n);
  const bool peers = D.g.size > 1 && D.d > 1;  // with d == 1 every operand is local
  for (int j = 0; j < NK_MAX; j++) {
    M.xs[j] = (peers && (roles & ROLE_X) && j < D.nk) ? lay.take(n) : nullptr;
    M.ys[j] = (peers && (roles & ROLE_Y) && j < D.nk) ? lay.take(n) : nullptr;
  }
  M.ts = (peers && (roles & ROLE_T)) ? lay.take(n) : nullptr;
  if (D.dry && D.trace) {
    const double* slots[2 * NK_MAX + 2] = {M.own, M.xs[0], M.xs[1], M.ys[0], M.ys[1], M.ts};
    for (const double* p : slots)
      if (p) const_cast<Dist&>(D).rec(T_MAT, 0, (const char*)p - D.P->arena, ld, cols);
  }
}

// partial-product buffers of the k-split exchange of one stream class, for products of up to `elems` output elements
void layout_exchange(Layout& lay, Dist& D, int q, int64_t m, int64_t n) {
  D.precv_stride[q] = 0;
  D.nsets[q] = 0;
  if (D.xmode != 1) return;
  D.nsets[q] = q == Q_CHAIN ? 3 : 2;
  D.precv_stride[q] = (size_t)round_up((int64_t)((size_t)packed_ld(m) * n), 128);
  for (int b = 0; b < D.nsets[q]; b++) {
    D.pown[q][b] = lay.take(D.precv_stride[q]);
    D.precv[q][b] = lay.take(D.precv_stride[q] * (size_t)(D.c - 1));
  }
}

// ---- push: a finished block goes to everybody who will read it ----------------------------------------------------------
// Logical event of class q (counted identically on every rank).  As a SOURCE: after the work enqueued so far on `after_sid`, DMA the
// window into the mirror slot of every rank that consumes from me in one of `roles`, then raise that rank's flag to the event id.
// As a CONSUMER: remember the id for every source that sends me this block.
capital_status_t push(Dist& D, int q, int after_sid, const DMat& M, int64_t r0, int64_t c0, int64_t rows, int64_t cols, int roles,
                      Token* tok, double* gather_slot = nullptr, int64_t gather_ld = 0) {
  Peer* P = D.P;
  const unsigned long long id = ++P->push_id[q];
  if (tok) { tok->q = q; tok->id = id; tok->roles = roles; }
  for (int s = 0; s < D.g.size; s++)
    if (roles & D.src_roles[s]) D.expect[s][q] = id;
  const int psid = S_PUSH0 + q;
  const double* src = M.own + r0 + c0 * M.ld;
  const size_t woff = (size_t)(r0 + c0 * M.ld);
  std::vector<Flag> fl;
  bool any = false;
  for (int t = 0; t < D.g.size; t++) {
    const int r = roles & D.cons_roles[t];
    if (!r) continue;
    if (!any) {
      int ev;
      CAP_TRY(D.ev_record(after_sid, &ev));
      CAP_TRY(D.ev_wait(psid, ev));
      any = true;
    }
    if (r & ROLE_G) CAP_TRY(D.dma2d(psid, t, peer_ptr(P, t, gather_slot), gather_ld, gather_slot, gather_ld, rows, cols));
    if (r & ROLE_X) CAP_TRY(D.dma2d(psid, t, peer_ptr(P, t, M.xs[D.cons_jx[t]]) + woff, M.ld, src, M.ld, rows, cols));
    if ((r & ROLE_Y) && !((r & ROLE_X) && M.xy_same)) CAP_TRY(D.dma2d(psid, t, peer_ptr(P, t, M.ys[D.cons_jy[t]]) + woff, M.ld, src, M.ld, rows, cols));
    if (r & ROLE_T) CAP_TRY(D.dma2d(psid, t, peer_ptr(P, t, M.ts) + woff, M.ld, src, M.ld, rows, cols));
    fl.push_back({t, CTRL_PUSH + (size_t)D.me * PEER_Q + q, id});
  }
  if (any) CAP_TRY(D.signal_flags(psid, fl));
  return CAPITAL_OK;
}

// flags stream `sid` has to see before it may read what source `s` pushed: everything of the chain class so far, plus the given
// deferred / bulk tokens when they were destined to me
inline void add_waits(const Dist& D, std::vector<Flag>& w, int s, const Token* t1, const Token* t2 = nullptr) {
  if (s == D.me) return;
  if (D.expect[s][Q_CHAIN]) w.push_back({D.me, CTRL_PUSH + (size_t)s * PEER_Q + Q_CHAIN, D.expect[s][Q_CHAIN]});
  const Token* ts[2] = {t1, t2};
  for (const Token* t : ts)
    if (t && t->id && t->q != Q_CHAIN && (t->roles & D.src_roles[s])) w.push_back({D.me, CTRL_PUSH + (size_t)s * PEER_Q + t->q, t->id});
}

// One distributed product  C <- beta*C + alpha * X^T Y  on stream class q (all matrices are windows of cyclically distributed
// globals; local windows: X: k x m, Y: k x n, C: m x n).  The blocks actually multiplied are the ones owned by the class sources;
// the result is complete in EVERY replica when the call's work has drained from the class stream.  `noff`: column position of the
// window inside the full operand (column-chunked products keep the triangular k ranges and the upper mask right).
//
// Two halves.  product_issue: wait for the operands, run the GEMM (storing this layer's partial into every layer's buffers when the
// contraction is split over the layers), tell the partners.  product_finish: wait for the partners, add the partials up.  Chunked
// products issue chunk j + 1 before finishing chunk j, so the (few-percent) skew between the two layers' GEMMs hides behind a GEMM.
struct PendingProduct {
  bool active = false;
  int q = 0;
  unsigned long long seq = 0;
  int64_t m = 0, n = 0, ldp = 0, ldc = 0;
  double beta = 0.0;
  double* Cown = nullptr;
  int upper = 0, noff = 0;
  PartialSrc src{};
};
inline std::vector<Flag> partner_flags(const Dist& D, size_t base, int q, unsigned long long v, bool mine) {
  std::vector<Flag> f;
  for (int l = 0; l < D.c; l++) {
    if (l == D.g.z) continue;
    const int partner = rank_of(D.g, D.g.x, D.g.y, l);
    if (mine) f.push_back({partner, base + (size_t)D.me * PEER_Q + q, v});   // my flag in the partner's block
    else f.push_back({D.me, base + (size_t)partner * PEER_Q + q, v});         // the partner's flag in mine
  }
  return f;
}
capital_status_t flush_posted_writes(Dist& D, int sid, const GemmXDev& x) {
  capital_ctx* ctx = D.ctx;
  if (D.dry || !D.flush_reads) return CAPITAL_OK;
  PeerTouch t{};
  for (int i = 0; i < x.c - 1 && i < GEMM_XPEERS_MAX; i++) t.p[t.n++] = x.Cpeer[i];
  flush_posted_writes_kernel<<<1, 32, 0, D.strm(sid)>>>(t, ctx->d_scalars + 15);
  ctx->counters.kernel_launches++;
  CAP_CUDA(cudaGetLastError());
  return CAPITAL_OK;
}
capital_status_t product_issue(Dist& D, int q, int64_t m, int64_t n, int64_t k, double alpha, Win X, Win Y, double beta, Win C, int flags,
                               const Token* farX, const Token* farY, int noff, PendingProduct* pd) {
  capital_ctx* ctx = D.ctx;
  Peer* P = D.P;
  const int sid = D.cstream(q);
  const bool trailing = flags & GEMM_TRAILING;
  flags &= ~GEMM_TRAILING;
  pd->active = false;
  if (m <= 0 || n <= 0 || k <= 0) return CAPITAL_OK;
  GemmOperands ops;
  ops.ncls = D.nk; ops.lda = X.M->ld; ops.ldb = Y.M->ld;
  std::vector<Flag> w;
  for (int j = 0; j < D.nk; j++) {
    const int sx = D.srcX[j], sy = D.srcY[j];
    const double* xb = sx == D.me ? X.M->own : X.M->xs[j];
    const double* yb = sy == D.me ? Y.M->own : ((Y.M->xy_same && D.y_in_x[j] >= 0 && Y.M->xs[D.y_in_x[j]]) ? Y.M->xs[D.y_in_x[j]] : Y.M->ys[j]);
    if (!xb || !yb) { ctx->set_error("distributed product: operand matrix has no mirror slot for its role"); return CAPITAL_ERR_INVALID; }
    ops.A[j] = xb + X.r0 + X.c0 * X.M->ld;
    ops.B[j] = yb + Y.r0 + Y.c0 * Y.M->ld;
    add_waits(D, w, sx, farX, farY);
    add_waits(D, w, sy, farX, farY);
  }
  CAP_TRY(D.wait_flags(sid, w));
  double* Cown = C.M->own + C.r0 + C.c0 * C.M->ld;
  const int64_t ldc = C.M->ld;
  if (D.xmode == 0) {
    if (D.dry) {
      for (int j = 0; j < D.nk; j++) { D.rd(sid, ops.A[j], ops.lda, k, m); D.rd(sid, ops.B[j], ops.ldb, k, n); }
      D.wr_align_scratch(sid, ops, m, n, k);
      D.wr(sid, D.me, Cown, ldc, m, n);
      D.rec(T_PRODUCT, sid, q, 0, 0);
    } else if (trailing && trailing_uses_tf32(ctx, k * D.nk)) {
      CAP_TRY(gemm_tn_tf32_x(ctx, D.strm(sid), m, n, k, alpha, ops, beta, Cown, ldc, flags, noff, ctx->trailing_mode));
    } else CAP_TRY(gemm_tn_x(ctx, D.strm(sid), m, n, k, alpha, ops, beta, Cown, ldc, flags, 0, noff, nullptr));
    return CAPITAL_OK;
  }
  // Flags of the depth handshake (CTRL_DONE): ready(p) = 2 seq - 1 ("nothing I enqueued before product p still reads its C
  // window"), done(p) = 2 seq ("my kernel has retired: everything it stored, here and in the partners' memory, is performed").
  const unsigned long long seq = ++P->prod_seq[q];
  GemmXDev x{};
  x.mode = D.xmode; x.c = D.c; x.z = D.g.z;
  if (D.xmode == 2) {
    // n split (d == 1): a layer stores final tiles into its partners' C without needing anything from them, so it must first know
    // that they are done reading it
    for (int l = 0; l < D.c; l++) {
      if (l == D.g.z) continue;
      x.Cpeer[l < D.g.z ? l : l - 1] = peer_ptr(P, rank_of(D.g, D.g.x, D.g.y, l), Cown);
    }
    CAP_TRY(D.signal_flags(sid, partner_flags(D, CTRL_DONE, q, 2 * seq - 1, true)));
    CAP_TRY(D.wait_flags(sid, partner_flags(D, CTRL_DONE, q, 2 * seq - 1, false)));
    if (D.dry) {
      D.rd(sid, ops.A[0], ops.lda, k, m); D.rd(sid, ops.B[0], ops.ldb, k, n);
      D.wr_align_scratch(sid, ops, m, n, k);
      const int64_t group = (int64_t)(seq * 8 + q + 1);
      D.wr(sid, D.me, Cown, ldc, m, n, group);
      for (int l = 0; l < D.c; l++)
        if (l != D.g.z) D.wr(sid, rank_of(D.g, D.g.x, D.g.y, l), Cown, ldc, m, n, group);
      D.rec(T_PRODUCT, sid, q, (int64_t)seq, 2);
    } else {
      CAP_TRY(gemm_tn_x(ctx, D.strm(sid), m, n, k, alpha, ops, beta, Cown, ldc, flags, 0, noff, &x));
      CAP_TRY(flush_posted_writes(D, sid, x));
    }
    CAP_TRY(D.signal_flags(sid, partner_flags(D, CTRL_DONE, q, 2 * seq, true)));
    return D.wait_flags(sid, partner_flags(D, CTRL_DONE, q, 2 * seq, false));
  }
  // k split (c == d): the GEMM stores this layer's partial product into its own buffer and, over NVLink, into the receive buffer
  // every other layer keeps for it.  The buffers rotate over D.nsets[q] sets; a set is written again only after every layer has
  // said (CTRL_RED) that it has added up the product that used it last.
  const int nsets = D.nsets[q];
  const int64_t ldp = packed_ld(m);
  const size_t stride = D.precv_stride[q];
  if ((size_t)ldp * (size_t)n > stride) {
    ctx->set_error("distributed product: exchange buffers too small for a " + std::to_string(m) + " x " + std::to_string(n) + " product");
    return CAPITAL_ERR_UNSUPPORTED;
  }
  const int set = (int)(seq % nsets);
  double* own_set = D.pown[q][set];
  double* recv_set = D.precv[q][set];
  pd->src = PartialSrc{};
  pd->src.n = D.c;
  for (int l = 0; l < D.c; l++) {
    if (l == D.g.z) { pd->src.p[l] = own_set; continue; }
    const int oi = l < D.g.z ? l : l - 1;          // index of layer l among MY others
    const int mi = D.g.z < l ? D.g.z : D.g.z - 1;  // index of my layer among layer l's others
    x.Cpeer[oi] = peer_ptr(P, rank_of(D.g, D.g.x, D.g.y, l), recv_set + (size_t)mi * stride);
    pd->src.p[l] = recv_set + (size_t)oi * stride;
  }
  if (seq > (unsigned long long)nsets) CAP_TRY(D.wait_flags(sid, partner_flags(D, CTRL_RED, q, seq - nsets, false)));
  if (D.dry) {
    for (int j = 0; j < D.nk; j++) { D.rd(sid, ops.A[j], ops.lda, k, m); D.rd(sid, ops.B[j], ops.ldb, k, n); }
    D.wr_align_scratch(sid, ops, m, n, k);
    D.wr(sid, D.me, own_set, ldp, m, n);
    for (int l = 0; l < D.c; l++)
      if (l != D.g.z) D.wr(sid, rank_of(D.g, D.g.x, D.g.y, l), recv_set + (size_t)(D.g.z < l ? D.g.z : D.g.z - 1) * stride, ldp, m, n);
    D.rec(T_PRODUCT, sid, q, (int64_t)seq, 1);
  } else {
    CAP_TRY(gemm_tn_x(ctx, D.strm(sid), m, n, k, alpha, ops, 0.0, own_set, ldp, flags, 0, noff, &x));
    CAP_TRY(flush_posted_writes(D, sid, x));
  }
  CAP_TRY(D.signal_flags(sid, partner_flags(D, CTRL_DONE, q, 2 * seq, true)));
  pd->active = true; pd->q = q; pd->seq = seq; pd->m = m; pd->n = n; pd->ldp = ldp; pd->ldc = ldc; pd->beta = beta; pd->Cown = Cown;
  pd->upper = (flags & CAPITAL_GEMM_C_UPPER) ? 1 : 0; pd->noff = noff;
  return CAPITAL_OK;
}
capital_status_t product_finish(Dist& D, PendingProduct* pd) {
  if (!pd->active) return CAPITAL_OK;
  capital_ctx* ctx = D.ctx;
  const int q = pd->q, sid = D.cstream(q);
  pd->active = false;
  CAP_TRY(D.wait_flags(sid, partner_flags(D, CTRL_DONE, q, 2 * pd->seq, false)));
  if (D.dry) {
    for (int l = 0; l < D.c; l++) D.rd(sid, pd->src.p[l], pd->ldp, pd->m, pd->n);
    D.wr(sid, D.me, pd->Cown, pd->ldc, pd->m, pd->n);
    D.rec(T_KERNEL, sid);
  } else {
    const int tli = ctx->tl_begin(D.strm(sid), 8, 4, (double)pd->m, (double)pd->n);
    const long long r2 = (pd->m + 1) / 2;
    dim3 grid((unsigned)std::min<long long>(std::max<long long>(1, (r2 + 255) / 256), 64), (unsigned)std::min<int64_t>(pd->n, 4 * (int64_t)ctx->num_sms));
    reduce_partials_kernel<<<grid, 256, 0, D.strm(sid)>>>(pd->m, pd->n, pd->src, pd->ldp, pd->beta, pd->Cown, pd->ldc, pd->upper, pd->noff);
    ctx->tl_end(D.strm(sid), tli);
    ctx->counters.kernel_launches++;
    CAP_CUDA(cudaGetLastError());
  }
  return D.signal_flags(sid, partner_flags(D, CTRL_RED, q, pd->seq, true));
}
capital_status_t product(Dist& D, int q, int64_t m, int64_t n, int64_t k, double alpha, Win X, Win Y, double beta, Win C, int flags,
                         const Token* farX = nullptr, const Token* farY = nullptr, int noff = 0) {
  PendingProduct pd;
  CAP_TRY(product_issue(D, q, m, n, k, alpha, X, Y, beta, C, flags, farX, farY, noff, &pd));
  return product_finish(D, &pd);
}

// The same product issued in `nch` column chunks of the output, each pushed to its consumers (roles != 0) as soon as it is complete:
// the transfer of chunk j hides behind the GEMM of chunk j + 1, the partners' skew of chunk j behind it too, and only the last
// chunk's handshake and travel time stay exposed.
capital_status_t product_pushed(Dist& D, int q, int64_t m, int64_t n, int64_t k, double alpha, Win X, Win Y, double beta, Win C, int flags,
                                const Token* farX, const Token* farY, int roles, Token* last, int nch) {
  if (nch < 1) nch = 1;
  const int64_t cw = round_up(ceil_div(n, nch), 128);
  PendingProduct prev;
  int64_t prev_c0 = 0, prev_nc = 0;
  auto finish_prev = [&]() -> capital_status_t {
    if (prev_nc == 0) return CAPITAL_OK;
    CAP_TRY(product_finish(D, &prev));
    if (roles) CAP_TRY(push(D, q, D.cstream(q), *C.M, C.r0, C.c0 + prev_c0, m, prev_nc, roles, last));
    prev_nc = 0;
    return CAPITAL_OK;
  };
  const bool pipelined = D.pipeline && D.xmode == 1 && D.nsets[q] >= 3;
  for (int64_t c0 = 0; c0 < n; c0 += cw) {
    const int64_t nc = std::min(cw, n - c0);
    PendingProduct cur;
    if (!pipelined) CAP_TRY(finish_prev());
    CAP_TRY(product_issue(D, q, m, nc, k, alpha, X, Win{Y.M, Y.r0, Y.c0 + c0}, beta, Win{C.M, C.r0, C.c0 + c0}, flags, farX, farY, (int)c0, &cur));
    CAP_TRY(finish_prev());
    prev = cur; prev_c0 = c0; prev_nc = nc;
  }
  return finish_prev();
}

// dst (local cols x rows block) = [rows x cols window of the transpose partner's `Src`]^T   (util::transpose, util.hpp:232-247,
// followed by the local transpose the reference defers to its BLAS flags).  The partner pushed the window in the T role.
capital_status_t transpose_dist(Dist& D, int q, const DMat& Src, int64_t r0, int64_t c0, int64_t rows, int64_t cols, const Token* tok, double* dst,
                                int64_t ldd) {
  const int sid = D.cstream(q);
  const double* src = Src.own;
  if (D.tpartner != D.me) {
    std::vector<Flag> w;
    add_waits(D, w, D.tpartner, tok);
    CAP_TRY(D.wait_flags(sid, w));
    src = Src.ts;
  }
  D.rd(sid, src + r0 + c0 * Src.ld, Src.ld, rows, cols);
  D.wr(sid, D.me, dst, ldd, cols, rows);
  DO(D, sid, transpose_block(D.ctx, D.strm(sid), rows, cols, src + r0 + c0 * Src.ld, Src.ld, dst, ldd, 1.0));
  return CAPITAL_OK;
}

// host-pointer callers: stream `sid` must not touch columns of W beyond what has arrived
capital_status_t need_cols(Dist& D, int sid, int64_t col_end) {
  if (D.in_chunks.empty() || col_end <= D.waited_cols[sid]) return CAPITAL_OK;
  for (auto& ch : D.in_chunks)
    if (ch.first >= col_end) {
      CAP_TRY(D.ev_wait(sid, ch.second));
      D.waited_cols[sid] = ch.first;
      return CAPITAL_OK;
    }
  return CAPITAL_OK;
}

// replicate-everything base case on the local window at offset `o` of size s (local); dense size b = s d
capital_status_t base_case(Dist& D, int64_t o, int64_t s, int pending) {
  capital_ctx* ctx = D.ctx;
  const capital_grid_t& g = D.g;
  const int d = D.d;
  if (s > D.bc_max) {  // dry runs too: a trace that passes here cannot write past a gather buffer into a peer's arena
    ctx->set_error("distributed base case: window of " + std::to_string(s) + " exceeds the reserved " + std::to_string(D.bc_max));
    return CAPITAL_ERR_UNSUPPORTED;
  }
  CAP_TRY(need_cols(D, S_CHAIN, o + s));
  CAP_TRY(D.ev_wait(S_CHAIN, pending));
  double* Wo = D.W.own + o * D.ld + o;
  double* Ro = D.R.own + o * D.ld + o;
  double* Rio = D.Ri.own + o * D.ld + o;
  double* RiTo = D.RiT.own + o * D.ld + o;
  if (d == 1) {
    // every layer holds the whole block: factor in place (the c replicas compute the same bits)
    D.wr(S_CHAIN, D.me, Wo, D.ld, s, s); D.wr(S_CHAIN, D.me, Ro, D.ld, s, s); D.wr(S_CHAIN, D.me, Rio, D.ld, s, s); D.wr(S_CHAIN, D.me, RiTo, D.ld, s, s);
    DO(D, S_CHAIN, cholinv_local(ctx, D.strm(S_CHAIN), s, Wo, D.ld, Ro, D.ld, Rio, D.ld, RiTo, D.ld, true, s, 1, nullptr, false));
    return CAPITAL_OK;
  }
  const int64_t b = s * d, ldb = round_up(b, 16), lds = packed_ld(s);
  // gather (policy.h:176): my block goes into slot x + d y of every slice member's gather buffer (two buffers: a rank can be at most
  // one base case ahead of a slice member, because it needs that member's block for every base case)
  double* gbuf = D.gath[D.bc_count & 1];
  D.bc_count++;
  double* myslot = gbuf + (size_t)(g.x + d * g.y) * lds * s;
  D.rd(S_CHAIN, Wo, D.ld, s, s);
  D.wr(S_CHAIN, D.me, myslot, lds, s, s);
  DO(D, S_CHAIN, copy_block(ctx, D.strm(S_CHAIN), s, s, Wo, D.ld, myslot, lds));
  Token tg;
  CAP_TRY(push(D, Q_CHAIN, S_CHAIN, D.W, o, o, s, s, ROLE_G, &tg, myslot, lds));
  std::vector<Flag> w;
  for (int t = 0; t < g.size; t++)
    if (D.src_roles[t] & ROLE_G) add_waits(D, w, t, nullptr);
  CAP_TRY(D.wait_flags(S_CHAIN, w));
  if (!D.dry) {
    cudaStream_t st = D.strm(S_CHAIN);
    blocks_to_dense_kernel<<<grid_for(ctx, b * b), 256, 0, st>>>((int)s, d, gbuf, lds, D.bcW, ldb);
    ctx->counters.kernel_launches++;
    CAP_CUDA(cudaGetLastError());
    CAP_TRY(zero_band(ctx, st, b, D.bcRi, ldb));
    CAP_TRY(zero_band(ctx, st, b, D.bcRiT, ldb));
    CAP_TRY(cholinv_local(ctx, st, b, D.bcW, ldb, D.bcR, ldb, D.bcRi, ldb, D.bcRiT, ldb, true, b, 1, nullptr, false));  // potrf + trtri, policy.h:199-201
    dense_to_local3_kernel<<<grid_for(ctx, s * s), 256, 0, st>>>((int)s, d, g.x, g.y, D.bcR, D.bcRi, D.bcRiT, ldb, Ro, Rio, RiTo, D.ld);
    ctx->counters.kernel_launches++;
    CAP_CUDA(cudaGetLastError());
  } else {
    D.rd(S_CHAIN, gbuf, (int64_t)lds * s * d * d, (int64_t)lds * s * d * d, 1);
    D.wr(S_CHAIN, D.me, Ro, D.ld, s, s); D.wr(S_CHAIN, D.me, Rio, D.ld, s, s); D.wr(S_CHAIN, D.me, RiTo, D.ld, s, s);
    D.rec(T_KERNEL, S_CHAIN);
  }
  // the inverse's diagonal block is an operand of the products above this node (X: R12 = Rinv11^T A12; Y: Rinv12 = -T Rinv22),
  // its transpose of T^T = R12^T Rinv11^T
  CAP_TRY(push(D, Q_CHAIN, S_CHAIN, D.Ri, o, o, s, s, ROLE_X | ROLE_Y, nullptr));
  CAP_TRY(push(D, Q_CHAIN, S_CHAIN, D.RiT, o, o, s, s, ROLE_Y, nullptr));
  return CAPITAL_OK;
}

// local columns [cols_out, col_end) of R are final (of Rinv too left of the top split, and up to the next split when the top-level
// inverse block is skipped): pack that contiguous range of the packed triangle and start its D2H on the copy-out stream
capital_status_t dist_left_done(Dist& D, int64_t col_end, int depth) {
  capital_ctx* ctx = D.ctx;
  const int64_t c0 = D.cols_out;
  if (col_end <= c0) return CAPITAL_OK;
  const bool rinv_too = depth == 0 || (depth == 1 && D.rinv_streams && D.rinv_cols_out == c0);
  const size_t off = (size_t)c0 * (c0 + 1) / 2, cnt = (size_t)col_end * (col_end + 1) / 2 - off;
  DO(D, S_CHAIN, pack_upper(ctx, D.strm(S_CHAIN), D.L, D.R.own, D.ld, D.dR, 0, c0, col_end));
  if (rinv_too) DO(D, S_CHAIN, pack_upper(ctx, D.strm(S_CHAIN), D.L, D.Ri.own, D.ld, D.dRinv, 0, c0, col_end));
  D.cols_out = col_end;
  if (rinv_too) D.rinv_cols_out = col_end;
  int e;
  CAP_TRY(D.ev_record(S_CHAIN, &e));
  CAP_TRY(D.ev_wait(S_COPYOUT, e));
  if (D.hR) { DO_CUDA(D, S_COPYOUT, cudaMemcpyAsync(D.hR + off, D.dR + off, cnt * 8, cudaMemcpyDeviceToHost, D.strm(S_COPYOUT))); ctx->counters.d2h_bytes += (int64_t)cnt * 8; }
  if (D.hRinv && rinv_too) { DO_CUDA(D, S_COPYOUT, cudaMemcpyAsync(D.hRinv + off, D.dRinv + off, cnt * 8, cudaMemcpyDeviceToHost, D.strm(S_COPYOUT))); ctx->counters.d2h_bytes += (int64_t)cnt * 8; }
  CAP_TRY(D.ev_record(S_COPYOUT, &D.e_out));
  return CAPITAL_OK;
}

inline bool node_splits(const Dist& D, int64_t s) {
  const int64_t s1 = s >> D.split;
  return !(s <= D.bc_local || s1 < D.split || s1 == 0);
}
// widest base-case window below a node of local size s.  Not bounded by bc_local alone: with split > 1 a node also stops when
// s >> split < split (up to 7 wide for split = 2, 23 for split = 3).
int64_t max_base_window(const Dist& D, int64_t s) {
  if (!node_splits(D, s)) return s;
  const int64_t s1 = s >> D.split;
  return std::max(max_base_window(D, s1), max_base_window(D, s - s1));
}
// the two gather buffers of the base case (d > 1): d^2 slots of the widest window each
void layout_gather(Layout& lay, Dist& D) {
  D.bc_max = max_base_window(D, D.L);
  D.gath_blk = 0;
  if (D.d > 1) {
    D.gath_blk = packed_ld(D.bc_max) * D.bc_max;
    for (int i = 0; i < 2; i++) D.gath[i] = lay.take((size_t)D.gath_blk * D.d * D.d);
  }
}

// cholinv::invoke (cholinv.hpp:87-165) on the local window [o, o+s).  `pending`: event after which the part of the window outside
// its leading block is final (the parent's deferred update); `pendW12`: the push of this node's A12 block issued by the parent
// right after that update.
capital_status_t invoke(Dist& D, int64_t o, int64_t s, bool complete, int pending, Token pendW12, int depth) {
  if (!node_splits(D, s)) return base_case(D, o, s, pending);
  const int64_t s1 = s >> D.split, s2 = s - s1;
  const Win W12{&D.W, o, o + s1}, W21{&D.W, o + s1, o}, W22{&D.W, o + s1, o + s1};
  const Win R12{&D.R, o, o + s1};
  const Win Ri11{&D.Ri, o, o}, Ri12{&D.Ri, o, o + s1}, Ri22{&D.Ri, o + s1, o + s1};
  const Win RiT11{&D.RiT, o, o};
  // A12 is the Y operand of the first product: when nothing deferred still updates it, it can start travelling now, while the
  // left child computes (bulk class: it must not delay the chain's small pushes)
  Token tW12 = pendW12;
  if (pending < 0) {
    const int qb = D.bulk_class ? Q_BULK : Q_CHAIN;
    CAP_TRY(need_cols(D, S_PUSH0 + qb, o + s));
    CAP_TRY(push(D, qb, S_CHAIN, D.W, o, o + s1, s1, s2, ROLE_Y, &tW12));
  }
  CAP_TRY(invoke(D, o, s1, true, -1, Token{}, depth + 1));
  if (D.stream_out && depth <= 3 && o + s == D.L) CAP_TRY(dist_left_done(D, o + s1, depth));  // right spine
  // "trsm" via the inverse (cholinv.hpp:116-122): R12 = Rinv11^T A12
  CAP_TRY(need_cols(D, S_CHAIN, o + s));
  CAP_TRY(D.ev_wait(S_CHAIN, pending));
  const int nch = (D.g.size > 1 && D.d > 1 && s2 >= D.chunk_min) ? D.chunks : 1;  // big blocks travel chunk by chunk behind the GEMM
  CAP_TRY(product_pushed(D, Q_CHAIN, s1, s2, s1, 1.0, Ri11, W12, 0.0, R12, CAPITAL_GEMM_A_UPPER, nullptr, &tW12, ROLE_X | ROLE_Y, nullptr, nch));
  // trailing update (cholinv.hpp:131-134): A22 -= R12^T R12, upper tiles only.  near = what the right child's left subtree reads
  // (leading h x h block) stays on the chain, far = everything else goes to the deferred class.
  const int64_t h = node_splits(D, s2) ? (s2 >> D.split) : 0;
  // deferred class of this depth (own stream, exchange buffers, flags): a deeper node's deferred work is wanted sooner than its
  // ancestors' and would be stuck behind it on a shared FIFO stream; below depth PEER_NFAR everything stays on the chain
  const int fq = depth < PEER_NFAR ? Q_FAR0 + depth : -1;
  const bool use_side = D.two_stream && fq >= 0 && s1 >= D.side_min;
  const int fs = use_side ? D.cstream(fq) : S_CHAIN;
  int e_r12 = -1, e_far = -1, e_tt = -1;
  Token tChildW12{}, tTT{};
  if (use_side) {
    CAP_TRY(D.ev_record(S_CHAIN, &e_r12));
    CAP_TRY(D.ev_wait(fs, e_r12));
  }
  if (use_side && h > 0 && s2 >= D.far_min) {
    const Win R12b{&D.R, o, o + s1 + h};
    CAP_TRY(product(D, Q_CHAIN, h, h, s1, -1.0, R12, R12, 1.0, W22, CAPITAL_GEMM_C_UPPER | GEMM_TRAILING));
    CAP_TRY(product(D, fq, h, s2 - h, s1, -1.0, R12, R12b, 1.0, Win{&D.W, o + s1, o + s1 + h}, GEMM_TRAILING));
    // that block is the right child's A12: its Y consumers get it as soon as it is final
    CAP_TRY(push(D, fq, fs, D.W, o + s1, o + s1 + h, h, s2 - h, ROLE_Y, &tChildW12));
    CAP_TRY(product(D, fq, s2 - h, s2 - h, s1, -1.0, R12b, R12b, 1.0, Win{&D.W, o + s1 + h, o + s1 + h}, CAPITAL_GEMM_C_UPPER | GEMM_TRAILING));
    CAP_TRY(D.ev_record(fs, &e_far));
  } else {
    CAP_TRY(product(D, Q_CHAIN, s2, s2, s1, -1.0, R12, R12, 1.0, W22, CAPITAL_GEMM_C_UPPER | GEMM_TRAILING));
  }
  if (complete) {
    // inverse combine, first half (cholinv.hpp:151): T^T = R12^T Rinv11^T  (B = RiT11, lower triangular) -- nobody needs it before
    // the right child is done
    const int qt = use_side ? fq : Q_CHAIN;
    CAP_TRY(product(D, qt, s2, s1, s1, 1.0, R12, RiT11, 0.0, W21, CAPITAL_GEMM_B_LOWER));
    CAP_TRY(push(D, qt, D.cstream(qt), D.W, o + s1, o, s2, s1, ROLE_X, &tTT));
    if (use_side) CAP_TRY(D.ev_record(fs, &e_tt));
  }
  CAP_TRY(invoke(D, o + s1, s2, true, e_far, tChildW12, depth + 1));
  if (complete) {
    CAP_TRY(D.ev_wait(S_CHAIN, e_tt));
    //   Rinv12 = -(T^T)^T Rinv22  (B = Ri22, upper triangular)   (cholinv.hpp:152-155)
    Token tRi12;
    CAP_TRY(product_pushed(D, Q_CHAIN, s1, s2, s2, -1.0, W21, Ri22, 0.0, Ri12, CAPITAL_GEMM_B_UPPER, &tTT, nullptr, ROLE_X | ROLE_Y | ROLE_T, &tRi12, nch));
    CAP_TRY(transpose_dist(D, Q_CHAIN, D.Ri, o, o + s1, s1, s2, &tRi12, D.RiT.own + o * D.ld + (o + s1), D.ld));
    CAP_TRY(push(D, Q_CHAIN, S_CHAIN, D.RiT, o + s1, o, s2, s1, ROLE_Y, nullptr));
  }
  return CAPITAL_OK;
}

// every stream of the schedule starts after the caller's stream and after every rank has entered the call (nobody may still be
// reading the mirrors / receive buffers the new call is about to overwrite)
capital_status_t fork_streams(Dist& D) {
  if (D.g.size > 1) {
    if (D.dry) {
      std::vector<Flag> s, w;
      const unsigned long long e = ++D.P->bar_epoch;
      for (int r = 0; r < D.g.size; r++) {
        if (r == D.me) continue;
        s.push_back({r, CTRL_BAR + (size_t)D.me, e});
        w.push_back({D.me, CTRL_BAR + (size_t)r, e});
      }
      CAP_TRY(D.signal_flags(S_USER, s));
      CAP_TRY(D.wait_flags(S_USER, w));
    } else {
      CAP_TRY(peer_barrier(D.ctx, D.strm(S_USER)));
    }
  }
  int e;
  CAP_TRY(D.ev_record(S_USER, &e));
  for (int sid = S_CHAIN; sid < S_COUNT; sid++) {
    if (D.g.size == 1 && sid >= S_PUSH0 && sid < S_COPYIN) continue;
    CAP_TRY(D.ev_wait(sid, e));
  }
  return CAPITAL_OK;
}
capital_status_t join_streams(Dist& D) {
  for (int sid = S_CHAIN; sid < S_COUNT; sid++) {
    if (D.g.size == 1 && sid >= S_PUSH0 && sid < S_COPYIN) continue;
    int e;
    CAP_TRY(D.ev_record(sid, &e));
    CAP_TRY(D.ev_wait(S_USER, e));
  }
  return CAPITAL_OK;
}

// arena of cholinv::factor: the four work matrices with their mirror slots, receive buffers of the fused products, gather buffers
// of the base case.  Returns the number of bytes; assigns pointers relative to `base`.
size_t cholinv_layout(Dist& D, char* base) {
  Layout lay(base);
  const int64_t L = D.L, ld = D.ld;
  layout_mat(lay, D, D.W, ld, L, ROLE_X | ROLE_Y, false);   // X: T^T blocks (lower part), Y: A12 blocks (upper part)
  layout_mat(lay, D, D.R, ld, L, ROLE_X | ROLE_Y, true);
  layout_mat(lay, D, D.Ri, ld, L, ROLE_X | ROLE_Y | ROLE_T, true);
  layout_mat(lay, D, D.RiT, ld, L, ROLE_Y, false);
  // the chain multiplies blocks of every level; the deferred class of depth k only the trailing-update and T^T blocks of that depth
  int64_t sz = L;
  for (int q = 0; q < PEER_QC; q++) {
    const int64_t s1q = sz >> D.split, mx = std::max(s1q, sz - s1q) + 2;
    layout_exchange(lay, D, q, mx, mx);
    if (q >= Q_FAR0) sz = sz - s1q;  // the right child is the larger one
  }
  layout_gather(lay, D);
  return lay.off;
}

// reserve the arena for a layout; a layout the arena has not held before starts from zeros (mirror slots are only ever written
// where a block is pushed; the triangular products read whole diagonal tiles and rely on zeros elsewhere)
capital_status_t arena_prepare(capital_ctx* ctx, size_t bytes, const std::string& signature) {
  CAP_TRY(peer_arena_reserve(ctx, bytes));
  if (ctx->arena_signature != signature) {
    // (every rank changes layout in the same call.)  A peer may still be pushing blocks of the previous layout that nobody waits
    // for: all ranks drain first, then clear, and a device barrier keeps new pushes behind everybody's clear.
    CAP_TRY(peer_host_barrier(ctx));
    CAP_CUDA(cudaMemsetAsync(peer_of(ctx)->arena, 0, bytes, ctx->stream));
    ctx->arena_signature = signature;
    if (ctx->grid.size > 1) CAP_TRY(peer_barrier(ctx, ctx->stream));  // nobody writes into a peer's arena before that peer has cleared it
  }
  return CAPITAL_OK;
}

capital_status_t cholinv_run(Dist& D, const double* A_local, const capital_cholinv_args_t* args, capital_structure_t ostruct,
                             double* R_local, double* Rinv_local, size_t out_count) {
  capital_ctx* ctx = D.ctx;
  const int64_t L = D.L, ld = D.ld;
  ctx->comm_used = 0;
  D.in_chunks.clear();
  CAP_TRY(fork_streams(D));
  const bool a_dev = D.dry || cap_is_device_ptr(A_local);
  if (!D.dry) CAP_CUDA(cudaMemsetAsync(ctx->d_info, 0, sizeof(int), D.strm(S_CHAIN)));
  const bool top_splits = node_splits(D, L);
  if (args->complete_inv == 0 && top_splits) {  // the skipped top-level block of Rinv (cholinv.hpp:147) reads as zeros in the output
    const int64_t s1 = L >> D.split;
    D.wr(S_CHAIN, D.me, D.Ri.own + s1 * ld, ld, s1, L - s1);
    DO(D, S_CHAIN, zero_block(ctx, D.strm(S_CHAIN), s1, L - s1, D.Ri.own + s1 * ld, ld));
  }
  if (a_dev) {
    D.wr(S_CHAIN, D.me, D.W.own, ld, L, L);
    DO(D, S_CHAIN, copy_block(ctx, D.strm(S_CHAIN), L, L, A_local, L, D.W.own, ld));  // serialize(A -> R), cholinv.hpp:13
  } else {
    // host caller: only the (local) upper triangle is read, so only rows [0, column chunk end) travel; the recursion consumes W left
    // to right and waits chunk by chunk
    const int64_t chunk = round_up(ceil_div(L, 16), 64);
    for (int64_t c0 = 0; c0 < L; c0 += chunk) {
      const int64_t nc = (c0 + chunk <= L) ? chunk : L - c0, rows = c0 + nc;
      CAP_CUDA(cudaMemcpy2DAsync(D.W.own + c0 * ld, (size_t)ld * 8, A_local + c0 * L, (size_t)L * 8, (size_t)rows * 8, (size_t)nc,
                                 cudaMemcpyHostToDevice, D.strm(S_COPYIN)));
      ctx->counters.h2d_bytes += rows * nc * 8;
      int e;
      CAP_TRY(D.ev_record(S_COPYIN, &e));
      D.in_chunks.push_back({c0 + nc, e});
    }
  }
  D.stream_out = !D.dry && ostruct == CAPITAL_UPPERTRI_PACKED && (D.hR || D.hRinv) && L >= 2048;
  D.rinv_streams = args->complete_inv == 0 && top_splits;
  D.cols_out = D.rinv_cols_out = 0;
  D.e_out = -1;
  CAP_TRY(invoke(D, 0, L, args->complete_inv != 0, -1, Token{}, 0));
  if (D.dry) return join_streams(D);
  cudaStream_t cs = D.strm(S_CHAIN);
  const int zd = D.g.y > D.g.x ? 1 : 0;
  (void)zd;  // base cases already wrote zeros on the local-diagonal slots of ranks below the global diagonal
  if (ostruct == CAPITAL_UPPERTRI_PACKED) {
    {
      const int64_t c0 = D.cols_out;
      const size_t off = (size_t)c0 * (c0 + 1) / 2, cnt = out_count - off;
      CAP_TRY(pack_upper(ctx, cs, L, D.R.own, ld, D.dR, 0, c0, L));
      if (D.hR) { CAP_CUDA(cudaMemcpyAsync(D.hR + off, D.dR + off, cnt * 8, cudaMemcpyDeviceToHost, cs)); ctx->counters.d2h_bytes += (int64_t)cnt * 8; }
    }
    {
      const int64_t c0 = D.rinv_cols_out;
      const size_t off = (size_t)c0 * (c0 + 1) / 2, cnt = out_count - off;
      CAP_TRY(pack_upper(ctx, cs, L, D.Ri.own, ld, D.dRinv, 0, c0, L));
      if (D.hRinv) { CAP_CUDA(cudaMemcpyAsync(D.hRinv + off, D.dRinv + off, cnt * 8, cudaMemcpyDeviceToHost, cs)); ctx->counters.d2h_bytes += (int64_t)cnt * 8; }
    }
  } else {
    CAP_TRY(triu_copy(ctx, cs, L, D.R.own, ld, D.dR, L, 0));
    CAP_TRY(triu_copy(ctx, cs, L, D.Ri.own, ld, D.dRinv, L, 0));
    if (D.hR) { CAP_CUDA(cudaMemcpyAsync(D.hR, D.dR, out_count * 8, cudaMemcpyDeviceToHost, cs)); ctx->counters.d2h_bytes += (int64_t)out_count * 8; }
    if (D.hRinv) { CAP_CUDA(cudaMemcpyAsync(D.hRinv, D.dRinv, out_count * 8, cudaMemcpyDeviceToHost, cs)); ctx->counters.d2h_bytes += (int64_t)out_count * 8; }
  }
  return join_streams(D);
}

capital_status_t cholinv_shape(Dist& D, int64_t n, const capital_cholinv_args_t* args) {
  const capital_grid_t& g = D.g;
  if (n % g.d != 0) { D.ctx->set_error("distributed cholinv needs d | n"); return CAPITAL_ERR_UNSUPPORTED; }
  D.L = n / g.d; D.ld = round_up(D.L, 16); D.split = (int)args->split;
  D.bc_local = capital_cholinv_bc_dimension(D.L, g.c, g.d, args->bc_mult_dim) / g.d;
  return CAPITAL_OK;
}

capital_status_t need_comm(capital_ctx* ctx) {
  if (ctx->grid.size > 1 && !ctx->peer) {
    ctx->set_error("multi-GPU grid but capital_comm_init was not called");
    return CAPITAL_ERR_COMM;
  }
  return CAPITAL_OK;
}

// the work buffers of the dense base-case block (local, not peer-visible)
capital_status_t bc_workspace(Dist& D) {
  capital_ctx* ctx = D.ctx;
  if (D.d == 1) return CAPITAL_OK;
  const int64_t b = D.bc_max * D.d, ldb = round_up(b, 16);
  const size_t bytes = (size_t)ldb * b * 8;
  void* old = ctx->pool.count("bc_Ri") ? ctx->pool["bc_Ri"].p : nullptr;
  CAP_TRY(ctx->workspace("bc_W", bytes, (void**)&D.bcW));
  CAP_TRY(ctx->workspace("bc_R", bytes, (void**)&D.bcR));
  CAP_TRY(ctx->workspace("bc_Ri", bytes, (void**)&D.bcRi));
  CAP_TRY(ctx->workspace("bc_RiT", bytes, (void**)&D.bcRiT));
  // the factor kernels rely on zeros outside what they write; the dense size (leading dimension) may differ from the last call's
  (void)old;
  CAP_CUDA(cudaMemsetAsync(D.bcR, 0, bytes, ctx->stream));
  CAP_CUDA(cudaMemsetAsync(D.bcRi, 0, bytes, ctx->stream));
  CAP_CUDA(cudaMemsetAsync(D.bcRiT, 0, bytes, ctx->stream));
  return CAPITAL_OK;
}

}  // namespace

void dist_destroy(capital_ctx* ctx) {
  peer_destroy(ctx);
  for (cudaEvent_t e : ctx->comm_pool) cudaEventDestroy(e);
  ctx->comm_pool.clear();
}
capital_status_t dist_release_peer_maps(capital_ctx* ctx) {
  ctx->arena_signature.clear();
  return peer_arena_release(ctx);
}

capital_status_t dist_cholinv_factor(capital_ctx* ctx, const double* A_local, int64_t n, const capital_cholinv_args_t* args,
                                     capital_structure_t ostruct, double* R_local, double* Rinv_local) {
  CAP_TRY(need_comm(ctx));
  Dist D;
  CAP_TRY(dist_setup(D, ctx, false));
  CAP_TRY(cholinv_shape(D, n, args));
  const int64_t L = D.L;
  const size_t out_count = ostruct == CAPITAL_UPPERTRI_PACKED ? (size_t)L * (L + 1) / 2 : (size_t)L * L;
  CAP_CUDA(cudaEventRecord(ctx->ev_start, ctx->stream));
  const size_t bytes = cholinv_layout(D, nullptr);
  CAP_TRY(arena_prepare(ctx, bytes, "cholinv:" + std::to_string(L) + ":" + std::to_string(D.bc_local) + ":" + std::to_string(D.split)));
  cholinv_layout(D, D.P->arena);
  CAP_TRY(bc_workspace(D));
  CAP_TRY(cap_stage_out_begin(ctx, R_local, out_count, "R_out", &D.dR));
  CAP_TRY(cap_stage_out_begin(ctx, Rinv_local, out_count, "Rinv_out", &D.dRinv));
  D.hR = D.dR != R_local ? R_local : nullptr;
  D.hRinv = D.dRinv != Rinv_local ? Rinv_local : nullptr;
  CAP_TRY(cholinv_run(D, A_local, args, ostruct, R_local, Rinv_local, out_count));
  CAP_CUDA(cudaEventRecord(ctx->ev_stop, ctx->stream));
  return cap_check_info(ctx);
}

// Dry run of cholinv::factor on one rank of a grid: the sequence of synchronisation-relevant operations, 8 int64 per record
// (kind, stream, a .. f).  No device is touched.
extern "C" capital_status_t capital_dist_trace_cholinv(const capital_grid_t* grid, int64_t n, const capital_cholinv_args_t* args,
                                                        int64_t* out, int64_t cap_records, int64_t* n_records) {
  if (!grid || !args || !n_records || args->split <= 0) return CAPITAL_ERR_INVALID;
  capital_ctx fake;
  fake.grid = *grid;
  Peer P;
  P.size = grid->size; P.rank = grid->rank;
  P.arena = (char*)(uintptr_t)0x100000000ull;
  P.ctrl = (unsigned long long*)(uintptr_t)0x10000000ull;
  for (int r = 0; r < grid->size && r < PEER_MAX_RANKS; r++) { P.peer_arena[r] = P.arena; P.peer_ctrl[r] = P.ctrl; }
  fake.peer = &P;
  std::vector<int64_t> trace;
  Dist D;
  capital_status_t st = dist_setup(D, &fake, true);
  if (st == CAPITAL_OK) st = cholinv_shape(D, n, args);
  if (st == CAPITAL_OK) {
    D.trace = &trace;
    cholinv_layout(D, P.arena);
    // two consecutive calls: the hazards between factorizations are part of the protocol
    for (int rep = 0; rep < 2 && st == CAPITAL_OK; rep++) st = cholinv_run(D, (const double*)P.arena, args, CAPITAL_UPPERTRI_PACKED, nullptr, nullptr, 0);
  }
  fake.peer = nullptr;
  if (st != CAPITAL_OK) return st;
  *n_records = (int64_t)trace.size() / TREC;
  if (out) memcpy(out, trace.data(), (size_t)std::min<int64_t>(cap_records, *n_records) * TREC * 8);
  return CAPITAL_OK;
}

capital_status_t dist_cholinv_residual(capital_ctx* ctx, const double* A_local, int64_t n, capital_structure_t structure,
                                       const double* R_local, double* residual) {
  CAP_TRY(need_comm(ctx));
  Dist D;
  CAP_TRY(dist_setup(D, ctx, false));
  const capital_grid_t& g = D.g;
  if (n % g.d != 0) return CAPITAL_ERR_UNSUPPORTED;
  const int64_t L = n / g.d, ld = round_up(L, 16);
  D.L = L; D.ld = ld; D.split = 1; D.bc_local = L;
  const size_t r_count = structure == CAPITAL_UPPERTRI_PACKED ? (size_t)L * (L + 1) / 2 : (size_t)L * L;
  const double *dA, *dRin;
  CAP_TRY(cap_stage_in(ctx, A_local, (size_t)L * L, "A_in", &dA));
  CAP_TRY(cap_stage_in(ctx, R_local, r_count, "R_in", &dRin));
  // layout: E (= R^T R - A) and R with its operand slots, receive buffers for one L x L product, 2 x size x 2 scalars for the sum
  DMat E, Rr;
  double* ar = nullptr;
  auto layout = [&](char* base) {
    Layout lay(base);
    layout_mat(lay, D, E, ld, L, 0, false);
    layout_mat(lay, D, Rr, ld, L, ROLE_X | ROLE_Y, true);
    layout_exchange(lay, D, Q_CHAIN, L, L);
    ar = lay.take((size_t)2 * g.size * 2);
    return lay.off;
  };
  const size_t bytes = layout(nullptr);
  CAP_TRY(arena_prepare(ctx, bytes, "cholres:" + std::to_string(L)));
  layout(D.P->arena);
  ctx->comm_used = 0;
  CAP_TRY(fork_streams(D));
  cudaStream_t st = D.strm(S_CHAIN);
  if (structure == CAPITAL_UPPERTRI_PACKED) CAP_TRY(unpack_upper(ctx, st, L, dRin, Rr.own, ld));
  else CAP_TRY(triu_copy(ctx, st, L, dRin, L, Rr.own, ld, 0));
  if (g.y > g.x) CAP_TRY(triu_copy(ctx, st, L, Rr.own, ld, Rr.own, ld, 1));  // util::remove_triangle (validate.hpp:11): the local diagonal is below the global one there
  CAP_TRY(copy_block(ctx, st, L, L, dA, L, E.own, ld));
  CAP_CUDA(cudaMemsetAsync(ctx->d_scalars, 0, 2 * sizeof(double), st));
  CAP_TRY(sumsq_block(ctx, st, L, L, E.own, ld, 1, g.x, g.y, g.d, ctx->d_scalars + 1));
  CAP_TRY(push(D, Q_CHAIN, S_CHAIN, Rr, 0, 0, L, L, ROLE_X | ROLE_Y, nullptr));
  // E = R^T R - A  (validate.hpp:35).  No C_UPPER: on ranks with y > x the local diagonal is outside the global upper part anyway.
  CAP_TRY(product(D, Q_CHAIN, L, L, L, 1.0, Win{&Rr, 0, 0}, Win{&Rr, 0, 0}, -1.0, Win{&E, 0, 0}, CAPITAL_GEMM_A_UPPER | CAPITAL_GEMM_B_UPPER));
  CAP_TRY(sumsq_block(ctx, st, L, L, E.own, ld, 1, g.x, g.y, g.d, ctx->d_scalars));
  CAP_TRY(peer_allreduce_sum(ctx, st, ctx->d_scalars, 2, ar));
  CAP_TRY(join_streams(D));
  double h[2];
  CAP_CUDA(cudaMemcpyAsync(h, ctx->d_scalars, 2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CAP_TRY(cap_check_info(ctx));
  *residual = sqrt(h[0]) / sqrt(h[1]);
  return CAPITAL_OK;
}

capital_status_t dist_summa_gemm_tn(capital_ctx* ctx, int64_t m, int64_t n, int64_t k, double alpha, const double* A_local,
                                    const double* B_local, double beta, double* C_local) {
  CAP_TRY(need_comm(ctx));
  const capital_grid_t& g = ctx->grid;
  if (m % g.d || n % g.d || k % g.d) {
    ctx->set_error("summa gemm: d must divide m, n, k");
    return CAPITAL_ERR_UNSUPPORTED;
  }
  const int64_t ml = m / g.d, nl = n / g.d, kl = k / g.d;
  cudaStream_t us = ctx->stream;
  const double *dA, *dB;
  CAP_TRY(cap_stage_in(ctx, A_local, (size_t)kl * ml, "summa_A", &dA));
  CAP_TRY(cap_stage_in(ctx, B_local, (size_t)kl * nl, "summa_B", &dB));
  const bool c_host = !cap_is_device_ptr(C_local);
  const double* dCin = C_local;
  if (c_host) CAP_TRY(cap_stage_in(ctx, C_local, (size_t)ml * nl, "summa_C", &dCin));
  const int64_t ldk = round_up(kl, 2), ldm = round_up(ml, 2);
  if (g.size == 1) {
    // TMA needs even leading dimensions: repack operands whose local row count is odd
    double *pA = const_cast<double*>(dA), *pB = const_cast<double*>(dB);
    if (ldk != kl) {
      CAP_TRY(ctx->workspace("summa_pA", (size_t)ldk * ml * 8, (void**)&pA));
      CAP_TRY(ctx->workspace("summa_pB", (size_t)ldk * nl * 8, (void**)&pB));
      CAP_TRY(copy_block(ctx, us, kl, ml, dA, kl, pA, ldk));
      CAP_TRY(copy_block(ctx, us, kl, nl, dB, kl, pB, ldk));
    }
    double* dC = const_cast<double*>(dCin);
    CAP_TRY(gemm_tn(ctx, us, ml, nl, kl, alpha, pA, ldk, pB, ldk, beta, dC, ml, 0));
    if (c_host) CAP_TRY(cap_stage_out_end(ctx, C_local, (size_t)ml * nl, dC));
    CAP_CUDA(cudaStreamSynchronize(us));
    return CAPITAL_OK;
  }
  Dist D;
  CAP_TRY(dist_setup(D, ctx, false));
  DMat A, B, C;
  auto layout = [&](char* base) {
    Layout lay(base);
    layout_mat(lay, D, A, ldk, ml, ROLE_X, false);
    layout_mat(lay, D, B, ldk, nl, ROLE_Y, false);
    layout_mat(lay, D, C, ldm, nl, 0, false);
    layout_exchange(lay, D, Q_CHAIN, ml, nl);
    return lay.off;
  };
  const size_t bytes = layout(nullptr);
  CAP_TRY(arena_prepare(ctx, bytes, "summa:" + std::to_string(ml) + ":" + std::to_string(nl) + ":" + std::to_string(kl)));
  layout(D.P->arena);
  ctx->comm_used = 0;
  CAP_TRY(fork_streams(D));
  cudaStream_t st = D.strm(S_CHAIN);
  CAP_TRY(copy_block(ctx, st, kl, ml, dA, kl, A.own, ldk));
  CAP_TRY(copy_block(ctx, st, kl, nl, dB, kl, B.own, ldk));
  CAP_TRY(copy_block(ctx, st, ml, nl, dCin, ml, C.own, ldm));
  CAP_TRY(push(D, Q_CHAIN, S_CHAIN, A, 0, 0, kl, ml, ROLE_X, nullptr));
  CAP_TRY(push(D, Q_CHAIN, S_CHAIN, B, 0, 0, kl, nl, ROLE_Y, nullptr));
  CAP_TRY(product(D, Q_CHAIN, ml, nl, kl, alpha, Win{&A, 0, 0}, Win{&B, 0, 0}, beta, Win{&C, 0, 0}, 0));
  double* dC;
  CAP_TRY(cap_stage_out_begin(ctx, C_local, (size_t)ml * nl, "summa_Cout", &dC));
  CAP_TRY(copy_block(ctx, st, ml, nl, C.own, ldm, dC, ml));
  CAP_TRY(join_streams(D));
  CAP_TRY(cap_stage_out_end(ctx, C_local, (size_t)ml * nl, dC));
  return cap_check_info(ctx);
}

// ---- CholeskyQR2, 1D --------------------------------------------------------------------------------------------
namespace {
struct Qr {
  capital_ctx* ctx;
  cudaStream_t st;
  int64_t lr, n, ldq, ldn, ldt;
  double *Q, *Qt, *Qt2, *G, *W, *R1, *R2, *Ri, *RiT, *Rt, *ar;
};

// sweep_1d (cacqr.hpp:5-29): G = Q^T Q, all-reduce, R = chol(G), Rinv, Q <- Q Rinv.  R lands in `Rout`.
capital_status_t sweep(Qr& q, double* Rout) {
  capital_ctx* ctx = q.ctx;
  cudaStream_t st = q.st;
  const int64_t n = q.n, lr = q.lr;
  CAP_TRY(gemm_tn_splitk(ctx, st, n, n, lr, 1.0, q.Q, q.ldq, q.Q, q.ldq, q.G, q.ldn, CAPITAL_GEMM_C_UPPER));  // dsyrk 'U','T' (:15), deterministic split-k
  if (ctx->grid.size > 1) CAP_TRY(peer_allreduce_sum(ctx, st, q.G, q.ldn * n, q.ar));                          // policy.h:82
  CAP_CUDA(cudaMemsetAsync(q.Ri, 0, (size_t)q.ldn * n * 8, st));
  CAP_CUDA(cudaMemsetAsync(q.RiT, 0, (size_t)q.ldn * n * 8, st));
  CAP_CUDA(cudaMemsetAsync(Rout, 0, (size_t)q.ldn * n * 8, st));
  CAP_TRY(cholinv_local(ctx, st, n, q.G, q.ldn, Rout, q.ldn, q.Ri, q.ldn, q.RiT, q.ldn, true, n, 1));  // potrf + trtri (:20-22)
  // Q <- Q Rinv (dtrmm Right/Upper/NoTrans, :25) as (Q Rinv)^T = Rinv^T Q^T : A = Rinv (upper), B = Q^T
  CAP_TRY(transpose_block(ctx, st, lr, n, q.Q, q.ldq, q.Qt, q.ldt, 1.0));
  CAP_TRY(gemm_tn(ctx, st, n, lr, n, 1.0, q.Ri, q.ldn, q.Qt, q.ldt, 0.0, q.Qt2, q.ldt, CAPITAL_GEMM_A_UPPER));
  CAP_TRY(transpose_block(ctx, st, n, lr, q.Qt2, q.ldt, q.Q, q.ldq, 1.0));
  return CAPITAL_OK;
}
// The same sweep with every layout change folded into GEMM epilogues [default; CAPITAL_QR_TSTORE=0 selects the plain sweep above]:
//   Qc   : the panel, column-major (lr x n), read by the Gram product (K = rows, contiguous)
//   QtIn : its transpose (n x lr), read by the apply
//   QtOut: (optional) transpose of the updated panel = plain store of the apply, for the next sweep
//   QcOut: the updated panel, column-major = TRANSPOSED store of the apply's epilogue (no separate transpose pass)
capital_status_t sweep_tstore(Qr& q, const double* Qc, int64_t ldqc, const double* QtIn, double* QtOut, double* QcOut, int64_t ldqo, double* Rout) {
  capital_ctx* ctx = q.ctx;
  cudaStream_t st = q.st;
  const int64_t n = q.n, lr = q.lr;
  CAP_TRY(gemm_tn_splitk(ctx, st, n, n, lr, 1.0, Qc, ldqc, Qc, ldqc, q.G, q.ldn, CAPITAL_GEMM_C_UPPER));  // dsyrk 'U','T' (:15)
  if (ctx->grid.size > 1) CAP_TRY(peer_allreduce_sum(ctx, st, q.G, q.ldn * n, q.ar));                    // policy.h:82
  CAP_CUDA(cudaMemsetAsync(q.Ri, 0, (size_t)q.ldn * n * 8, st));
  CAP_CUDA(cudaMemsetAsync(q.RiT, 0, (size_t)q.ldn * n * 8, st));
  CAP_CUDA(cudaMemsetAsync(Rout, 0, (size_t)q.ldn * n * 8, st));
  CAP_TRY(cholinv_local(ctx, st, n, q.G, q.ldn, Rout, q.ldn, q.Ri, q.ldn, q.RiT, q.ldn, true, n, 1));  // potrf + trtri (:20-22)
  // Q <- Q Rinv (dtrmm Right/Upper/NoTrans, :25): (Q Rinv)^T = Rinv^T Q^T, A = Rinv (upper), B = Q^T
  return gemm_tn_t(ctx, st, n, lr, n, 1.0, q.Ri, q.ldn, QtIn, q.ldt, QtOut, q.ldt, QcOut, ldqo, CAPITAL_GEMM_A_UPPER);
}
// small all-reduce scratch of the 1D path: an arena region of 2 * size * count doubles
capital_status_t qr1d_arena(capital_ctx* ctx, int64_t count, double** ar) {
  *ar = nullptr;
  if (ctx->grid.size == 1) return CAPITAL_OK;
  const size_t bytes = (size_t)2 * ctx->grid.size * count * 8 + 4096;
  CAP_TRY(arena_prepare(ctx, bytes, "qr1d:" + std::to_string(count)));
  *ar = (double*)peer_of(ctx)->arena;
  return CAPITAL_OK;
}
}  // namespace

// ---- CholeskyQR2, 3D grid (c == d) ---------------------------------------------------------------------------------
// qr::cacqr::invoke_3d / sweep_3d (cacqr.hpp:75-120,195-215): Gram matrix by a SUMMA step, cholinv::factor on the n x n Gram
// matrix over the same grid, Q <- Q R^{-1} by a SUMMA trmm.  Here each of those is the distributed A^T B product of this file:
//   G    = Q^T Q                      product(X = Q, Y = Q)                   [row Bcast + dgemm + column Reduce + depth Bcast, :92-99]
//   R, R^{-1} from invoke() on G                                                 [cholinv::factor, :103]
//   Q^T <- R^{-T} Q^T                  product(X = Rinv (upper), Y = Q^T)      [summa trmm Right/Upper, :111]
// with the global transposes done through the transpose partner's mirror slot (util::transpose).  The complete inverse is always
// formed (the reference's block `solve` for complete_inv == 0, :44-73, yields the same Q).
namespace {
struct Qr3 {
  Dist* D;
  int64_t ml, nl, ldq, ldn;
  DMat Q, T1, T2, R1, R2, Rt, Rf;
};
size_t qr3_layout(Qr3& q, char* base) {
  Dist& D = *q.D;
  Layout lay(base);
  const int64_t nl = q.nl, ml = q.ml, ld = q.ldn;
  layout_mat(lay, D, D.W, ld, nl, ROLE_X | ROLE_Y, false);
  layout_mat(lay, D, D.R, ld, nl, ROLE_X | ROLE_Y, true);
  layout_mat(lay, D, D.Ri, ld, nl, ROLE_X | ROLE_Y | ROLE_T, true);
  layout_mat(lay, D, D.RiT, ld, nl, ROLE_Y, false);
  layout_mat(lay, D, q.Q, q.ldq, nl, ROLE_X | ROLE_Y | ROLE_T, true);
  layout_mat(lay, D, q.T1, ld, ml, ROLE_Y, false);
  layout_mat(lay, D, q.T2, ld, ml, ROLE_T, false);
  layout_mat(lay, D, q.R1, ld, nl, ROLE_Y, false);
  layout_mat(lay, D, q.R2, ld, nl, ROLE_T, false);
  layout_mat(lay, D, q.Rt, ld, nl, ROLE_X, false);
  layout_mat(lay, D, q.Rf, ld, nl, 0, false);
  layout_exchange(lay, D, Q_CHAIN, nl, std::max(ml, nl));
  layout_gather(lay, D);
  return lay.off;
}
capital_status_t qr3_setup(capital_ctx* ctx, Dist& D, Qr3& q, int64_t m, int64_t n, const capital_cholinv_args_t* ci_args, const char* tag) {
  CAP_TRY(dist_setup(D, ctx, false));
  const capital_grid_t& g = D.g;
  if (m % g.d || n % g.d) {
    ctx->set_error("cacqr 3D: d must divide m and n");
    return CAPITAL_ERR_UNSUPPORTED;
  }
  q.D = &D;
  q.ml = m / g.d; q.nl = n / g.d; q.ldq = round_up(q.ml, 16); q.ldn = round_up(q.nl, 16);
  D.L = q.nl; D.ld = q.ldn; D.split = ci_args ? (int)ci_args->split : 1;
  if (D.split <= 0) D.split = 1;
  D.bc_local = capital_cholinv_bc_dimension(q.nl, g.c, g.d, ci_args ? ci_args->bc_mult_dim : 0) / g.d;
  D.two_stream = false;  // the Gram matrix is small: everything on the chain
  if (g.size == 1) {
    // degenerate grid (tests force the 3D code onto 1 x 1 x 1): a private arena-like buffer, no peers
    const size_t bytes = qr3_layout(q, nullptr);
    char* buf;
    CAP_TRY(ctx->workspace("q3arena", bytes, (void**)&buf));
    if (ctx->arena_signature != std::string(tag)) { CAP_CUDA(cudaMemsetAsync(buf, 0, bytes, ctx->stream)); ctx->arena_signature = tag; }
    qr3_layout(q, buf);
  } else {
    const size_t bytes = qr3_layout(q, nullptr);
    CAP_TRY(arena_prepare(ctx, bytes, std::string(tag) + ":" + std::to_string(q.ml) + ":" + std::to_string(q.nl) + ":" + std::to_string(D.bc_local) + ":" + std::to_string(D.split)));
    qr3_layout(q, D.P->arena);
  }
  CAP_TRY(bc_workspace(D));
  return CAPITAL_OK;
}
capital_status_t sweep3d(Qr3& q, DMat& Rout) {
  Dist& D = *q.D;
  capital_ctx* ctx = D.ctx;
  cudaStream_t st = D.strm(S_CHAIN);
  const int64_t ml = q.ml, nl = q.nl, ld = q.ldn;
  Token tq;
  CAP_TRY(push(D, Q_CHAIN, S_CHAIN, q.Q, 0, 0, ml, nl, ROLE_X | ROLE_Y | ROLE_T, &tq));
  CAP_TRY(product(D, Q_CHAIN, nl, nl, ml, 1.0, Win{&q.Q, 0, 0}, Win{&q.Q, 0, 0}, 0.0, Win{&D.W, 0, 0}, 0));
  CAP_TRY(invoke(D, 0, nl, true, -1, Token{}, 0));
  CAP_TRY(copy_block(ctx, st, nl, nl, D.R.own, ld, Rout.own, ld));
  CAP_TRY(transpose_dist(D, Q_CHAIN, q.Q, 0, 0, ml, nl, &tq, q.T1.own, ld));                                        // T1 = Q^T
  CAP_TRY(push(D, Q_CHAIN, S_CHAIN, q.T1, 0, 0, nl, ml, ROLE_Y, nullptr));
  CAP_TRY(product(D, Q_CHAIN, nl, ml, nl, 1.0, Win{&D.Ri, 0, 0}, Win{&q.T1, 0, 0}, 0.0, Win{&q.T2, 0, 0}, CAPITAL_GEMM_A_UPPER));  // T2 = Rinv^T Q^T
  Token t2;
  CAP_TRY(push(D, Q_CHAIN, S_CHAIN, q.T2, 0, 0, nl, ml, ROLE_T, &t2));
  CAP_TRY(transpose_dist(D, Q_CHAIN, q.T2, 0, 0, nl, ml, &t2, q.Q.own, q.ldq));                                     // Q = T2^T
  return CAPITAL_OK;
}
capital_status_t cacqr3d_factor(capital_ctx* ctx, const double* A_local, int64_t m, int64_t n, int num_iter, const capital_cholinv_args_t* ci_args,
                                capital_structure_t rstruct, double* Q_local, double* R_local) {
  CAP_CUDA(cudaEventRecord(ctx->ev_start, ctx->stream));
  Dist D;
  Qr3 q{};
  CAP_TRY(qr3_setup(ctx, D, q, m, n, ci_args, "qr3d"));
  const capital_grid_t& g = D.g;
  const int64_t ml = q.ml, nl = q.nl, ld = q.ldn;
  const double* dA;
  CAP_TRY(cap_stage_in(ctx, A_local, (size_t)ml * nl, "A_in", &dA));
  const size_t r_count = rstruct == CAPITAL_UPPERTRI_PACKED ? (size_t)nl * (nl + 1) / 2 : (size_t)nl * nl;
  double *dQ, *dR;
  CAP_TRY(cap_stage_out_begin(ctx, Q_local, (size_t)ml * nl, "Q_out", &dQ));
  CAP_TRY(cap_stage_out_begin(ctx, R_local, r_count, "R_out", &dR));
  ctx->comm_used = 0;
  CAP_TRY(fork_streams(D));
  cudaStream_t st = D.strm(S_CHAIN);
  CAP_CUDA(cudaMemsetAsync(ctx->d_info, 0, sizeof(int), st));
  CAP_TRY(copy_block(ctx, st, ml, nl, dA, ml, q.Q.own, q.ldq));
  CAP_TRY(sweep3d(q, q.R1));
  const double* Rfinal = q.R1.own;
  if (num_iter > 1) {
    CAP_TRY(sweep3d(q, q.R2));
    // R = R2 R1 = (R2^T)^T R1  (cacqr.hpp:207-209)
    Token t2;
    CAP_TRY(push(D, Q_CHAIN, S_CHAIN, q.R2, 0, 0, nl, nl, ROLE_T, &t2));
    CAP_TRY(transpose_dist(D, Q_CHAIN, q.R2, 0, 0, nl, nl, &t2, q.Rt.own, ld));
    CAP_TRY(push(D, Q_CHAIN, S_CHAIN, q.Rt, 0, 0, nl, nl, ROLE_X, nullptr));
    CAP_TRY(push(D, Q_CHAIN, S_CHAIN, q.R1, 0, 0, nl, nl, ROLE_Y, nullptr));
    CAP_CUDA(cudaMemsetAsync(q.Rf.own, 0, (size_t)ld * nl * 8, st));
    CAP_TRY(product(D, Q_CHAIN, nl, nl, nl, 1.0, Win{&q.Rt, 0, 0}, Win{&q.R1, 0, 0}, 0.0, Win{&q.Rf, 0, 0}, CAPITAL_GEMM_A_LOWER | CAPITAL_GEMM_B_UPPER));
    Rfinal = q.Rf.own;
  }
  const int zd = g.y > g.x ? 1 : 0;  // local diagonal is below the global diagonal on those ranks
  if (rstruct == CAPITAL_UPPERTRI_PACKED) CAP_TRY(pack_upper(ctx, st, nl, Rfinal, ld, dR, zd));
  else CAP_TRY(triu_copy(ctx, st, nl, Rfinal, ld, dR, nl, zd));
  CAP_TRY(copy_block(ctx, st, ml, nl, q.Q.own, q.ldq, dQ, ml));
  CAP_TRY(join_streams(D));
  CAP_TRY(cap_stage_out_end(ctx, Q_local, (size_t)ml * nl, dQ));
  CAP_TRY(cap_stage_out_end(ctx, R_local, r_count, dR));
  CAP_CUDA(cudaEventRecord(ctx->ev_stop, ctx->stream));
  return cap_check_info(ctx);
}
capital_status_t cacqr3d_residual(capital_ctx* ctx, const double* A_local, int64_t m, int64_t n, const double* Q_local,
                                  capital_structure_t rstruct, const double* R_local, double* residual, double* orthogonality) {
  Dist D;
  Qr3 q{};
  capital_cholinv_args_t dummy{1, 1, 0, 'U'};
  CAP_TRY(qr3_setup(ctx, D, q, m, n, &dummy, "qr3dres"));
  const capital_grid_t& g = D.g;
  const int64_t ml = q.ml, nl = q.nl, ld = q.ldn;
  const size_t r_count = rstruct == CAPITAL_UPPERTRI_PACKED ? (size_t)nl * (nl + 1) / 2 : (size_t)nl * nl;
  const double *dA, *dQ, *dRin;
  CAP_TRY(cap_stage_in(ctx, A_local, (size_t)ml * nl, "A_in", &dA));
  CAP_TRY(cap_stage_in(ctx, Q_local, (size_t)ml * nl, "Q_in", &dQ));
  CAP_TRY(cap_stage_in(ctx, R_local, r_count, "R_in", &dRin));
  double* ar;
  CAP_TRY(ctx->workspace("q3ar_local", 64, (void**)&ar));  // placeholder when size == 1
  ctx->comm_used = 0;
  CAP_TRY(fork_streams(D));
  cudaStream_t st = D.strm(S_CHAIN);
  // Rr lives in D.R (operand of X role), Q^T in T1 (Y), A^T in T2 (accumulator), Q^T Q in W
  DMat& Rr = D.R;
  if (rstruct == CAPITAL_UPPERTRI_PACKED) CAP_TRY(unpack_upper(ctx, st, nl, dRin, Rr.own, ld));
  else CAP_TRY(triu_copy(ctx, st, nl, dRin, nl, Rr.own, ld, 0));
  if (g.y > g.x) CAP_TRY(triu_copy(ctx, st, nl, Rr.own, ld, Rr.own, ld, 1));  // util::remove_triangle (validate.hpp:42)
  CAP_CUDA(cudaMemsetAsync(ctx->d_scalars, 0, 3 * sizeof(double), st));
  // residual: (Q R)^T - A^T = R^T Q^T - A^T
  Token t;
  CAP_TRY(copy_block(ctx, st, ml, nl, dA, ml, q.Q.own, q.ldq));
  CAP_TRY(push(D, Q_CHAIN, S_CHAIN, q.Q, 0, 0, ml, nl, ROLE_T, &t));
  CAP_TRY(transpose_dist(D, Q_CHAIN, q.Q, 0, 0, ml, nl, &t, q.T2.own, ld));   // A^T
  CAP_TRY(sumsq_block(ctx, st, nl, ml, q.T2.own, ld, 0, 0, 0, 1, ctx->d_scalars + 1));
  if (g.size > 1) CAP_TRY(peer_barrier(ctx, st));  // the partner has read its copy of A before Q overwrites the slot
  CAP_TRY(copy_block(ctx, st, ml, nl, dQ, ml, q.Q.own, q.ldq));
  CAP_TRY(push(D, Q_CHAIN, S_CHAIN, q.Q, 0, 0, ml, nl, ROLE_X | ROLE_Y | ROLE_T, &t));
  CAP_TRY(transpose_dist(D, Q_CHAIN, q.Q, 0, 0, ml, nl, &t, q.T1.own, ld));   // Q^T
  CAP_TRY(push(D, Q_CHAIN, S_CHAIN, q.T1, 0, 0, nl, ml, ROLE_Y, nullptr));
  CAP_TRY(push(D, Q_CHAIN, S_CHAIN, Rr, 0, 0, nl, nl, ROLE_X | ROLE_Y, nullptr));
  CAP_TRY(product(D, Q_CHAIN, nl, ml, nl, 1.0, Win{&Rr, 0, 0}, Win{&q.T1, 0, 0}, -1.0, Win{&q.T2, 0, 0}, CAPITAL_GEMM_A_UPPER));
  CAP_TRY(sumsq_block(ctx, st, nl, ml, q.T2.own, ld, 0, 0, 0, 1, ctx->d_scalars));
  // orthogonality: Q^T Q - I
  CAP_TRY(product(D, Q_CHAIN, nl, nl, ml, 1.0, Win{&q.Q, 0, 0}, Win{&q.Q, 0, 0}, 0.0, Win{&D.W, 0, 0}, 0));
  if (g.x == g.y) CAP_TRY(sub_identity_local(ctx, st, nl, D.W.own, ld));
  CAP_TRY(sumsq_block(ctx, st, nl, nl, D.W.own, ld, 0, 0, 0, 1, ctx->d_scalars + 2));
  if (g.size > 1) CAP_TRY(peer_allreduce_sum(ctx, st, ctx->d_scalars, 3, q.Rf.own));  // every layer holds a replica: all three sums carry the same factor c
  CAP_TRY(join_streams(D));
  double h[3];
  CAP_CUDA(cudaMemcpyAsync(h, ctx->d_scalars, 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  CAP_TRY(cap_check_info(ctx));
  *residual = sqrt(h[0]) / sqrt(h[1]);
  *orthogonality = sqrt(h[2] / g.c) / sqrt((double)n * (double)n);
  return CAPITAL_OK;
}
inline bool use_3d(const capital_grid_t& g) {
  if (g.c != g.d) return false;
  if (g.c > 1) return true;
  const char* e = getenv("CAPITAL_FORCE_QR3D");  // 1x1x1: the reference takes the 1D path (cacqr.hpp:229); tests may force the 3D code
  return e && atoi(e) != 0;
}
}  // namespace

capital_status_t dist_cacqr_factor(capital_ctx* ctx, const double* A_local, int64_t m, int64_t n, int num_iter,
                                   const capital_cholinv_args_t* ci_args, capital_structure_t rstruct, double* Q_local, double* R_local) {
  const capital_grid_t& g = ctx->grid;
  CAP_TRY(need_comm(ctx));
  if (use_3d(g)) return cacqr3d_factor(ctx, A_local, m, n, num_iter, ci_args, rstruct, Q_local, R_local);
  if (g.c != 1 || g.size != g.d) {
    // rows are split over d and the Gram matrix is summed over the whole world: that is only right when the world IS the d ranks
    // (topo::rect with c == 1, cacqr.hpp:229)
    ctx->set_error("cacqr: 1D (rect grid, c == 1, d == size; cacqr.hpp:229) and 3D (c == d, :232) grids are implemented; the tunable c < d grid (:234-246) is not");
    return CAPITAL_ERR_UNSUPPORTED;
  }
  const int64_t lr = ceil_div(m, g.d);
  cudaStream_t st = ctx->stream;
  CAP_CUDA(cudaEventRecord(ctx->ev_start, st));
  Qr q{ctx, st};
  q.lr = lr; q.n = n; q.ldq = round_up(lr, 16); q.ldn = round_up(n, 16); q.ldt = q.ldn;
  const double* dA;
  CAP_TRY(cap_stage_in(ctx, A_local, (size_t)lr * n, "A_in", &dA));
  const size_t r_count = rstruct == CAPITAL_UPPERTRI_PACKED ? (size_t)n * (n + 1) / 2 : (size_t)n * n;
  double *dQ, *dR;
  CAP_TRY(cap_stage_out_begin(ctx, Q_local, (size_t)lr * n, "Q_out", &dQ));
  CAP_TRY(cap_stage_out_begin(ctx, R_local, r_count, "R_out", &dR));
  CAP_TRY(ctx->workspace("qrQ", (size_t)q.ldq * n * 8, (void**)&q.Q));
  CAP_TRY(ctx->workspace("qrQt", (size_t)q.ldt * lr * 8, (void**)&q.Qt));
  CAP_TRY(ctx->workspace("qrQt2", (size_t)q.ldt * lr * 8, (void**)&q.Qt2));
  const size_t nn = (size_t)q.ldn * n * 8;
  CAP_TRY(ctx->workspace("qrG", nn, (void**)&q.G));
  CAP_TRY(ctx->workspace("qrR1", nn, (void**)&q.R1));
  CAP_TRY(ctx->workspace("qrR2", nn, (void**)&q.R2));
  CAP_TRY(ctx->workspace("qrRi", nn, (void**)&q.Ri));
  CAP_TRY(ctx->workspace("qrRiT", nn, (void**)&q.RiT));
  CAP_TRY(ctx->workspace("qrRt", nn, (void**)&q.Rt));
  CAP_TRY(qr1d_arena(ctx, q.ldn * n, &q.ar));
  CAP_CUDA(cudaMemsetAsync(ctx->d_info, 0, sizeof(int), st));
  const char* ets = getenv("CAPITAL_QR_TSTORE");
  const bool tstore = !(ets && atoi(ets) == 0);
  const double* Rfinal = q.R1;
  bool q_in_place = false;  // the final panel already sits in the caller's Q
  if (tstore) {
    // Q <- A (cacqr.hpp:226): the Gram product reads A where it lies when its leading dimension suits TMA (even, 16-byte aligned
    // base); the apply wants the transpose, made once here -- every later layout change happens inside a GEMM epilogue
    const double* Qc = dA;
    int64_t ldqc = lr;
    if ((lr & 1) || ((uintptr_t)dA & 15)) {
      CAP_TRY(copy_block(ctx, st, lr, n, dA, lr, q.Q, q.ldq));
      Qc = q.Q; ldqc = q.ldq;
    }
    CAP_TRY(transpose_block(ctx, st, lr, n, dA, lr, q.Qt, q.ldt, 1.0));
    q_in_place = (dQ == Q_local);  // device output: the last apply writes it directly (leading dimension lr)
    double* Qlast = q_in_place ? dQ : q.Q;
    const int64_t ldlast = q_in_place ? lr : q.ldq;
    if (num_iter > 1) {
      CAP_TRY(sweep_tstore(q, Qc, ldqc, q.Qt, q.Qt2, q.Q, q.ldq, q.R1));
      CAP_TRY(sweep_tstore(q, q.Q, q.ldq, q.Qt2, nullptr, Qlast, ldlast, q.R2));  // (the apply reads Q^T: the panel may be overwritten)
    } else {
      CAP_TRY(sweep_tstore(q, Qc, ldqc, q.Qt, nullptr, Qlast, ldlast, q.R1));
    }
  } else {
    CAP_TRY(copy_block(ctx, st, lr, n, dA, lr, q.Q, q.ldq));  // Q <- A (cacqr.hpp:226)
    CAP_TRY(sweep(q, q.R1));
    if (num_iter > 1) CAP_TRY(sweep(q, q.R2));
  }
  if (num_iter > 1) {
    // R = R2 R1 (dtrmm, cacqr.hpp:185-187) = (R2^T)^T R1 : A = R2^T (lower), B = R1 (upper)
    CAP_TRY(transpose_block(ctx, st, n, n, q.R2, q.ldn, q.Rt, q.ldn, 1.0));
    CAP_TRY(gemm_tn(ctx, st, n, n, n, 1.0, q.Rt, q.ldn, q.R1, q.ldn, 0.0, q.G, q.ldn,
                    CAPITAL_GEMM_A_LOWER | CAPITAL_GEMM_B_UPPER | CAPITAL_GEMM_C_UPPER));
    Rfinal = q.G;
  }
  if (rstruct == CAPITAL_UPPERTRI_PACKED) CAP_TRY(pack_upper(ctx, st, n, Rfinal, q.ldn, dR, 0));
  else CAP_TRY(triu_copy(ctx, st, n, Rfinal, q.ldn, dR, n, 0));
  if (!q_in_place) CAP_TRY(copy_block(ctx, st, lr, n, q.Q, q.ldq, dQ, lr));
  CAP_TRY(cap_stage_out_end(ctx, Q_local, (size_t)lr * n, dQ));
  CAP_TRY(cap_stage_out_end(ctx, R_local, r_count, dR));
  CAP_CUDA(cudaEventRecord(ctx->ev_stop, st));
  return cap_check_info(ctx);
}

capital_status_t dist_cacqr_residual(capital_ctx* ctx, const double* A_local, int64_t m, int64_t n, const double* Q_local,
                                     capital_structure_t rstruct, const double* R_local, double* residual, double* orthogonality) {
  const capital_grid_t& g = ctx->grid;
  CAP_TRY(need_comm(ctx));
  if (use_3d(g)) return cacqr3d_residual(ctx, A_local, m, n, Q_local, rstruct, R_local, residual, orthogonality);
  if (g.c != 1 || g.size != g.d) return CAPITAL_ERR_UNSUPPORTED;
  const int64_t lr = ceil_div(m, g.d);
  cudaStream_t st = ctx->stream;
  const int64_t ldq = round_up(lr, 16), ldn = round_up(n, 16);
  const size_t r_count = rstruct == CAPITAL_UPPERTRI_PACKED ? (size_t)n * (n + 1) / 2 : (size_t)n * n;
  const double *dA, *dQ, *dRin;
  CAP_TRY(cap_stage_in(ctx, A_local, (size_t)lr * n, "A_in", &dA));
  CAP_TRY(cap_stage_in(ctx, Q_local, (size_t)lr * n, "Q_in", &dQ));
  CAP_TRY(cap_stage_in(ctx, R_local, r_count, "R_in", &dRin));
  double *Q, *Qt, *Et, *R, *G, *ar;
  CAP_TRY(ctx->workspace("qrQ", (size_t)ldq * n * 8, (void**)&Q));
  CAP_TRY(ctx->workspace("qrQt", (size_t)ldn * lr * 8, (void**)&Qt));
  CAP_TRY(ctx->workspace("qrQt2", (size_t)ldn * lr * 8, (void**)&Et));
  CAP_TRY(ctx->workspace("qrR1", (size_t)ldn * n * 8, (void**)&R));
  CAP_TRY(ctx->workspace("qrG", (size_t)ldn * n * 8, (void**)&G));
  CAP_TRY(qr1d_arena(ctx, ldn * n, &ar));
  CAP_TRY(copy_block(ctx, st, lr, n, dQ, lr, Q, ldq));
  if (rstruct == CAPITAL_UPPERTRI_PACKED) CAP_TRY(unpack_upper(ctx, st, n, dRin, R, ldn));
  else CAP_TRY(triu_copy(ctx, st, n, dRin, n, R, ldn, 0));
  CAP_CUDA(cudaMemsetAsync(ctx->d_scalars, 0, 3 * sizeof(double), st));
  // residual (validate.hpp:37-52): ||QR - A||_F / ||A||_F, via (QR)^T - A^T = R^T Q^T - A^T
  CAP_TRY(transpose_block(ctx, st, lr, n, Q, ldq, Qt, ldn, 1.0));
  CAP_TRY(transpose_block(ctx, st, lr, n, dA, lr, Et, ldn, 1.0));
  CAP_TRY(sumsq_block(ctx, st, n, lr, Et, ldn, 0, 0, 0, 1, ctx->d_scalars + 1));
  CAP_TRY(gemm_tn(ctx, st, n, lr, n, 1.0, R, ldn, Qt, ldn, -1.0, Et, ldn, CAPITAL_GEMM_A_UPPER));
  CAP_TRY(sumsq_block(ctx, st, n, lr, Et, ldn, 0, 0, 0, 1, ctx->d_scalars));
  // orthogonality (validate.hpp:7-35): ||Q^T Q - I||_F / sqrt(n^2)
  CAP_TRY(gemm_tn_splitk(ctx, st, n, n, lr, 1.0, Q, ldq, Q, ldq, G, ldn, 0));
  if (g.size > 1) CAP_TRY(peer_allreduce_sum(ctx, st, G, ldn * n, ar));
  CAP_TRY(sub_identity_local(ctx, st, n, G, ldn));
  CAP_TRY(sumsq_block(ctx, st, n, n, G, ldn, 0, 0, 0, 1, ctx->d_scalars + 2));
  if (g.size > 1) CAP_TRY(peer_allreduce_sum(ctx, st, ctx->d_scalars, 2, ar));  // numerator/denominator of the residual are row-partitioned sums
  double h[3];
  CAP_CUDA(cudaMemcpyAsync(h, ctx->d_scalars, 3 * sizeof(double), cudaMemcpyDeviceToHost, st));
  CAP_TRY(cap_check_info(ctx));
  *residual = sqrt(h[0]) / sqrt(h[1]);
  *orthogonality = sqrt(h[2]) / sqrt((double)n * (double)n);
  return CAPITAL_OK;
}
