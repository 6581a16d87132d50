// hifgpu.h -- internal host-side structures of the device backend.
#pragma once

#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/hifir_b200.h"
#include "common.cuh"

namespace hifgpu {

// device buffer with ownership
template <class T>
struct DevBuf {
  T *         p = nullptr;
  std::size_t n = 0;
  DevBuf()      = default;
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  DevBuf(DevBuf &&o) noexcept : p(o.p), n(o.n) { o.p = nullptr, o.n = 0; }
  DevBuf &operator=(DevBuf &&o) noexcept {
    if (this != &o) {
      release();
      p = o.p, n = o.n;
      o.p = nullptr, o.n = 0;
    }
    return *this;
  }
  ~DevBuf() { release(); }
  void release() {
    if (p) cudaFree(p);
    p = nullptr, n = 0;
  }
  void alloc(std::size_t count, std::size_t *tally = nullptr) {
    release();
    n = count;
    if (count) {
      HIF_CUDA(cudaMalloc(&p, count * sizeof(T)));
      HIF_CUDA(cudaMemset(p, 0, count * sizeof(T)));
      // the handle's stream is non-blocking: make sure the (legacy-stream) memset has landed
      // before any kernel of the handle can touch the buffer (tagged buffers rely on it)
      HIF_CUDA(cudaDeviceSynchronize());
      if (tally) *tally += count * sizeof(T);
    }
  }
  void upload(const T *host, std::size_t count, std::size_t *tally = nullptr) {
    alloc(count, tally);
    if (count) HIF_CUDA(cudaMemcpy(p, host, count * sizeof(T), cudaMemcpyHostToDevice));
  }
  void upload(const std::vector<T> &v, std::size_t *tally = nullptr) { upload(v.data(), v.size(), tally); }
};

// compressed-row matrix on the device (row-gather form of a reference CCS block)
struct DevCsr {
  std::size_t      nrows = 0, ncols = 0, nnz = 0;
  DevBuf<unsigned> ptr;  // nrows+1
  DevBuf<int>      col;  // nnz, ascending within a row
  DevBuf<double>   val;  // nnz
};

// host CSR used during attach
struct HostCsr {
  std::size_t           nrows = 0, ncols = 0;
  std::vector<unsigned> ptr;
  std::vector<int>      col;
  std::vector<double>   val;
  // "sweep form" of a triangular factor (merge.cu): rows in sweep order, every entry references
  // an earlier row, and gid[r] is the ROW CODE of row r (empty = identity):
  //   bits 0..30  slot of the row's result in the tagged solution buffer (2 * orig_rows slots:
  //               [0, orig_rows) the solution itself, [orig_rows, 2 orig_rows) auxiliary unknowns)
  //   bit 31      the row's right-hand side is zero
  // right-hand side index of a row = slot < orig_rows ? slot : slot - orig_rows
  std::vector<unsigned> gid;
  std::size_t           orig_rows = 0;
};
constexpr unsigned kMrhsWidth = 8;  // columns processed together by the multi-rhs kernels
constexpr unsigned kSyncStride = 32;  // ints between two level counters of a streaming sweep (stream.cu)
constexpr unsigned kCodeZeroRhs = 0x80000000u, kCodeSlotMask = 0x7fffffffu;

// algebraic level merging (merge.cu)
struct MergeParams {
  bool     enabled   = true;
  double   gain      = 1000000.0;  // fill (in nonzeros) one saved dependent step may cost
  unsigned row_cap   = 256;       // longest row of an inverted diagonal block
  unsigned bmax      = 64;        // most level sets merged into one super level
  double   row_cost  = 2.0;       // cost of one auxiliary row, in nonzeros
  bool     chain     = true;      // chain the t rows of consecutive super levels (one step per super level)
  int      alap      = 1;         // as-late-as-possible level sets: 0 never, 1 fan-out sweeps (U: leaves last), 2 always
  double   sl_cap    = 300000.0;  // a super level stops growing at this many entries: beyond, its two
                                  // steps are throughput bound and more fill only costs (measured optimum 4e5-8e5)
  bool     slack     = false;     // slack-aware merging (merge_slack): only rows pinned to the critical core pay fill
  unsigned steps     = 0;         // > 0: proportional scheduling into this many steps (merge_prop)
  bool     chain_all = true;      // chain every row (not only the pinned ones) to the t rows of the previous step
  bool     auto_caps = true;      // choose sl_cap per factor with the cost model below (merge_levels)
  // Cost model of one warp-stream sweep over a plan (us, B200 at 1000 W):
  //   t = tau_step * dependent steps + c_entry * stored entries
  // [0]: the packed plan (~12 B per entry + 8 B per row) is larger than l2_bytes and streams from HBM,
  // [1]: it stays L2-resident.  Least-squares fit to the merge-cap curve of Poisson 128^3 (fused L-then-U
  // launches of all four levels, 9 plans each; profiles/r03_tune_poisson128.log): rms error 21 us over
  // 13 launches of 370-1000 us [0], 30 us over 23 launches of 47-1200 us [1].  A small factor does not
  // fill the machine, so its entries cost six times more: fill pays off far earlier than in a large one.
  double   tau_step[2] = {1.31, 1.11};
  double   c_entry[2]  = {3.44e-6, 2.13e-5};
  double   l2_bytes    = 40.0e6;
  static MergeParams from_env();
  // predicted time of one sweep over a plan with these statistics
  double plan_cost(std::size_t steps, std::size_t entries, std::size_t rows) const;
  template <class St>
  double plan_cost(const St &s) const { return plan_cost(s.ext_depth, s.ext_nnz, s.ext_rows); }
};
struct MergeStats {
  std::size_t rows = 0, ext_rows = 0, nnz = 0, ext_nnz = 0, depth = 0, ext_depth = 0, super_levels = 0;
};
HostCsr to_sweep_form(const HostCsr &T, bool upper);
void    validate_sweep_form(const HostCsr &S);  // throws std::invalid_argument
HostCsr merge_levels(const HostCsr &S, const MergeParams &prm, MergeStats *st, bool fan_out = false);

// ---- arena.cu : factor arena serialization (SURVEY.md 8f rank 3)
struct MergedFactor {  // result of to_sweep_form + merge_levels for one L_B / U_B
  HostCsr    S;
  MergeStats st;
  bool       upper = false;
};
struct PlanCache {  // in attach order: level 0 L, level 0 U, level 1 L, ...
  std::vector<MergedFactor> f;
  std::size_t               next = 0;
};
extern thread_local PlanCache *tls_plan_cache;  // non-null while attaching from an arena file with plans
// to_sweep_form + merge_levels (when enabled) of one factor, or the stored plan of the arena file
HostCsr merged_sweep_form(const HostCsr &Tnat, bool upper, const MergeParams &mp, MergeStats *ms);
void    save_levels_file(const char *path, std::size_t nlevels, const LhfdGpuLevel *lv, bool f32, bool with_plans);
struct ArenaFile {  // an arena file read back: the level description (+ plans) with the arrays it points into
  std::vector<LhfdGpuLevel> lv;
  bool                      f32 = false, has_plans = false;
  std::size_t               nnz_total = 0;
  PlanCache                 plans;
  ArenaFile();
  ~ArenaFile();
  ArenaFile(const ArenaFile &) = delete;
  ArenaFile &operator=(const ArenaFile &) = delete;
  void load(const char *path, bool want_plans);
 private:
  struct Impl;
  Impl *impl;
};
struct Handle;
Handle *attach_file(int device, const char *path, bool want_f32);

// a strictly triangular factor prepared for the device sweeps
struct SweepPlan {
  unsigned               m = 0, nblocks = 0, nr = 1;  // nblocks: slices; nr: right-hand sides per slot
  bool                   upper = false;
  MergeStats             merge;
  // level-major streaming layout (stream.cu); nblocks = number of 32-row slices
  bool                        stream = false;
  std::size_t                 st_depth = 0, st_padded = 0;
  unsigned                    st_chunks = 0;  // 8 slices each, all of one level set
  unsigned                    st_u = 8;       // entries per lane held in registers (kernel variant)
  DevBuf<unsigned>            st_need;   // chunks per level set
  DevBuf<unsigned>            st_sdesc;  // uint4 per slice: offset (units of 32 entries), entries per lane, log2 lanes per row, level
  DevBuf<unsigned>            st_codes;  // 32 row codes per slice
  DevBuf<unsigned>            st_cols;   // solution slot of every entry, slice-interleaved
  DevBuf<double>              st_vals;
  bool                        f32 = false;  // factor values stored in single precision (st_vals32 instead of st_vals)
  DevBuf<float>               st_vals32;
  // warp-stream layout (wsweep.cu): one private segment stream per warp of a persistent CTA per SM
  bool                        ws = false;
  bool                        fused = false;  // L segments followed by U segments: one launch per LDU solve
  unsigned                    ws_grid = 0, ws_warps = 0, ws_stages = 0, ws_window = 0, ws_nslots = 0, ws_nsegs = 0;
  DevBuf<unsigned>            ws_wdesc;   // 8 words per global warp: offset (16 B units), segments, -, -, first 4 sizes
  DevBuf<unsigned>            ws_stream;  // segments
  std::vector<unsigned>       slot_of;    // host: solution slot of every original row (empty: identity)
  std::size_t            slab_bytes = 0, nnz = 0;  // slab_bytes: bytes the sweep streams
};

// one hif::Prec level on the device (reference alg/Prec.hpp:309-323)
struct DevLevel {
  std::size_t m = 0, n = 0, nm = 0;
  SweepPlan   L, U;  // L_B, U_B
  SweepPlan   LU;    // fused: L then U in one launch (wsweep.cu); L and U then only carry slot maps / statistics
  DevCsr      E, F;
  DevBuf<double> d;        // m
  // consumers of the sweeps' renumbered solution slots (wsweep.cu): built once at attach
  DevBuf<double> d_ls;     // d permuted to the slots of the L sweep (the U sweep divides its right-hand side)
  DevBuf<int>    E_xcol;   // E.col mapped to the slots of the U sweep
  // rows of F that have entries (46 % at Poisson 128^3 level 0): g = bhat - F y is formed IN PLACE on those
  DevBuf<unsigned> F_rows, F_cptr;  // row ids; F.ptr at those rows (+ end): entries are those of F.col / F.val
  DevBuf<int>    q_slot;   // q_inv mapped: < nslots(U) -> slot of the U sweep, else nslots + (q_inv - m)
  DevBuf<unsigned> L_slot, U_slot;  // slot of every original row (indirection for the off-path kernels)
  DevBuf<double> s, t;     // n
  DevBuf<double> sp;       // n: s[p[i]] (the gather reads it coalesced: one scattered load per row instead of two)
  DevBuf<int>    p, q_inv; // n
  // triangular-sweep schedule
  int         rows_per_block = 1024;
  std::size_t depthL = 0, depthU = 0;  // dependency depth (number of level sets)
  // per-apply work vectors (nrhs = 1 path); tagged = produced by a sync-free sweep
  DevBuf<double>             bhat;                      // n   s[p]*b[p]
  DevBuf<unsigned long long> xL_dn, xU_dn, xL_up, xU_up;  // m   tagged
  DevBuf<double>             r;                         // nm  Schur rhs = child's b
  DevBuf<double>             ychild;                    // nm  child's solution
  // multi-rhs (kMrhsWidth columns, row-interleaved): plans + work vectors, built on first use
  HostCsr                    hostL, hostU;  // kept for the lazily built multi-rhs plans
  // host copies kept for the transposed twin (LHF_SH / LHF_MH) and the product (LHF_M / LHF_MH)
  HostCsr             hostE, hostF;
  std::vector<double> h_d, h_s, h_t;
  std::vector<int>    h_p, h_pinv, h_q, h_qinv;  // h_pinv / h_q empty when the caller did not give them
  // multilevel product: row-gather CSR of L_B and U_B, gather index and scalings (uploaded on first use)
  DevCsr                     Lcsr, Ucsr;
  DevBuf<int>                q_dev, pinv_dev;
  DevBuf<double>             pw, pw1, pw2, pf;          // n, m, nm, m work vectors of prec_prod
  DevBuf<unsigned long long> p_xL, p_xU;                // tagged results of the product's one LDU solve
  DevBuf<double>             py;                        // n: product of this level (input of the level above)
  SweepPlan                  Lm, Um;
  DevBuf<double>             m_bhat, m_g, m_r, m_ychild;
  DevBuf<unsigned long long> m_xL_dn, m_xU_dn, m_xL_up, m_xU_up;
};

// dense last level: QRCP state (reference small_scale/QRCP.hpp:544-555)
struct DevDense {
  std::size_t    nm = 0, rank = 0;
  DevBuf<double> Q;     // nm x nm column-major explicit Q = H_1 ... H_nm (column k = row k of Q^T)
  DevBuf<double> R;     // nm x nm column-major, upper triangle = R
  DevBuf<double> tinv;  // ceil(nm/32) inverted 32x32 diagonal tiles of R, column-major, zero padded
  DevBuf<int>    jpvt;  // nm, 1-based verbatim
  DevBuf<double> c;     // nm work (Q^T b)
  bool           transposed = false;  // twin handle: solve / multiply with (Q R P^T)^T
  std::vector<double> h_mat, h_tau;    // host copies for the twin
  std::vector<int>    h_jpvt;
};

struct DevMatrix {  // user matrix A in CRS
  std::size_t n = 0, nnz = 0;
  DevCsr      A;
};

struct AsyncIo {  // pipelined host-buffer solves (lhfdGpuSolveAsync, capi.cu)
  cudaStream_t   h2d = nullptr, d2h = nullptr;
  DevBuf<double> b[2], x[2];
  cudaEvent_t    copied_in[2] = {nullptr, nullptr}, applied[2] = {nullptr, nullptr}, copied_out[2] = {nullptr, nullptr};
  std::size_t    count = 0;
};

struct ApplyGraph {  // one captured apply (apply.cu)
  const double *  b;
  double *        x;
  std::size_t     rank;
  unsigned        parity;
  bool            nsp_on;
  std::size_t     nsp_start, nsp_end;
  unsigned        uses;  // uses at short intervals (capture on the third)
  cudaGraphExec_t exec;
  std::size_t     launches;
  unsigned        last_epoch;
};

struct Handle {
  int                   device = 0, num_sms = 148;
  std::vector<ApplyGraph> graphs;
  AsyncIo                 aio;
  bool                    graphs_off = false;  // the handle's stream can not be captured
  std::vector<DevLevel> levels;
  DevDense              dense;
  DevMatrix             A;
  bool                  has_A = false;
  bool                  nsp_on = false;
  std::size_t           nsp_start = 0, nsp_end = 0;
  // filter of the TRANSPOSED solve (hif::HIF::nsp_tran, builder.hpp:421-422): lives on the primary
  // handle, copied to the twin before every transposed solve
  bool                  nspt_on = false;
  std::size_t           nspt_start = 0, nspt_end = 0;
  cudaStream_t          own_stream = nullptr, stream = nullptr;
  unsigned              epoch = 0;        // apply counter; parity tags the sync-free buffers
  unsigned              epoch_m = 0;      // same for the multi-rhs work vectors
  unsigned              epoch_p = 0;      // same for the product's LDU solve
  Handle *              twin = nullptr;   // transposed preconditioner (built on first LHF_SH / LHF_MH)
  bool                  is_twin = false, prod_ready = false;
  bool                  f32 = false;      // attached to single-precision factors (lhfsGpuAttachLevels): the
                                          // streamed sweep values are stored as float, arithmetic stays double
  // host copy of the user matrix (for the twin's A^T)
  std::vector<LhfIndPtr> hA_ptr;
  std::vector<LhfInt>    hA_idx;
  std::vector<double>    hA_val;
  bool                   hA_rowmajor = true;
  // per sweep of an apply: a ticket counter + the level-completion counters of stream.cu
  // (tick_stride ints per sweep, zeroed once per apply)
  DevBuf<int>           tickets;
  std::size_t           tick_stride = 1;
  int *                 tick(std::size_t sweep) const { return tickets.p + sweep * tick_stride; }
  DevBuf<int>           error_flag;       // set by a sweep whose spin limit tripped
  int *                 h_error = nullptr;  // pinned mirror
  // scratch for host-buffer entry points / IR / Krylov
  DevBuf<double> io_b, io_x;
  DevBuf<float>  io_f;  // staging of single-precision caller vectors (lhfsGpuSolve / lhfsGpuApply)
  std::size_t    io_cols = 0;
  DevBuf<double> ir_xk, ir_r, ir_t;
  DevBuf<double> kr_v, kr_w, kr_Q, kr_Z, kr_scal, kr_part;
  DevBuf<unsigned> kr_count;        // arrival counter of the fused Gram-Schmidt step (krylov.cu)
  // persistent Gram-Schmidt kernel (krylov.cu): block partials of every step, grid barrier counter (only ever
  // incremented: a launch with B barriers adds B * grid; the host keeps the value it starts from)
  DevBuf<double>             kr_mpart;
  DevBuf<unsigned long long> kr_bar;
  unsigned long long         kr_bar_base = 0;
  bool                       kr_no_coop  = false;  // the cooperative launch was refused once: per-step kernels from then on
  // block Krylov (krylov.cu): bases [restart][n][nrhs] (Z: FGMRES only), [n][nrhs] work blocks, per-column
  // scalars (Hessenberg column [restart+1][nrhs], y [restart][nrhs], norms), block partials, retired-column mask
  DevBuf<double>   kb_Q, kb_Z, kb_v, kb_w, kb_r, kb_t, kb_H, kb_y, kb_red, kb_part;
  DevBuf<int>      kb_mask;
  DevBuf<unsigned> kb_count;  // arrival counter of mgs_step_cols_kernel
  double *       h_scal = nullptr;  // pinned
  int            kr_restart = 0;
  // multi-rhs column staging
  DevBuf<double> mr_b, mr_x, mr_c;
  bool           mrhs_ready = false;
  std::size_t    wide_nc = 0;         // row stride (columns) the multi-rhs work vectors are laid out for
  std::size_t    wide_cap = 0;        // columns they can hold
  // statistics
  std::size_t bytes_factors = 0, bytes_vec = 0, bytes_dense = 0, device_bytes = 0, nnz_total = 0;
  std::size_t kernels_per_apply = 0, launch_count = 0;
  // debug: one triangular sweep on its own (lhfdGpuDebugSweepDev), per (level, factor) tagged scratch with its
  // own epoch counter -- every tagged buffer is written exactly once per epoch, as the apply's are
  struct DebugSweep {
    DevBuf<unsigned long long> x1, x2, rhs;  // results (fused plan: L in x1, U in x2); tagged input of a U sweep
    DevBuf<double>             b;            // plain right-hand side of an L / fused sweep
    DevBuf<int>                sync;
    unsigned                   epoch = 0;
  };
  std::vector<DebugSweep> dbg_sweeps;  // 3 per level: L, U, fused LU
  // debug: per-segment trace of one warp-stream sweep (lhfdGpuDebugTraceSweep)
  int                        trace_level = -1, trace_which = -1;
  DevBuf<unsigned long long> trace_buf;
  // optional per-kernel timing of one apply (lhfdGpuProfileSolveDev)
  bool                                  profiling = false;
  std::vector<std::pair<std::string, cudaEvent_t>> prof_marks;
  std::size_t n0() const { return levels.empty() ? 0 : levels[0].n; }
};

// ---- attach.cu
Handle *attach_levels(int device, std::size_t nlevels, const LhfdGpuLevel *levels, bool dense_transposed = false,
                      bool f32 = false);
Handle *ensure_twin(Handle *h);   // transposed preconditioner sharing the stream of h
void    destroy_handle(Handle *h);
void    set_matrix(Handle *h, bool rowmajor, std::size_t n, const LhfIndPtr *indptr, const LhfInt *indices,
                   const double *vals);
HostCsr ccs_to_csr(const LhfdGpuCcs &c, const char *name);

// ---- sweep.cu : plan construction / launch dispatch of the triangular sweeps
// kind: 2 = warp streams (wsweep.cu), 1 = round-1 streaming kernel (stream.cu), -1 = HIFIR_B200_SWEEP
// nsm = SMs of the device the plan is built for; rhs_index (nullable) = position of original row r in
// the sweep's right-hand side array (the U sweep reads the L sweep's result at the L plan's slots)
void build_sweep_plan(const HostCsr &T, bool upper, SweepPlan &plan, std::size_t *tally, unsigned nsm,
                      const unsigned *rhs_index = nullptr, int kind = -1);
void sweep_host_emulate(const HostCsr &T, bool upper, const double *rhs, const double *diag, double *x,
                        std::size_t stats[4], bool f32 = false, int parity = -1);
void launch_sweep(Handle *h, const SweepPlan &plan, const double *rhs_plain, const unsigned long long *rhs_tagged,
                  const double *diag, unsigned long long *x, unsigned parity, int *sync,
                  unsigned nr = 0, unsigned long long *trace = nullptr);  // nr = 0: the plan's own width
// ---- stream.cu
void build_stream_plan(const HostCsr &S, bool upper, SweepPlan &plan, std::size_t *tally);
void stream_host_emulate(const HostCsr &S, bool upper, const double *rhs, const double *diag, double *x,
                         std::size_t stats[4], bool f32 = false, int parity = -1);
// the emulation of a streaming plan on the arrays copied back from the device; x: 2 m entries
void stream_emulate_device_plan(const SweepPlan &plan, const double *rhs, const double *diag, double *x, unsigned parity);
void launch_stream_sweep(Handle *h, const SweepPlan &plan, const double *rhs_plain,
                         const unsigned long long *rhs_tagged, const double *diag, unsigned long long *x,
                         unsigned parity, int *ticket, unsigned long long *trace = nullptr, unsigned nr = 1);

// ---- apply.cu : the multilevel M^{-1} apply on device vectors
void apply_dev(Handle *h, const double *d_b, double *d_x, std::size_t rank);
void clear_apply_graphs(Handle *h);
void reset_tagged_state(Handle *h);
void check_sweep_error(Handle *h);  // synchronizes; throws if a sweep tripped its spin limit

void dense_solve_dev(Handle *h, const double *d_in, double *d_out, std::size_t rank);     // QRCP::solve
void dense_multiply_dev(Handle *h, const double *d_in, double *d_out, std::size_t rank);  // QRCP::multiply
void launch_ldu_solve(Handle *h, DevLevel &D, const double *rhs, unsigned long long *xL, unsigned long long *xU,
                      unsigned parity, int *tickets);

// ---- product.cu : y = M x (prec_prod.hpp:54-134)
void prod_dev(Handle *h, const double *d_x, double *d_y, std::size_t rank);

// ---- krylov.cu
void   spmv_dev(Handle *h, const double *d_x, double *d_y);
void   hifir_dev(Handle *h, const double *d_b, std::size_t nirs, double *d_x, std::size_t rank);
void   hifir_betas_dev(Handle *h, const double *d_b, std::size_t nirs, const double *betas, double *d_x,
                       std::size_t rank, long *iters, int *flag);
void   krylov_dev(Handle *h, bool flexible, const double *d_b, int restart, double rtol, int maxit,
                  bool full_rank, double *d_x, int *flag, int *iters, int *num_mv);
double norm2_dev(Handle *h, const double *d_v, std::size_t n);
// the same on row-interleaved blocks of nrhs columns (nrhs == 1: the single-rhs functions above)
void   check_krylov_mrhs(Handle *h, std::size_t nrhs, int restart);  // matrix, restart and block size
void   hifir_mrhs_dev(Handle *h, std::size_t nrhs, const double *d_B, std::size_t nirs, double *d_X, std::size_t rank);
void   krylov_mrhs_dev(Handle *h, bool flexible, std::size_t nrhs, const double *d_B, int restart, double rtol, int maxit,
                       bool full_rank, double *d_X, int *flag, int *iters, int *num_mv);

// ---- wsweep.cu : statically scheduled warp-stream sweeps
struct WsHost {  // packed plan on the host
  unsigned                           nwarps = 0, nslots = 0, depth = 0, slices = 0;
  std::vector<unsigned>              wdesc, stream, slot_of;
  std::vector<std::vector<unsigned>> seg_off;                        // per warp: word offsets of its segments (private stream)
  std::size_t                        entries = 0, padded = 0, copy_rows = 0, max_segs = 0, nsegs = 0;
};
void pack_warp_streams(const HostCsr &S, WsHost &H, unsigned nwarps, unsigned window, bool f32,
                       const unsigned *rhs_index, unsigned umin_force = 0);
void ws_finalize_ring(WsHost &H, unsigned stages);
// parity < 0: plain values; 0 / 1: published values carry the readiness tag as on the device (wsweep.cu)
void ws_host_emulate_packed(const WsHost &H, bool upper, bool f32, const double *rhs, const double *diag, double *x,
                            int parity = -1, double *x2 = nullptr);
// the emulation of a warp-stream plan on the bytes copied back from the device (x2: U results of a fused plan)
void ws_emulate_device_plan(const SweepPlan &plan, const double *rhs, const double *diag, double *x, double *x2,
                            unsigned parity);
void build_ws_plan(const HostCsr &S, bool upper, SweepPlan &plan, std::size_t *tally, unsigned nsm,
                   const unsigned *rhs_index, unsigned warps = 0, unsigned stages = 0);  // 0: HIFIR_B200_WS_WARPS / _STAGES
void launch_ws_sweep_cols(Handle *h, const SweepPlan &plan, const double *rhs_plain, const double *diag, unsigned long long *xL,
                          unsigned long long *xU, unsigned parity, int *sync, unsigned nc);  // fused plan, nc = 16 | 32 | 64
void ws_host_emulate(const HostCsr &S, bool upper, const double *rhs, const double *diag, double *x_by_row,
                     std::size_t stats[4], bool f32, int parity = -1);
void launch_ws_sweep(Handle *h, const SweepPlan &plan, const double *rhs_plain, const unsigned long long *rhs_tagged,
                     const double *diag, unsigned long long *x, unsigned parity, int *sync,
                     unsigned long long *trace = nullptr, unsigned long long *x2 = nullptr);
void build_ws_ldu_plan(const HostCsr &SL, const HostCsr &SU, SweepPlan &plan, SweepPlan &L, SweepPlan &U, std::size_t *tally,
                       unsigned nsm);
void ws_debug_graph(const HostCsr &S, unsigned nsm, std::vector<unsigned> &dep_ptr, std::vector<unsigned> &dep_idx);
int  sweep_kind();  // HIFIR_B200_SWEEP = ws (default) | stream | slab  ->  2 | 1 | 0

// ---- planlab.cu (developer tool, host only)
void plan_lab(const HostCsr &Tnat, bool upper, const int *user_key, const double *opts, double *out);

// ---- mrhs.cu
void apply_mrhs_dev(Handle *h, std::size_t nrhs, const double *d_B, double *d_X, std::size_t rank);

}  // namespace hifgpu
