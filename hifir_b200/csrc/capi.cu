// capi.cu -- the C-ABI of include/hifir_b200.h.  Exceptions never cross this boundary:
// they become LhfStatus + a thread-local message (cf. libhifir.cpp:45-53, 224-229).
#include <cstring>
#include <memory>
#include <new>

#include "debug_api.h"
#include "hifgpu.h"

using namespace hifgpu;

namespace {

thread_local std::string g_msg;

// Every entry point selects the handle's device; the caller's current device is restored on the way
// out (a single-process multi-GPU host -- PETSc, torch -- must not find itself on another device).
struct DeviceGuard {
  int  prev = -1;
  bool ok;
  DeviceGuard() : ok(cudaGetDevice(&prev) == cudaSuccess) {
    if (!ok) cudaGetLastError();  // no device at all: the host-only entry points still work
  }
  ~DeviceGuard() {
    if (ok) cudaSetDevice(prev);
  }
};

template <class F>
LhfStatus guarded(F &&f) {
  DeviceGuard guard;
  try {
    f();
    return LHF_SUCCESS;
  } catch (const std::length_error &e) {
    g_msg = e.what();
    return LHF_MISMATCHED_SIZES;
  } catch (const std::invalid_argument &e) {
    g_msg = e.what();
    return LHF_BAD_PREC;
  } catch (const std::logic_error &e) {
    g_msg = e.what();
    return LHF_BAD_PREC;
  } catch (const std::exception &e) {
    g_msg = e.what();
    return LHF_HIFIR_ERROR;
  } catch (...) {
    g_msg = "unknown error";
    return LHF_HIFIR_ERROR;
  }
}

Handle *H(LhfdGpuHdl hdl) { return reinterpret_cast<Handle *>(hdl); }

#define REQUIRE_HANDLE(hdl)                 \
  if (!(hdl)) {                             \
    g_msg = "NULL device-backend handle";   \
    return LHF_NULL_OBJ;                    \
  }
#define REQUIRE_PTR(p, what)                \
  if (!(p)) {                               \
    g_msg = "NULL pointer: " what;          \
    return LHF_NULL_OBJ;                    \
  }

void ensure_io(Handle *h, std::size_t cols) {
  const std::size_t need = h->n0() * cols;
  if (h->io_b.n < need) {
    h->io_b.alloc(need, &h->device_bytes);
    h->io_x.alloc(need, &h->device_bytes);
  }
}

// host <-> device copies of the hot path: asynchronous on the handle's stream; pinned
// caller memory is transferred by DMA directly, pageable memory is staged by the driver
void h2d(Handle *h, double *dst, const double *src, std::size_t count) {
  HIF_CUDA(cudaMemcpyAsync(dst, src, count * sizeof(double), cudaMemcpyHostToDevice, h->stream));
}
void d2h(Handle *h, double *dst, const double *src, std::size_t count) {
  HIF_CUDA(cudaMemcpyAsync(dst, src, count * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
}

// single-precision caller vectors (lhfsGpuSolve / lhfsGpuApply): half the PCIe bytes, widened /
// narrowed on the device; the apply itself works on double vectors
__global__ void widen_kernel(const float *__restrict__ in, double *__restrict__ out, std::size_t n) {
  for (std::size_t i = blockIdx.x * static_cast<std::size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<std::size_t>(gridDim.x) * blockDim.x)
    out[i] = static_cast<double>(in[i]);
}
__global__ void narrow_kernel(const double *__restrict__ in, float *__restrict__ out, std::size_t n) {
  for (std::size_t i = blockIdx.x * static_cast<std::size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<std::size_t>(gridDim.x) * blockDim.x)
    out[i] = static_cast<float>(in[i]);
}
unsigned cast_grid(std::size_t n) {
  return static_cast<unsigned>(std::min<std::size_t>((n + 255) / 256, static_cast<std::size_t>(kNumSMs) * 8u));
}
void h2d(Handle *h, double *dst, const float *src, std::size_t count) {
  if (h->io_f.n < count) h->io_f.alloc(count, &h->device_bytes);
  HIF_CUDA(cudaMemcpyAsync(h->io_f.p, src, count * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  if (count) widen_kernel<<<cast_grid(count), 256, 0, h->stream>>>(h->io_f.p, dst, count);
  HIF_KERNEL_CHECK();
  ++h->launch_count;
}
void d2h(Handle *h, float *dst, const double *src, std::size_t count) {
  if (h->io_f.n < count) h->io_f.alloc(count, &h->device_bytes);
  if (count) narrow_kernel<<<cast_grid(count), 256, 0, h->stream>>>(src, h->io_f.p, count);
  HIF_KERNEL_CHECK();
  ++h->launch_count;
  HIF_CUDA(cudaMemcpyAsync(dst, h->io_f.p, count * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
}

Handle *H(LhfsGpuHdl hdl) { return reinterpret_cast<Handle *>(hdl); }

// lhfdGpuSolveAsync: host-buffer solves as a three-stage pipeline.  Two staging slots; the copies
// run on their own streams, ordered against the apply by events, so that H2D(k+1), apply(k) and
// D2H(k-1) overlap.  The apply of slot s always sees the same device pointers: its CUDA graph is
// captured once.
void solve_host_async(Handle *h, const double *b, double *x) {
  HIF_CUDA(cudaSetDevice(h->device));
  const std::size_t n = h->n0();
  AsyncIo &         A = h->aio;
  if (!A.h2d) {
    HIF_CUDA(cudaStreamCreateWithFlags(&A.h2d, cudaStreamNonBlocking));
    HIF_CUDA(cudaStreamCreateWithFlags(&A.d2h, cudaStreamNonBlocking));
    for (int s = 0; s < 2; ++s) {
      A.b[s].alloc(n, &h->device_bytes);
      A.x[s].alloc(n, &h->device_bytes);
      HIF_CUDA(cudaEventCreateWithFlags(&A.copied_in[s], cudaEventDisableTiming));
      HIF_CUDA(cudaEventCreateWithFlags(&A.applied[s], cudaEventDisableTiming));
      HIF_CUDA(cudaEventCreateWithFlags(&A.copied_out[s], cudaEventDisableTiming));
    }
  }
  const int s = static_cast<int>(A.count++ & 1u);
  if (A.count > 2) {
    HIF_CUDA(cudaStreamWaitEvent(A.h2d, A.applied[s], 0));  // the previous apply of this slot has consumed b[s]
  }
  HIF_CUDA(cudaMemcpyAsync(A.b[s].p, b, n * sizeof(double), cudaMemcpyHostToDevice, A.h2d));
  HIF_CUDA(cudaEventRecord(A.copied_in[s], A.h2d));
  HIF_CUDA(cudaStreamWaitEvent(h->stream, A.copied_in[s], 0));
  if (A.count > 2) HIF_CUDA(cudaStreamWaitEvent(h->stream, A.copied_out[s], 0));  // x[s] has left the device
  apply_dev(h, A.b[s].p, A.x[s].p, 0);
  HIF_CUDA(cudaEventRecord(A.applied[s], h->stream));
  HIF_CUDA(cudaStreamWaitEvent(A.d2h, A.applied[s], 0));
  HIF_CUDA(cudaMemcpyAsync(x, A.x[s].p, n * sizeof(double), cudaMemcpyDeviceToHost, A.d2h));
  HIF_CUDA(cudaEventRecord(A.copied_out[s], A.d2h));
}
void wait_host_async(Handle *h) {
  AsyncIo &A = h->aio;
  if (A.h2d) {
    HIF_CUDA(cudaStreamSynchronize(A.h2d));
    HIF_CUDA(cudaStreamSynchronize(h->stream));
    HIF_CUDA(cudaStreamSynchronize(A.d2h));
  }
}

// lhf?Solve (libhifir.cpp:151-158): IO = the caller's vector type
template <class IO>
void solve_host(Handle *h, const IO *b, IO *x) {
  HIF_CUDA(cudaSetDevice(h->device));
  ensure_io(h, 1);
  h2d(h, h->io_b.p, b, h->n0());
  apply_dev(h, h->io_b.p, h->io_x.p, 0);  // lhfdSolve: M->solve(b, x), rank defaults to 0
  d2h(h, x, h->io_x.p, h->n0());
  check_sweep_error(h);
}

// The handle that serves `op` (libhifir.cpp:447-472): the transposed twin for S^H / M^H, with the
// filter hif::HIF::solve applies in that orientation -- nsp for the plain solve, nsp_tran for the
// transposed one (builder.hpp:419-422) -- shared by the host- and the device-pointer entry points.
Handle *handle_for_op(Handle *h0, LhfOperationType op) {
  if (op != LHF_S && op != LHF_SH && op != LHF_M && op != LHF_MH) throw std::logic_error("unknown operation");
  if (op == LHF_S || op == LHF_M) return h0;
  Handle *t    = ensure_twin(h0);
  t->stream    = h0->stream;
  t->nsp_on    = h0->nspt_on;
  t->nsp_start = h0->nspt_start;
  t->nsp_end   = h0->nspt_end;
  return t;
}

// lhf?Apply (libhifir.cpp:447-472; lhfsdApply :1192-1218): IO = the caller's vector type
template <class IO>
void apply_host(Handle *h0, LhfOperationType op, const IO *b, int nirs, const double *betas, int rank, IO *x,
                int *ir_status) {
  HIF_CUDA(cudaSetDevice(h0->device));
  Handle *h = handle_for_op(h0, op);  // the transposed twin serves S^H and M^H with the kernels of S and M
  if (op == LHF_M || op == LHF_MH) {  // libhifir.cpp:458-459: mmultiply(b, x, trans), numerical rank
    ensure_io(h0, 1);
    h2d(h0, h0->io_b.p, b, h0->n0());
    prod_dev(h, h0->io_b.p, h0->io_x.p, 0);
    d2h(h0, x, h0->io_x.p, h0->n0());
    check_sweep_error(h);
    return;
  }
  // rank defaulting rule, libhifir.cpp:451-455
  const std::size_t rnk = rank == LHF_DEFAULT_RANK ? (nirs > 1 ? static_cast<std::size_t>(-1) : 0)
                                                   : static_cast<std::size_t>(static_cast<long long>(rank));
  ensure_io(h0, 1);
  h2d(h0, h0->io_b.p, b, h0->n0());
  if (h != h0) {
    if (h->io_b.n < h0->n0()) {  // the twin works on the primary handle's staging buffers
      h->io_b.release();
      h->io_x.release();
    }
  }
  double *io_b = h0->io_b.p, *io_x = h0->io_x.p;
  if (nirs <= 1) {
    apply_dev(h, io_b, io_x, 0);  // plain solve ignores `rank` (libhifir.cpp:461)
  } else if (!betas) {
    hifir_dev(h, io_b, static_cast<std::size_t>(nirs), io_x, rnk);
  } else {
    long iters = 0;
    int  flag  = 0;
    hifir_betas_dev(h, io_b, static_cast<std::size_t>(nirs), betas, io_x, rnk, &iters, &flag);
    if (ir_status) {
      ir_status[0] = static_cast<int>(iters);
      ir_status[1] = flag;
    }
  }
  d2h(h0, x, io_x, h0->n0());
  check_sweep_error(h);
}

// widen the description of a single-precision preconditioner (hif::HIF<float>): integers verbatim,
// values float -> double (exact).  The widened arrays live until attach_levels returns.
struct WidenedLevels {
  std::vector<LhfdGpuLevel>        lv;
  std::vector<std::vector<double>> keep;
  const double *widen(const float *p, std::size_t n) {
    if (!p) return nullptr;
    keep.emplace_back(p, p + n);
    return keep.back().data();
  }
  LhfdGpuCcs widen(const LhfsGpuCcs &c) {
    LhfdGpuCcs d;
    d.nrows     = c.nrows;
    d.ncols     = c.ncols;
    d.col_start = c.col_start;
    d.row_ind   = c.row_ind;
    const LhfIndPtr nnz = (c.col_start && c.ncols) ? c.col_start[c.ncols] : 0;
    if (nnz < 0) throw std::invalid_argument("negative nonzero count in a factor block");
    if (nnz && !c.vals) throw std::invalid_argument("null value array in a factor block");
    d.vals = widen(c.vals, static_cast<std::size_t>(nnz));
    return d;
  }
  WidenedLevels(std::size_t nlevels, const LhfsGpuLevel *s) : lv(nlevels) {
    keep.reserve(12 * nlevels);
    for (std::size_t l = 0; l < nlevels; ++l) {
      const LhfsGpuLevel &S = s[l];
      LhfdGpuLevel &      D = lv[l];
      std::memset(&D, 0, sizeof(D));
      D.m = S.m, D.n = S.n;
      D.L_B = widen(S.L_B), D.U_B = widen(S.U_B), D.E = widen(S.E), D.F = widen(S.F);
      D.d_B = widen(S.d_B, S.m), D.s = widen(S.s, S.n), D.t = widen(S.t, S.n);
      D.p = S.p, D.p_inv = S.p_inv, D.q = S.q, D.q_inv = S.q_inv;
      D.dense_n = S.dense_n, D.dense_rank = S.dense_rank;
      D.qr_mat  = widen(S.qr_mat, S.dense_n * S.dense_n);
      D.qr_tau  = widen(S.qr_tau, S.dense_n);
      D.qr_jpvt = S.qr_jpvt;
      D.has_symm_dense = S.has_symm_dense;
    }
  }
};

}  // namespace

extern "C" {

const char *lhfGpuGetErrorMsg(void) { return g_msg.c_str(); }
const char *lhfGpuVersion(void) { return "hifir_b200 0.1.0 (sm_100a)"; }

LhfStatus lhfdGpuAttachLevels(int device, size_t nlevels, const LhfdGpuLevel *levels, LhfdGpuHdl *out) {
  REQUIRE_PTR(out, "out");
  *out = nullptr;
  REQUIRE_PTR(levels, "levels");
  return guarded([&] { *out = reinterpret_cast<LhfdGpuHdl>(attach_levels(device, nlevels, levels)); });
}

LhfStatus lhfdGpuDestroy(LhfdGpuHdl hdl) {
  REQUIRE_HANDLE(hdl);
  return guarded([&] { destroy_handle(H(hdl)); });
}

LhfStatus lhfdGpuSetMatrix(LhfdGpuHdl hdl, int is_rowmajor, size_t n, const LhfIndPtr *indptr,
                           const LhfInt *indices, const double *vals) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(indptr, "indptr");
  return guarded([&] { set_matrix(H(hdl), is_rowmajor != 0, n, indptr, indices, vals); });
}

LhfStatus lhfdGpuSetNspConst(LhfdGpuHdl hdl, size_t start, size_t end) {
  REQUIRE_HANDLE(hdl);
  return guarded([&] {
    Handle *          h = H(hdl);
    const std::size_t n = h->n0();
    const std::size_t e = (end == static_cast<std::size_t>(-1) || end < start) ? n : end;
    if (e < start || e > n) throw std::invalid_argument("null-space filter: wrong range (start,end,n)");
    h->nsp_on    = true;
    h->nsp_start = start;
    h->nsp_end   = end;
  });
}

LhfStatus lhfdGpuSetNspTranConst(LhfdGpuHdl hdl, size_t start, size_t end) {
  REQUIRE_HANDLE(hdl);
  return guarded([&] {
    Handle *          h = H(hdl);
    const std::size_t n = h->n0();
    const std::size_t e = (end == static_cast<std::size_t>(-1) || end < start) ? n : end;
    if (e < start || e > n) throw std::invalid_argument("null-space filter: wrong range (start,end,n)");
    h->nspt_on    = true;
    h->nspt_start = start;
    h->nspt_end   = end;
  });
}

LhfStatus lhfdGpuClearNsp(LhfdGpuHdl hdl) {
  REQUIRE_HANDLE(hdl);
  H(hdl)->nsp_on = H(hdl)->nspt_on = false;
  return LHF_SUCCESS;
}

LhfStatus lhfdGpuSetStream(LhfdGpuHdl hdl, void *cuda_stream, int use_own_stream) {
  REQUIRE_HANDLE(hdl);
  return guarded([&] {
    Handle *h = H(hdl);
    HIF_CUDA(cudaSetDevice(h->device));
    HIF_CUDA(cudaStreamSynchronize(h->stream));
    h->stream = use_own_stream ? h->own_stream : static_cast<cudaStream_t>(cuda_stream);
    h->graphs_off = false;  // the new stream may be capturable (apply.cu)
    if (h->twin) h->twin->stream = h->stream, h->twin->graphs_off = false;
  });
}

LhfStatus lhfdGpuSynchronize(LhfdGpuHdl hdl) {
  REQUIRE_HANDLE(hdl);
  return guarded([&] {
    HIF_CUDA(cudaSetDevice(H(hdl)->device));
    wait_host_async(H(hdl));
    check_sweep_error(H(hdl));
  });
}

LhfStatus lhfdGpuSolveAsync(LhfdGpuHdl hdl, const double *b, double *x) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(b, "b");
  REQUIRE_PTR(x, "x");
  return guarded([&] { solve_host_async(H(hdl), b, x); });
}

LhfStatus lhfdGpuSolveDev(LhfdGpuHdl hdl, const double *d_b, double *d_x, size_t rank) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(d_b, "b");
  REQUIRE_PTR(d_x, "x");
  return guarded([&] { apply_dev(H(hdl), d_b, d_x, rank); });
}

LhfStatus lhfdGpuSolveMrhsDev(LhfdGpuHdl hdl, size_t nrhs, const double *d_B, double *d_X, size_t rank) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(d_B, "B");
  REQUIRE_PTR(d_X, "X");
  if (!nrhs) return LHF_SUCCESS;
  return guarded([&] {
    if (H(hdl)->nsp_on) throw std::logic_error("multiple RHS does not support null space filter.");  // builder.hpp:440
    apply_mrhs_dev(H(hdl), nrhs, d_B, d_X, rank);
  });
}

LhfStatus lhfdGpuHifirDev(LhfdGpuHdl hdl, const double *d_b, size_t nirs, double *d_x, size_t rank) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(d_b, "b");
  REQUIRE_PTR(d_x, "x");
  return guarded([&] { hifir_dev(H(hdl), d_b, nirs, d_x, rank); });
}

LhfStatus lhfdGpuSpmvDev(LhfdGpuHdl hdl, const double *d_x, double *d_y) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(d_x, "x");
  REQUIRE_PTR(d_y, "y");
  return guarded([&] { spmv_dev(H(hdl), d_x, d_y); });
}

LhfStatus lhfdGpuSolve(LhfdGpuHdl hdl, const double *b, double *x) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(b, "b");
  REQUIRE_PTR(x, "x");
  return guarded([&] { solve_host(H(hdl), b, x); });
}

LhfStatus lhfdGpuSolveMrhs(LhfdGpuHdl hdl, size_t nrhs, const double *B, double *X) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(B, "B");
  REQUIRE_PTR(X, "X");
  if (!nrhs) return LHF_SUCCESS;
  return guarded([&] {
    Handle *h = H(hdl);
    if (h->nsp_on) throw std::logic_error("multiple RHS does not support null space filter.");  // builder.hpp:440
    HIF_CUDA(cudaSetDevice(h->device));
    ensure_io(h, nrhs);
    h2d(h, h->io_b.p, B, h->n0() * nrhs);
    apply_mrhs_dev(h, nrhs, h->io_b.p, h->io_x.p, 0);
    d2h(h, X, h->io_x.p, h->n0() * nrhs);
    check_sweep_error(h);
  });
}

// libhifir.cpp:447-472
LhfStatus lhfdGpuApply(LhfdGpuHdl hdl, LhfOperationType op, const double *b, int nirs, const double *betas,
                       int rank, double *x, int *ir_status) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(b, "b");
  REQUIRE_PTR(x, "x");
  if (op != LHF_S && op != LHF_SH && op != LHF_M && op != LHF_MH) {
    g_msg = "unknown LhfOperationType";
    return LHF_BAD_PREC;
  }
  return guarded([&] { apply_host(H(hdl), op, b, nirs, betas, rank, x, ir_status); });
}

// ---- single-precision factors (hif::HIF<float>): lhfs* and the mixed lhfsd* of libhifir ----

LhfStatus lhfsGpuAttachLevels(int device, size_t nlevels, const LhfsGpuLevel *levels, LhfsGpuHdl *out) {
  REQUIRE_PTR(out, "out");
  *out = nullptr;
  REQUIRE_PTR(levels, "levels");
  return guarded([&] {
    if (!nlevels) throw std::invalid_argument("empty preconditioner (no levels)");
    WidenedLevels W(nlevels, levels);
    *out = reinterpret_cast<LhfsGpuHdl>(attach_levels(device, nlevels, W.lv.data(), false, true));
  });
}

LhfStatus lhfsGpuDestroy(LhfsGpuHdl hdl) {
  REQUIRE_HANDLE(hdl);
  return guarded([&] { destroy_handle(H(hdl)); });
}

LhfdGpuHdl lhfsGpuAsDouble(LhfsGpuHdl hdl) { return reinterpret_cast<LhfdGpuHdl>(hdl); }

LhfStatus lhfsGpuSetMatrix(LhfsGpuHdl hdl, int is_rowmajor, size_t n, const LhfIndPtr *indptr, const LhfInt *indices,
                           const float *vals) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(indptr, "indptr");
  return guarded([&] {
    if (n != H(hdl)->n0()) throw std::length_error("matrix size does not match the preconditioner");
    const LhfIndPtr nnz = indptr[n];
    if (nnz < 0) throw std::invalid_argument("A: negative nonzero count");
    if (nnz && !vals) throw std::invalid_argument("A: null value array");
    std::vector<double> v(vals, vals + nnz);
    set_matrix(H(hdl), is_rowmajor != 0, n, indptr, indices, v.data());
  });
}

LhfStatus lhfsdGpuUpdate(LhfsGpuHdl hdl, int is_rowmajor, size_t n, const LhfIndPtr *indptr, const LhfInt *indices,
                         const double *vals) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(indptr, "indptr");
  return guarded([&] { set_matrix(H(hdl), is_rowmajor != 0, n, indptr, indices, vals); });
}

LhfStatus lhfsGpuSolve(LhfsGpuHdl hdl, const float *b, float *x) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(b, "b");
  REQUIRE_PTR(x, "x");
  return guarded([&] { solve_host(H(hdl), b, x); });
}

LhfStatus lhfsdGpuSolve(LhfsGpuHdl hdl, const double *b, double *x) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(b, "b");
  REQUIRE_PTR(x, "x");
  return guarded([&] { solve_host(H(hdl), b, x); });
}

#define REQUIRE_OP(op)                                                  \
  if (op != LHF_S && op != LHF_SH && op != LHF_M && op != LHF_MH) {   \
    g_msg = "unknown LhfOperationType";                                 \
    return LHF_BAD_PREC;                                                \
  }

LhfStatus lhfsGpuApply(LhfsGpuHdl hdl, LhfOperationType op, const float *b, int nirs, const double *betas, int rank,
                       float *x, int *ir_status) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(b, "b");
  REQUIRE_PTR(x, "x");
  REQUIRE_OP(op);
  return guarded([&] { apply_host(H(hdl), op, b, nirs, betas, rank, x, ir_status); });
}

LhfStatus lhfsdGpuApply(LhfsGpuHdl hdl, LhfOperationType op, const double *b, int nirs, const double *betas, int rank,
                        double *x, int *ir_status) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(b, "b");
  REQUIRE_PTR(x, "x");
  REQUIRE_OP(op);
  return guarded([&] { apply_host(H(hdl), op, b, nirs, betas, rank, x, ir_status); });
}

// device-pointer form of lhfdGpuApply without residual bounds
LhfStatus lhfdGpuApplyDev(LhfdGpuHdl hdl, LhfOperationType op, const double *d_b, int nirs, int rank, double *d_x) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(d_b, "b");
  REQUIRE_PTR(d_x, "x");
  return guarded([&] {
    Handle *h0 = H(hdl);
    HIF_CUDA(cudaSetDevice(h0->device));
    Handle *h = handle_for_op(h0, op);
    const std::size_t rnk = rank == LHF_DEFAULT_RANK ? (((op != LHF_S && op != LHF_SH) || nirs > 1) ? static_cast<std::size_t>(-1) : 0)
                                                     : static_cast<std::size_t>(static_cast<long long>(rank));
    if (op == LHF_M || op == LHF_MH)
      prod_dev(h, d_b, d_x, 0);
    else if (nirs <= 1)
      apply_dev(h, d_b, d_x, 0);
    else
      hifir_dev(h, d_b, static_cast<std::size_t>(nirs), d_x, rnk);
  });
}

static LhfStatus krylov_host(LhfdGpuHdl hdl, bool flexible, const double *b, int restart, double rtol, int maxit,
                             int full_rank, double *x, int *flag, int *iters, int *num_mv) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(b, "b");
  REQUIRE_PTR(x, "x");
  return guarded([&] {
    Handle *h = H(hdl);
    HIF_CUDA(cudaSetDevice(h->device));
    ensure_io(h, 1);
    h2d(h, h->io_b.p, b, h->n0());
    int f = 0, it = 0, nmv = 0;
    krylov_dev(h, flexible, h->io_b.p, restart, rtol, maxit, full_rank != 0, h->io_x.p, &f, &it, &nmv);
    d2h(h, x, h->io_x.p, h->n0());
    check_sweep_error(h);
    if (flag) *flag = f;
    if (iters) *iters = it;
    if (num_mv) *num_mv = nmv;
  });
}

LhfStatus lhfdGpuFgmres(LhfdGpuHdl hdl, const double *b, int restart, double rtol, int maxit, int full_rank,
                        double *x, int *flag, int *iters, int *num_mv) {
  return krylov_host(hdl, true, b, restart, rtol, maxit, full_rank, x, flag, iters, num_mv);
}

LhfStatus lhfdGpuGmres(LhfdGpuHdl hdl, const double *b, int restart, double rtol, int maxit, double *x, int *flag,
                       int *iters) {
  return krylov_host(hdl, false, b, restart, rtol, maxit, 0, x, flag, iters, nullptr);
}

// nrhs independent Krylov solves on one row-interleaved host block (krylov_mrhs_dev); nrhs == 1 is krylov_host
static LhfStatus krylov_mrhs_host(LhfdGpuHdl hdl, bool flexible, size_t nrhs, const double *B, int restart, double rtol,
                                  int maxit, int full_rank, double *X, int *flag, int *iters, int *num_mv) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(B, "B");
  REQUIRE_PTR(X, "X");
  if (!nrhs) return LHF_SUCCESS;
  return guarded([&] {
    Handle *h = H(hdl);
    if (h->nsp_on) throw std::logic_error("multiple RHS does not support null space filter.");  // builder.hpp:440
    HIF_CUDA(cudaSetDevice(h->device));
    check_krylov_mrhs(h, nrhs, restart);  // before the staging buffers are sized for the block
    ensure_io(h, nrhs);
    h2d(h, h->io_b.p, B, h->n0() * nrhs);
    std::vector<int> f(nrhs), it(nrhs), nmv(nrhs);
    krylov_mrhs_dev(h, flexible, nrhs, h->io_b.p, restart, rtol, maxit, full_rank != 0, h->io_x.p, f.data(), it.data(),
                    nmv.data());
    d2h(h, X, h->io_x.p, h->n0() * nrhs);
    check_sweep_error(h);
    if (flag) std::copy(f.begin(), f.end(), flag);
    if (iters) std::copy(it.begin(), it.end(), iters);
    if (num_mv) std::copy(nmv.begin(), nmv.end(), num_mv);
  });
}

LhfStatus lhfdGpuFgmresMrhs(LhfdGpuHdl hdl, size_t nrhs, const double *B, int restart, double rtol, int maxit,
                            int full_rank, double *X, int *flag, int *iters, int *num_mv) {
  return krylov_mrhs_host(hdl, true, nrhs, B, restart, rtol, maxit, full_rank, X, flag, iters, num_mv);
}

LhfStatus lhfdGpuGmresMrhs(LhfdGpuHdl hdl, size_t nrhs, const double *B, int restart, double rtol, int maxit,
                           double *X, int *flag, int *iters) {
  return krylov_mrhs_host(hdl, false, nrhs, B, restart, rtol, maxit, 0, X, flag, iters, nullptr);
}

LhfStatus lhfdGpuHifirMrhsDev(LhfdGpuHdl hdl, size_t nrhs, const double *d_B, size_t nirs, double *d_X, size_t rank) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(d_B, "B");
  REQUIRE_PTR(d_X, "X");
  if (!nrhs) return LHF_SUCCESS;
  return guarded([&] {
    Handle *h = H(hdl);
    if (h->nsp_on) throw std::logic_error("multiple RHS does not support null space filter.");  // builder.hpp:440
    HIF_CUDA(cudaSetDevice(h->device));
    hifir_mrhs_dev(h, nrhs, d_B, nirs, d_X, rank);
  });
}

LhfStatus lhfdGpuProfileSolveDev(LhfdGpuHdl hdl, const double *d_b, double *d_x, size_t rank, size_t max_entries,
                                 float *ms, size_t *count, char *names, size_t names_len) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(d_b, "b");
  REQUIRE_PTR(d_x, "x");
  REQUIRE_PTR(ms, "ms");
  REQUIRE_PTR(count, "count");
  return guarded([&] {
    Handle *h    = H(hdl);
    h->profiling = true;
    h->prof_marks.clear();
    try {
      apply_dev(h, d_b, d_x, rank);
      check_sweep_error(h);
    } catch (...) {
      h->profiling = false;
      throw;
    }
    h->profiling = false;
    std::string all;
    size_t      n = 0;
    for (size_t k = 1; k < h->prof_marks.size(); ++k) {
      float t = 0.f;
      HIF_CUDA(cudaEventElapsedTime(&t, h->prof_marks[k - 1].second, h->prof_marks[k].second));
      if (n < max_entries) {
        ms[n++] = t;
        all += h->prof_marks[k].first + "\n";
      }
    }
    for (auto &m : h->prof_marks) cudaEventDestroy(m.second);
    h->prof_marks.clear();
    *count = n;
    if (names && names_len) {
      std::strncpy(names, all.c_str(), names_len - 1);
      names[names_len - 1] = '\0';
    }
  });
}

LhfStatus lhfdGpuDebugSweepHost(const LhfdGpuCcs *T, int upper, const double *rhs, const double *diag, double *x,
                                size_t stats[4], int parity) {
  REQUIRE_PTR(T, "T");
  REQUIRE_PTR(rhs, "rhs");
  REQUIRE_PTR(x, "x");
  REQUIRE_PTR(stats, "stats");
  return guarded([&] {
    if (upper && !diag) throw std::invalid_argument("upper sweep needs the diagonal");
    HostCsr R = ccs_to_csr(*T, "T");
    R.nrows = R.ncols = T->ncols;
    R.ptr.resize(T->ncols + 1, R.ptr.empty() ? 0u : R.ptr.back());
    sweep_host_emulate(R, upper != 0, rhs, diag, x, stats, false, parity < 0 ? -1 : parity & 1);
  });
}

LhfStatus lhfdGpuDebugMergePlan(const LhfdGpuCcs *T, int upper, double out[8]) {
  REQUIRE_PTR(T, "T");
  REQUIRE_PTR(out, "out");
  return guarded([&] {
    HostCsr R = ccs_to_csr(*T, "T");
    R.nrows = R.ncols = T->ncols;
    R.ptr.resize(T->ncols + 1, R.ptr.empty() ? 0u : R.ptr.back());
    const MergeParams mp = MergeParams::from_env();
    MergeStats        ms;
    const HostCsr     S = merged_sweep_form(R, upper != 0, mp, &ms);
    if (!mp.enabled) {  // the sweep form itself: one step per level set
      std::vector<unsigned> lev(S.nrows, 0u);
      std::size_t           depth = 0;
      for (std::size_t i = 0; i < S.nrows; ++i) {
        unsigned l = 0;
        for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k) l = std::max(l, lev[S.col[k]] + 1u);
        lev[i] = l;
        depth  = std::max<std::size_t>(depth, l + 1u);
      }
      ms.rows = ms.ext_rows = S.nrows, ms.nnz = ms.ext_nnz = S.col.size();
      ms.depth = ms.ext_depth = ms.super_levels = depth;
    }
    const double v[8] = {double(ms.rows),      double(ms.nnz),          double(ms.depth),     double(ms.ext_rows),
                         double(ms.ext_nnz),   double(ms.ext_depth),    double(ms.super_levels), mp.plan_cost(ms)};
    std::copy(v, v + 8, out);
  });
}

LhfStatus lhfdGpuDebugPlanLab(const LhfdGpuCcs *T, int upper, const int *key, const double *opts, double *out) {
  REQUIRE_PTR(T, "T");
  REQUIRE_PTR(opts, "opts");
  REQUIRE_PTR(out, "out");
  return guarded([&] {
    HostCsr R = ccs_to_csr(*T, "T");
    R.nrows = R.ncols = T->ncols;
    R.ptr.resize(T->ncols + 1, R.ptr.empty() ? 0u : R.ptr.back());
    plan_lab(R, upper != 0, key, opts, out);
  });
}

// ---- factor arena files (arena.cu; SURVEY.md 8f rank 3) ----

LhfStatus lhfdGpuSaveLevels(size_t nlevels, const LhfdGpuLevel *levels, int with_plans, const char *path) {
  REQUIRE_PTR(levels, "levels");
  REQUIRE_PTR(path, "path");
  return guarded([&] { save_levels_file(path, nlevels, levels, false, with_plans != 0); });
}

LhfStatus lhfsGpuSaveLevels(size_t nlevels, const LhfsGpuLevel *levels, int with_plans, const char *path) {
  REQUIRE_PTR(levels, "levels");
  REQUIRE_PTR(path, "path");
  return guarded([&] {
    if (!nlevels) throw std::invalid_argument("empty preconditioner (no levels)");
    WidenedLevels W(nlevels, levels);
    save_levels_file(path, nlevels, W.lv.data(), true, with_plans != 0);
  });
}

LhfStatus lhfdGpuAttachFile(int device, const char *path, LhfdGpuHdl *out) {
  REQUIRE_PTR(out, "out");
  *out = nullptr;
  REQUIRE_PTR(path, "path");
  return guarded([&] { *out = reinterpret_cast<LhfdGpuHdl>(attach_file(device, path, false)); });
}

LhfStatus lhfsGpuAttachFile(int device, const char *path, LhfsGpuHdl *out) {
  REQUIRE_PTR(out, "out");
  *out = nullptr;
  REQUIRE_PTR(path, "path");
  return guarded([&] { *out = reinterpret_cast<LhfsGpuHdl>(attach_file(device, path, true)); });
}

LhfStatus lhfGpuFileInfo(const char *path, size_t info[8]) {
  REQUIRE_PTR(path, "path");
  REQUIRE_PTR(info, "info");
  return guarded([&] {
    ArenaFile A;
    A.load(path, true);  // reads everything: validates the checksum as well
    std::size_t plan_nnz = 0, plan_depth = 0;
    for (const MergedFactor &mf : A.plans.f) plan_nnz += mf.S.col.size(), plan_depth += mf.st.ext_depth;
    info[0] = 1, info[1] = A.f32, info[2] = A.lv.size(), info[3] = A.lv[0].n, info[4] = A.nnz_total;
    info[5] = A.has_plans, info[6] = plan_nnz, info[7] = plan_depth;
  });
}

// host-only: the sweep of lhfdGpuDebugSweepHost on factor (level, upper) of an arena file, using the
// plan stored in the file when it has one -- lets the CPU tests check that a stored plan reproduces
// what the attach-time analysis computes
LhfStatus lhfGpuDebugFileSweepHost(const char *path, size_t level, int upper, const double *rhs, double *x,
                                   size_t stats[4]) {
  REQUIRE_PTR(path, "path");
  REQUIRE_PTR(rhs, "rhs");
  REQUIRE_PTR(x, "x");
  REQUIRE_PTR(stats, "stats");
  return guarded([&] {
    ArenaFile A;
    A.load(path, true);
    if (level >= A.lv.size()) throw std::invalid_argument("no such level in the arena file");
    const LhfdGpuLevel &P = A.lv[level];
    HostCsr             R = ccs_to_csr(upper ? P.U_B : P.L_B, "T");
    R.nrows = R.ncols = P.m;
    R.ptr.resize(P.m + 1, R.ptr.empty() ? 0u : R.ptr.back());
    struct Scope {
      explicit Scope(PlanCache *p) { tls_plan_cache = p; }
      ~Scope() { tls_plan_cache = nullptr; }
    } scope(A.has_plans ? &A.plans : nullptr);
    A.plans.next = 2 * level + (upper ? 1 : 0);
    sweep_host_emulate(R, upper != 0, rhs, P.d_B, x, stats, A.f32);
  });
}

// single-precision factor block: widened, merged and packed as at attach, packed values rounded to
// float (what the device streams), emulated on the host in double
LhfStatus lhfsGpuDebugSweepHost(const LhfsGpuCcs *T, int upper, const double *rhs, const double *diag, double *x,
                                size_t stats[4], int parity) {
  REQUIRE_PTR(T, "T");
  REQUIRE_PTR(rhs, "rhs");
  REQUIRE_PTR(x, "x");
  REQUIRE_PTR(stats, "stats");
  return guarded([&] {
    if (upper && !diag) throw std::invalid_argument("upper sweep needs the diagonal");
    const LhfIndPtr     nnz = (T->col_start && T->ncols) ? T->col_start[T->ncols] : 0;
    std::vector<double> wide(T->vals, T->vals + (nnz > 0 ? nnz : 0));
    const LhfdGpuCcs    Td{T->nrows, T->ncols, T->col_start, T->row_ind, wide.data()};
    HostCsr             R = ccs_to_csr(Td, "T");
    R.nrows = R.ncols = T->ncols;
    R.ptr.resize(T->ncols + 1, R.ptr.empty() ? 0u : R.ptr.back());
    sweep_host_emulate(R, upper != 0, rhs, diag, x, stats, true, parity < 0 ? -1 : parity & 1);
  });
}

LhfStatus lhfdGpuDebugSegmentGraph(const LhfdGpuCcs *T, int upper, size_t max_segs, size_t max_deps, unsigned *dep_ptr,
                                   unsigned *dep_idx, size_t *nsegs) {
  REQUIRE_PTR(T, "T");
  REQUIRE_PTR(nsegs, "nsegs");
  return guarded([&] {
    HostCsr R = ccs_to_csr(*T, "T");
    R.nrows = R.ncols = T->ncols;
    R.ptr.resize(T->ncols + 1, R.ptr.empty() ? 0u : R.ptr.back());
    const MergeParams mp = MergeParams::from_env();
    MergeStats        ms;
    HostCsr           S = merged_sweep_form(R, upper != 0, mp, &ms);
    std::vector<unsigned> dp, di;
    ws_debug_graph(S, 148u, dp, di);
    if (dp.size() - 1 > max_segs || di.size() > max_deps) throw std::length_error("segment graph exceeds the output buffers");
    std::copy(dp.begin(), dp.end(), dep_ptr);
    std::copy(di.begin(), di.end(), dep_idx);
    *nsegs = dp.size() - 1;
  });
}

LhfStatus lhfdGpuDebugTraceSweep(LhfdGpuHdl hdl, const double *d_b, double *d_x, int level, int which,
                                 unsigned long long *out, size_t max_segs, size_t *nsegs) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(out, "out");
  REQUIRE_PTR(nsegs, "nsegs");
  return guarded([&] {
    Handle *h = H(hdl);
    if (level < 0 || static_cast<size_t>(level) >= h->levels.size() || which < 0 || which > 3)
      throw std::invalid_argument("bad level / sweep selector");
    const SweepPlan &plan = (which & 1) ? h->levels[level].U : h->levels[level].L;
    if (!plan.ws) throw std::invalid_argument("tracing is implemented for the warp-stream sweeps");
    if (h->trace_buf.n < 4ull * plan.ws_nsegs) h->trace_buf.alloc(4ull * plan.ws_nsegs);
    HIF_CUDA(cudaMemsetAsync(h->trace_buf.p, 0, h->trace_buf.n * 8, h->stream));
    h->trace_level = level;
    h->trace_which = which;
    try {
      apply_dev(h, d_b, d_x, 0);
      check_sweep_error(h);
    } catch (...) {
      h->trace_level = h->trace_which = -1;
      throw;
    }
    h->trace_level = h->trace_which = -1;
    const size_t ns = std::min<size_t>(plan.ws_nsegs, max_segs);
    HIF_CUDA(cudaMemcpy(out, h->trace_buf.p, ns * 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    *nsegs = ns;
  });
}

LhfStatus lhfdGpuDebugSweepDev(LhfdGpuHdl hdl, int transposed, size_t level, int which, const double *rhs, double *x,
                               unsigned long long *words, unsigned long long *emul, size_t cap, size_t *nwords,
                               unsigned *slot_of, unsigned *parity) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(rhs, "rhs");
  REQUIRE_PTR(x, "x");
  REQUIRE_PTR(words, "words");
  REQUIRE_PTR(emul, "emul");
  REQUIRE_PTR(nwords, "nwords");
  REQUIRE_PTR(slot_of, "slot_of");
  REQUIRE_PTR(parity, "parity");
  return guarded([&] {
    Handle *h0 = H(hdl);
    HIF_CUDA(cudaSetDevice(h0->device));
    Handle *h = transposed ? handle_for_op(h0, LHF_SH) : h0;
    if (level >= h->levels.size() || which < 0 || which > 2) throw std::invalid_argument("bad level / factor selector");
    DevLevel &       D     = h->levels[level];
    const bool       fused = which == 2;
    const SweepPlan &plan  = fused ? D.LU : which == 1 ? D.U : D.L;
    if (!plan.nblocks) throw std::invalid_argument("the handle launches no sweep of this factor (fused plans: which = 2)");
    const std::size_t m = D.m, ns = 2 * m;  // every slot number is below 2 m (auxiliary unknowns: [m, 2 m))
    if (cap < (fused ? 2 : 1) * ns) throw std::length_error("word buffers of 2 m entries (fused plan: 4 m) needed");
    if (h->dbg_sweeps.size() < 3 * h->levels.size()) h->dbg_sweeps.resize(3 * h->levels.size());
    Handle::DebugSweep &S = h->dbg_sweeps[3 * level + which];
    if (!S.x1.p) {  // zeroed at allocation; the first call runs with parity 1, so the zeros never read as ready
      S.x1.alloc(ns), S.x2.alloc(ns), S.rhs.alloc(ns), S.b.alloc(m), S.sync.alloc(h->tick_stride);
      S.epoch = 0;
    }
    const unsigned par = ++S.epoch & 1u;
    // what the sweep reads: b in original row order (L, fused), or the tagged input of a U sweep at the slots of
    // the L plan (there the L sweep's result lives), divided by d permuted to the same slots
    std::vector<double> rt(ns, tag_set_host(0.0, par)), dls(D.d_ls.n);
    if (which == 1)
      for (std::size_t r = 0; r < m; ++r) rt[D.L.slot_of.empty() ? r : D.L.slot_of[r]] = tag_set_host(rhs[r], par);
    std::vector<double> xw((fused ? 2 : 1) * ns, 0.0), xe((fused ? 2 : 1) * ns, 0.0);
    try {
      HIF_CUDA(cudaMemcpyAsync(S.b.p, rhs, m * sizeof(double), cudaMemcpyHostToDevice, h->stream));
      HIF_CUDA(cudaMemcpyAsync(S.rhs.p, rt.data(), ns * sizeof(double), cudaMemcpyHostToDevice, h->stream));
      HIF_CUDA(cudaMemsetAsync(S.sync.p, 0, S.sync.n * sizeof(int), h->stream));
      // the launch apply_schedule issues for this factor (launch_sweeps, apply.cu)
      if (fused)
        launch_ws_sweep(h, plan, S.b.p, nullptr, D.d_ls.p, S.x1.p, par, S.sync.p, nullptr, S.x2.p);
      else if (which == 0)
        launch_sweep(h, plan, S.b.p, nullptr, nullptr, S.x1.p, par, S.sync.p);
      else
        launch_sweep(h, plan, nullptr, S.rhs.p, D.d_ls.p, S.x1.p, par, S.sync.p);
      check_sweep_error(h);
      HIF_CUDA(cudaMemcpy(xw.data(), S.x1.p, ns * sizeof(double), cudaMemcpyDeviceToHost));
      if (fused) HIF_CUDA(cudaMemcpy(xw.data() + ns, S.x2.p, ns * sizeof(double), cudaMemcpyDeviceToHost));
    } catch (...) {
      S = Handle::DebugSweep();  // slots left unwritten: start over with zeroed buffers on the next call
      throw;
    }
    HIF_CUDA(cudaMemcpy(dls.data(), D.d_ls.p, dls.size() * sizeof(double), cudaMemcpyDeviceToHost));
    const double *ein = which == 1 ? rt.data() : rhs;
    if (plan.ws)
      ws_emulate_device_plan(plan, ein, dls.data(), xe.data(), fused ? xe.data() + ns : nullptr, par);
    else
      stream_emulate_device_plan(plan, ein, dls.data(), xe.data(), par);
    // words: the result buffer(s) in slot order, the fused plan's L buffer first; slot_of: word of every row
    const std::size_t nl = fused ? D.L.ws_nslots : 0, nf = plan.ws ? (fused ? D.U.ws_nslots : plan.ws_nslots) : ns;
    const std::vector<unsigned> &map = which == 0 ? D.L.slot_of : D.U.slot_of;
    for (std::size_t k = 0; k < nl; ++k) std::memcpy(&words[k], &xw[k], 8), std::memcpy(&emul[k], &xe[k], 8);
    for (std::size_t k = 0; k < nf; ++k)
      std::memcpy(&words[nl + k], &xw[(fused ? ns : 0) + k], 8), std::memcpy(&emul[nl + k], &xe[(fused ? ns : 0) + k], 8);
    for (std::size_t r = 0; r < m; ++r) {
      slot_of[r] = static_cast<unsigned>(nl + (map.empty() ? r : map[r]));
      if (fused) slot_of[m + r] = D.L.slot_of[r];
      std::memcpy(&x[r], &words[slot_of[r]], 8);
    }
    *nwords = nl + nf;
    *parity = par;
  });
}

LhfStatus lhfdGpuDebugNorm2Dev(LhfdGpuHdl hdl, const double *d_v, size_t n, double *out) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(d_v, "v");
  REQUIRE_PTR(out, "out");
  return guarded([&] {
    HIF_CUDA(cudaSetDevice(H(hdl)->device));
    *out = norm2_dev(H(hdl), d_v, n);
  });
}

LhfStatus lhfdGpuDebugExportInts(LhfdGpuHdl hdl, size_t level, int which, int *out, size_t max, size_t *count) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(out, "out");
  REQUIRE_PTR(count, "count");
  return guarded([&] {
    Handle *h = H(hdl);
    HIF_CUDA(cudaSetDevice(h->device));
    const void *src = nullptr;
    std::size_t n   = 0;
    if (which == 6) {
      src = h->dense.jpvt.p, n = h->dense.jpvt.n;
    } else {
      if (level >= h->levels.size()) throw std::invalid_argument("no such level");
      const DevLevel &D = h->levels[level];
      switch (which) {
        case 0: src = D.p.p, n = D.p.n; break;
        case 1: src = D.q_inv.p, n = D.q_inv.n; break;
        case 2: src = D.E.ptr.p, n = D.E.ptr.n; break;
        case 3: src = D.E.col.p, n = D.E.col.n; break;
        case 4: src = D.F.ptr.p, n = D.F.ptr.n; break;
        case 5: src = D.F.col.p, n = D.F.col.n; break;
        default: throw std::invalid_argument("bad array selector");
      }
    }
    *count = n;
    HIF_CUDA(cudaStreamSynchronize(h->stream));
    if (n && max) HIF_CUDA(cudaMemcpy(out, src, std::min(n, max) * sizeof(int), cudaMemcpyDeviceToHost));
  });
}

LhfStatus lhfdGpuGetStats(LhfdGpuHdl hdl, size_t stats[]) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(stats, "stats");
  Handle *h                             = H(hdl);
  stats[LHF_GPU_STAT_LEVELS]            = h->levels.size();
  stats[LHF_GPU_STAT_N]                 = h->n0();
  stats[LHF_GPU_STAT_NNZ]               = h->nnz_total;
  stats[LHF_GPU_STAT_DENSE_N]           = h->dense.nm;
  stats[LHF_GPU_STAT_DENSE_RANK]        = h->dense.rank;
  stats[LHF_GPU_STAT_BYTES_FACTORS]     = h->bytes_factors;
  stats[LHF_GPU_STAT_BYTES_VEC_PER_RHS] = h->bytes_vec;
  stats[LHF_GPU_STAT_BYTES_DENSE]       = h->bytes_dense;
  stats[LHF_GPU_STAT_DEVICE_BYTES]      = h->device_bytes;
  stats[LHF_GPU_STAT_KERNELS_PER_APPLY] = h->kernels_per_apply;
  std::size_t depth = 0;
  for (const auto &D : h->levels) depth += (D.nm ? 2 : 1) * (D.depthL + D.depthU);
  stats[LHF_GPU_STAT_DEPTH_TOTAL]  = depth;
  std::size_t dm = 0, sb = 0, se = 0;
  for (const auto &D : h->levels) {
    const std::size_t k = D.nm ? 2 : 1;
    for (const SweepPlan *p : {&D.L, &D.U}) {
      dm += k * p->st_depth;
      sb += k * p->slab_bytes;
    }
    se += k * ((D.L.merge.ext_nnz ? D.L.merge.ext_nnz : D.L.nnz) + (D.U.merge.ext_nnz ? D.U.merge.ext_nnz : D.U.nnz));
  }
  stats[LHF_GPU_STAT_DEPTH_MERGED]  = dm ? dm : depth;
  stats[LHF_GPU_STAT_SWEEP_BYTES]   = sb;
  stats[LHF_GPU_STAT_SWEEP_ENTRIES] = se;
  stats[LHF_GPU_STAT_LAUNCH_COUNT] = h->launch_count;
  return LHF_SUCCESS;
}

LhfStatus lhfdGpuGetDepths(LhfdGpuHdl hdl, size_t nlevels, size_t *depth) {
  REQUIRE_HANDLE(hdl);
  REQUIRE_PTR(depth, "depth");
  Handle *h = H(hdl);
  if (nlevels != h->levels.size()) {
    g_msg = "level count mismatch";
    return LHF_MISMATCHED_SIZES;
  }
  for (std::size_t l = 0; l < nlevels; ++l) {
    depth[2 * l]     = h->levels[l].depthL;
    depth[2 * l + 1] = h->levels[l].depthU;
  }
  return LHF_SUCCESS;
}

}  // extern "C"
