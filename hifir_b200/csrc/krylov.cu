// krylov.cu -- iterative refinement and (F)GMRES around the device apply.
//
// Mirrors reference src/hif/alg/IterRefine.hpp:77-165 (hifir, both variants) and
// examples/advanced/gmres.hpp:18-230 (gmres_hif / fgmres_hifir) with every vector
// operation as a hand-written kernel: CSR SpMV fused with the residual, deterministic
// two-stage warp-shuffle reductions (dot, sum of squares, max-scaled 2-norm of
// utils/math.hpp:83-137), fused modified Gram-Schmidt steps whose coefficients stay in
// device memory.  Only the O(restart) Hessenberg/Givens scalars travel to the host, once
// per inner iteration, exactly where the reference evaluates its stopping tests.
#include <cmath>
#include <cstdlib>

#include "hifgpu.h"

namespace hifgpu {

constexpr int kRB = 4 * kNumSMs;  // reduction blocks (fixed -> run-to-run deterministic sums)
constexpr int kRT = 256;

__device__ __forceinline__ double block_sum(double v, double *sm) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  v = threadIdx.x < kRT / 32 ? sm[threadIdx.x] : 0.0;
  if (threadIdx.x < 32) v = warp_sum(v);
  __syncthreads();
  return v;  // valid in thread 0
}
__device__ __forceinline__ double block_max(double v, double *sm) {
  v = warp_max(v);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  v = threadIdx.x < kRT / 32 ? sm[threadIdx.x] : 0.0;
  if (threadIdx.x < 32) v = warp_max(v);
  __syncthreads();
  return v;
}

// y = A x, or y = b - A x (IterRefine.hpp:96-99, gmres.hpp:155-157); thread per row is the
// right shape for the 7-point matrices of the BASELINE configs, 4 lanes for denser rows.
template <int kLanes, bool RESID>
__global__ void spmv_kernel(const unsigned n, const unsigned *__restrict__ ptr, const int *__restrict__ col,
                            const double *__restrict__ val, const double *__restrict__ x,
                            const double *__restrict__ b, double *__restrict__ y) {
  const unsigned gid = blockIdx.x * blockDim.x + threadIdx.x, row = gid / kLanes, lane = gid % kLanes;
  double         acc = 0.0;
  if (row < n) {
    const unsigned e = ptr[row + 1];
    for (unsigned k = ptr[row] + lane; k < e; k += kLanes) acc = fma(val[k], x[col[k]], acc);
  }
#pragma unroll
  for (int o = kLanes / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (row < n && lane == 0) y[row] = RESID ? b[row] - acc : acc;
}

// mode 0: sum a[i]*b[i] ; 1: max |a[i]| ; 2: sum (a[i]*alpha)^2 with alpha = 1/part_in max
// stage 1 writes kRB partials, stage 2 (final_kernel) folds them in fixed order.
template <int MODE>
__global__ void __launch_bounds__(kRT) reduce_kernel(const unsigned n, const double *__restrict__ a,
                                                     const double *__restrict__ b, const double *scal_in,
                                                     double *__restrict__ part) {
  __shared__ double sm[kRT / 32];
  double            acc = 0.0;
  const double      alpha = MODE == 2 ? 1.0 / *scal_in : 0.0;
  for (unsigned i = blockIdx.x * kRT + threadIdx.x; i < n; i += gridDim.x * kRT) {
    if (MODE == 0) acc = fma(a[i], b[i], acc);
    if (MODE == 1) acc = fmax(acc, fabs(a[i]));
    if (MODE == 2) {
      const double t = a[i] * alpha;
      acc            = fma(t, t, acc);
    }
  }
  acc = MODE == 1 ? block_max(acc, sm) : block_sum(acc, sm);
  if (threadIdx.x == 0) part[blockIdx.x] = acc;
}
template <int MODE>
__global__ void __launch_bounds__(kRT) final_kernel(const unsigned nparts, const double *__restrict__ part,
                                                    double *out) {
  __shared__ double sm[kRT / 32];
  double            acc = 0.0;
  for (unsigned i = threadIdx.x; i < nparts; i += kRT) acc = MODE == 1 ? fmax(acc, part[i]) : acc + part[i];
  acc = MODE == 1 ? block_max(acc, sm) : block_sum(acc, sm);
  if (threadIdx.x == 0) *out = acc;
}

// y = a*x + y*by with a read from device memory (scaled by sign), used for MGS / updates
__global__ void axpy_dev_kernel(const unsigned n, const double *coef, const double sign,
                                const double *__restrict__ x, double *__restrict__ y) {
  const double a = sign * *coef;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    y[i] = fma(a, x[i], y[i]);
}
__global__ void axpy_kernel(const unsigned n, const double a, const double *__restrict__ x, double *__restrict__ y) {
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    y[i] = fma(a, x[i], y[i]);
}
// out = x + y
__global__ void add_kernel(const unsigned n, const double *__restrict__ x, const double *y, double *out) {
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = x[i] + y[i];
}
// out = x / (*den)   (true division like the reference: Q(i,j+1) = v[i] / v_norm)
__global__ void div_dev_kernel(const unsigned n, const double *__restrict__ x, const double *den, const bool take_sqrt,
                               double *__restrict__ out) {
  const double d = take_sqrt ? sqrt(*den) : *den;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = x[i] / d;
}

// One modified Gram-Schmidt step in ONE pass and ONE launch (gmres.hpp:174-177):
//   v <- v - h_k q_k   and, on the updated v,   h_next = <v, q_next>   (q_next = v itself: ||v||^2).
// The block partials are folded by the block that arrives last, in fixed order (deterministic:
// iteration counts must reproduce); it also re-arms the arrival counter.
__global__ void __launch_bounds__(kRT) mgs_step_kernel(const unsigned n, const double *coef,
                                                       const double *__restrict__ qk, const double *qnext,
                                                       double *v, double *__restrict__ part, unsigned *counter,
                                                       double *out) {
  __shared__ double sm[kRT / 32];
  __shared__ bool   last;
  const double      a   = -*coef;
  const bool        self = qnext == v;
  double            acc = 0.0;
  for (unsigned i = blockIdx.x * kRT + threadIdx.x; i < n; i += gridDim.x * kRT) {
    const double vi = fma(a, qk[i], v[i]);
    v[i]            = vi;
    acc             = fma(vi, self ? vi : qnext[i], acc);
  }
  acc = block_sum(acc, sm);
  if (threadIdx.x == 0) {
    part[blockIdx.x] = acc;
    __threadfence();
    last = atomicAdd(counter, 1u) == gridDim.x - 1u;
  }
  __syncthreads();
  if (last) {
    __threadfence();
    double t = 0.0;
    for (unsigned i = threadIdx.x; i < gridDim.x; i += kRT) t += reinterpret_cast<volatile double *>(part)[i];
    t = block_sum(t, sm);
    if (threadIdx.x == 0) {
      *out     = t;
      *counter = 0u;
    }
  }
}

// The whole modified Gram-Schmidt sweep of one Arnoldi step in ONE persistent launch (gmres.hpp:174-181):
//   h_k = <v, q_k>, v <- v - h_k q_k for k = 0 .. j, then ||v||^2 and q_{j+1} = v / ||v||.
// One CTA per SM keeps its contiguous slice of v in shared memory for the whole sweep (2 M doubles = 113 KB per
// SM), so a step reads q_k (L2: it was q_next of the step before) and q_{k+1} (HBM) and nothing else; the steps
// are separated by a grid barrier, after which EVERY block folds the block partials of the step in the same
// fixed order (deterministic, and all blocks subtract the same h_k).  Same products in the same order as the
// dot-then-axpy loop of the reference; one launch instead of j + 4, ~6 us per step instead of ~20.
constexpr int kMT = 512;
__device__ __forceinline__ double block_sum_mt(double v, double *sm) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  v = threadIdx.x < kMT / 32 ? sm[threadIdx.x] : 0.0;
  if (threadIdx.x < 32) v = warp_sum(v);
  __syncthreads();
  return v;  // valid in thread 0
}
__device__ __forceinline__ void grid_barrier(unsigned long long *cnt, unsigned long long target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(cnt, 1ull);
    unsigned long long seen;
    do {
      asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(seen) : "l"(cnt) : "memory");
    } while (seen < target);
    __threadfence();
  }
  __syncthreads();
}
// sum of the `nb` block partials of one step, folded by warp 0 in a fixed order; result in shared `s_h`
__device__ __forceinline__ void fold_partials(const double *part, unsigned nb, double *s_h) {
  if (threadIdx.x < 32) {
    double t = 0.0;
    for (unsigned b = threadIdx.x; b < nb; b += 32) t += __ldcg(part + b);
    t = warp_sum(t);
    if (threadIdx.x == 0) *s_h = t;
  }
  __syncthreads();
}
__global__ void __launch_bounds__(kMT, 1)
    mgs_persistent_kernel(const unsigned n, const unsigned j, const unsigned slice, const double *__restrict__ Q,
                          const double *__restrict__ v, double *__restrict__ qout, double *__restrict__ coef,
                          double *__restrict__ nrm2_out, double *part, unsigned long long *bar, unsigned long long target) {
  extern __shared__ double sw[];  // this block's slice of v
  __shared__ double sm[kMT / 32];
  __shared__ double s_h;
  const unsigned nb = gridDim.x, tid = threadIdx.x;
  const unsigned lo = min(n, blockIdx.x * slice), hi = min(n, lo + slice);
  double         acc = 0.0;
  for (unsigned i = lo + tid; i < hi; i += kMT) {
    const double w = v[i];
    sw[i - lo]     = w;
    acc            = fma(w, Q[i], acc);
  }
  acc = block_sum_mt(acc, sm);
  if (tid == 0) part[blockIdx.x] = acc;
  target += nb;
  grid_barrier(bar, target);
  for (unsigned k = 0; k <= j; ++k) {
    fold_partials(part + static_cast<std::size_t>(k) * nb, nb, &s_h);
    const double h = s_h;
    if (blockIdx.x == 0 && tid == 0) coef[k] = h;
    const double *qk   = Q + static_cast<std::size_t>(k) * n;
    const double *qn   = qk + n;
    const bool    self = k == j;
    acc                = 0.0;
    for (unsigned i = lo + tid; i < hi; i += kMT) {
      const double w = fma(-h, qk[i], sw[i - lo]);
      sw[i - lo]     = w;
      acc            = fma(w, self ? w : qn[i], acc);
    }
    acc = block_sum_mt(acc, sm);  // (its barriers also order the reads of s_h before the next fold writes it)
    if (tid == 0) part[static_cast<std::size_t>(k + 1u) * nb + blockIdx.x] = acc;
    target += nb;
    grid_barrier(bar, target);
  }
  fold_partials(part + static_cast<std::size_t>(j + 1u) * nb, nb, &s_h);
  const double nrm2 = s_h;
  if (blockIdx.x == 0 && tid == 0) *nrm2_out = nrm2;
  if (qout) {  // Q(:, j+1) = v / ||v||  (true division, gmres.hpp:181)
    const double d = sqrt(nrm2);
    for (unsigned i = lo + tid; i < hi; i += kMT) qout[i] = sw[i - lo] / d;
  }
}

namespace {

inline unsigned cdiv(std::size_t a, std::size_t b) { return static_cast<unsigned>((a + b - 1) / b); }
inline unsigned nblk(std::size_t n) { return std::min<unsigned>(kRB, std::max(1u, cdiv(n, kRT))); }
constexpr int   kEW = 2 * kNumSMs;  // grid of the grid-stride element-wise kernels

void ensure(Handle *h, DevBuf<double> &buf, std::size_t n) {
  if (buf.n < n) buf.alloc(n, &h->device_bytes);
}
void ensure_scal(Handle *h) {
  ensure(h, h->kr_scal, 256);
  ensure(h, h->kr_part, kRB);
  if (!h->kr_count.n) h->kr_count.alloc(1, &h->device_bytes);  // zeroed: arrival counter of mgs_step_kernel
}

// out (device scalar) = <a, b>
void dot_to(Handle *h, std::size_t n, const double *a, const double *b, double *d_out) {
  const unsigned nb = nblk(n);
  reduce_kernel<0><<<nb, kRT, 0, h->stream>>>(static_cast<unsigned>(n), a, b, nullptr, h->kr_part.p);
  final_kernel<0><<<1, kRT, 0, h->stream>>>(nb, h->kr_part.p, d_out);
  HIF_KERNEL_CHECK();
  h->launch_count += 2;
}

double fetch(Handle *h, const double *d_scalar) {
  HIF_CUDA(cudaMemcpyAsync(h->h_scal, d_scalar, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  HIF_CUDA(cudaStreamSynchronize(h->stream));
  return h->h_scal[0];
}

}  // namespace

void spmv_dev(Handle *h, const double *d_x, double *d_y) {
  if (!h->has_A) throw std::logic_error("no matrix attached: call lhfdGpuSetMatrix first");
  const DevCsr &A = h->A.A;
  const double  avg = static_cast<double>(A.nnz) / static_cast<double>(A.nrows ? A.nrows : 1);
  const unsigned n  = static_cast<unsigned>(A.nrows);
  if (avg > 16.0)
    spmv_kernel<4, false><<<cdiv(A.nrows * 4, kRT), kRT, 0, h->stream>>>(n, A.ptr.p, A.col.p, A.val.p, d_x, nullptr, d_y);
  else
    spmv_kernel<1, false><<<cdiv(A.nrows, kRT), kRT, 0, h->stream>>>(n, A.ptr.p, A.col.p, A.val.p, d_x, nullptr, d_y);
  HIF_KERNEL_CHECK();
  ++h->launch_count;
}

static void resid_dev(Handle *h, const double *d_b, const double *d_x, double *d_r) {  // r = b - A x
  if (!h->has_A) throw std::logic_error("no matrix attached: call lhfdGpuSetMatrix first");
  const DevCsr &A = h->A.A;
  const double  avg = static_cast<double>(A.nnz) / static_cast<double>(A.nrows ? A.nrows : 1);
  const unsigned n  = static_cast<unsigned>(A.nrows);
  if (avg > 16.0)
    spmv_kernel<4, true><<<cdiv(A.nrows * 4, kRT), kRT, 0, h->stream>>>(n, A.ptr.p, A.col.p, A.val.p, d_x, d_b, d_r);
  else
    spmv_kernel<1, true><<<cdiv(A.nrows, kRT), kRT, 0, h->stream>>>(n, A.ptr.p, A.col.p, A.val.p, d_x, d_b, d_r);
  HIF_KERNEL_CHECK();
  ++h->launch_count;
}

// max-scaled two-pass 2-norm, utils/math.hpp:112-137; returns the value on the host
double norm2_dev(Handle *h, const double *d_v, std::size_t n) {
  if (!n) return 0.0;
  ensure_scal(h);
  const unsigned nb  = nblk(n);
  double *       mx  = h->kr_scal.p + 201, *ss = h->kr_scal.p + 202;
  reduce_kernel<1><<<nb, kRT, 0, h->stream>>>(static_cast<unsigned>(n), d_v, nullptr, nullptr, h->kr_part.p);
  final_kernel<1><<<1, kRT, 0, h->stream>>>(nb, h->kr_part.p, mx);
  HIF_KERNEL_CHECK();
  h->launch_count += 2;
  const double max_mag = fetch(h, mx);
  if (max_mag == 0.0) return 0.0;  // sum of |v_i| of an all-zero vector
  reduce_kernel<2><<<nb, kRT, 0, h->stream>>>(static_cast<unsigned>(n), d_v, nullptr, mx, h->kr_part.p);
  final_kernel<2><<<1, kRT, 0, h->stream>>>(nb, h->kr_part.p, ss);
  HIF_KERNEL_CHECK();
  h->launch_count += 2;
  return max_mag * std::sqrt(fetch(h, ss));
}

// IterRefine::iter_refine, fixed count (IterRefine.hpp:77-105)
void hifir_dev(Handle *h, const double *d_b, std::size_t nirs, double *d_x, std::size_t rank) {
  const std::size_t n = h->n0();
  if (nirs <= 1) {
    apply_dev(h, d_b, d_x, rank);
    return;
  }
  if (!h->has_A) throw std::logic_error("iterative refinement needs the matrix: call lhfdGpuSetMatrix first");
  ensure(h, h->ir_r, n);
  ensure(h, h->ir_t, n);
  // i = 0: xk = 0, x = b -> r = M^{-1} b ; x = r + 0
  apply_dev(h, d_b, d_x, rank);
  for (std::size_t i = 1; i < nirs; ++i) {
    // xk = x ; t = b - A xk ; r = M^{-1} t ; x = r + xk
    resid_dev(h, d_b, d_x, h->ir_t.p);
    apply_dev(h, h->ir_t.p, h->ir_r.p, rank);
    add_kernel<<<kEW, kRT, 0, h->stream>>>(static_cast<unsigned>(n), h->ir_r.p, d_x, d_x);
    HIF_KERNEL_CHECK();
    ++h->launch_count;
  }
}

// IterRefine::iter_refine with residual bounds (IterRefine.hpp:121-165)
void hifir_betas_dev(Handle *h, const double *d_b, std::size_t nirs, const double *betas, double *d_x,
                     std::size_t rank, long *iters_out, int *flag_out) {
  const std::size_t n = h->n0();
  if (nirs <= 1) {
    apply_dev(h, d_b, d_x, rank);
    *iters_out = 1;
    *flag_out  = -1;
    return;
  }
  if (!h->has_A) throw std::logic_error("iterative refinement needs the matrix: call lhfdGpuSetMatrix first");
  const double bnorm = norm2_dev(h, d_b, n);
  HIF_CUDA(cudaMemsetAsync(d_x, 0, n * sizeof(double), h->stream));
  if (bnorm == 0.0) {
    *iters_out = 0;
    *flag_out  = 0;
    return;
  }
  ensure(h, h->ir_r, n);
  ensure(h, h->ir_xk, n);
  HIF_CUDA(cudaMemcpyAsync(h->ir_r.p, d_b, n * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
  long iters = 0;
  int  flag  = 0;
  for (;;) {
    apply_dev(h, h->ir_r.p, h->ir_xk.p, rank);
    add_kernel<<<kEW, kRT, 0, h->stream>>>(static_cast<unsigned>(n), h->ir_xk.p, d_x, d_x);
    HIF_KERNEL_CHECK();
    ++h->launch_count;
    if (++iters >= static_cast<long>(nirs)) {
      flag = -1;
      break;
    }
    resid_dev(h, d_b, d_x, h->ir_r.p);
    const double res = norm2_dev(h, h->ir_r.p, n) / bnorm;
    if (res <= betas[0]) break;
    if (res > betas[1]) {
      flag = 1;
      break;
    }
  }
  *iters_out = iters;
  *flag_out  = flag;
}

// gmres_hif / fgmres_hifir (examples/advanced/gmres.hpp:18-122 / 126-230)
void krylov_dev(Handle *h, bool flexible, const double *d_b, int restart, double rtol, int maxit, bool full_rank,
                double *d_x, int *flag_out, int *iters_out, int *nmv_out) {
  if (!h->has_A) throw std::logic_error("Krylov solve needs the matrix: call lhfdGpuSetMatrix first");
  if (restart < 1 || restart > 96) throw std::invalid_argument("restart must be in [1, 96]");
  const std::size_t n  = h->n0();
  const unsigned    un = static_cast<unsigned>(n);
  const std::size_t rr = full_rank ? static_cast<std::size_t>(-1) : 0;
  int               iter = 0, flag = 0, num_mv = 0;
  ensure_scal(h);
  const double beta0 = norm2_dev(h, d_b, n);
  HIF_CUDA(cudaMemsetAsync(d_x, 0, n * sizeof(double), h->stream));
  *flag_out = *iters_out = *nmv_out = 0;
  if (beta0 == 0.0) return;
  ensure(h, h->kr_v, n);
  ensure(h, h->kr_w, n);
  ensure(h, h->kr_Q, n * static_cast<std::size_t>(restart));
  if (flexible) ensure(h, h->kr_Z, n * static_cast<std::size_t>(restart));
  double *v = h->kr_v.p, *w = h->kr_w.p, *Q = h->kr_Q.p, *Z = h->kr_Z.p;
  double *d_w2 = h->kr_scal.p;  // [0, restart): MGS coefficients ; [restart]: ||v||^2 ; [restart+1 ..]: y
  std::vector<double> y(restart + 1, 0.0), w2(restart, 0.0), R(static_cast<std::size_t>(restart) * restart, 0.0),
      J(2 * static_cast<std::size_t>(restart), 0.0);
  const int max_outer = static_cast<int>(std::ceil(static_cast<double>(maxit) / restart));
  double    resid     = 1.0;
  for (int it_outer = 0; it_outer < max_outer; ++it_outer) {
    if (iter)
      resid_dev(h, d_b, d_x, v);
    else
      HIF_CUDA(cudaMemcpyAsync(v, d_b, n * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    const double beta = norm2_dev(h, v, n);
    y[0]              = beta;
    {
      // Q(:,0) = v / beta
      h->h_scal[1] = beta;
      HIF_CUDA(cudaMemcpyAsync(d_w2 + 200, h->h_scal + 1, sizeof(double), cudaMemcpyHostToDevice, h->stream));
      div_dev_kernel<<<kEW, kRT, 0, h->stream>>>(un, v, d_w2 + 200, false, Q);
      HIF_KERNEL_CHECK();
      HIF_CUDA(cudaStreamSynchronize(h->stream));  // h_scal[1] is reused below
      h->launch_count += 2;
    }
    int               j    = 0;
    const std::size_t nirs = static_cast<std::size_t>(1) << it_outer;
    for (;;) {
      const double *qj = Q + static_cast<std::size_t>(j) * n;
      if (flexible) {
        double *zj = Z + static_cast<std::size_t>(j) * n;
        hifir_dev(h, qj, nirs, zj, rr);  // M.hifir(A, v, nirs, w, false, rr) ; Z(:,j) = w
        num_mv += static_cast<int>(nirs);
        spmv_dev(h, zj, v);              // v = A w
      } else {
        apply_dev(h, qj, w, rr);
        num_mv += 1;
        spmv_dev(h, w, v);
      }
      // modified Gram-Schmidt, coefficients stay on the device (gmres.hpp:174-177): h_0 = <v, q_0>, then
      // one fused launch per k: v -= h_k q_k and h_{k+1} = <v, q_{k+1}> (after the last k: norm2_sq(v),
      // math.hpp:97-105) -- the same products in the same order as dot-then-axpy, one pass instead of two
      static const bool fused_mgs = [] {
        const char *e = std::getenv("HIFIR_B200_MGS_FUSED");
        return !e || std::atoi(e) != 0;
      }();
      // one persistent launch for the whole sweep when a slice of v fits the shared memory of an SM
      static const bool persist_mgs = [] {
        const char *e = std::getenv("HIFIR_B200_MGS_PERSIST");
        return !e || std::atoi(e) != 0;
      }();
      const unsigned    pgrid  = static_cast<unsigned>(std::max(1, h->num_sms));
      const unsigned    pslice = cdiv(n, pgrid);
      const std::size_t psmem  = static_cast<std::size_t>(pslice) * sizeof(double);
      const bool        persist = fused_mgs && persist_mgs && !h->kr_no_coop && psmem <= 200u * 1024u;
      bool              launched = false;
      if (persist) {
        if (h->kr_mpart.n < static_cast<std::size_t>(restart + 2) * pgrid)
          h->kr_mpart.alloc(static_cast<std::size_t>(restart + 2) * pgrid, &h->device_bytes);
        if (!h->kr_bar.n) {
          h->kr_bar.alloc(1, &h->device_bytes);
          h->kr_bar_base = 0;
        }
        static bool configured[64] = {false};
        if (h->device >= 64 || !configured[h->device]) {
          HIF_CUDA(cudaFuncSetAttribute(mgs_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
          if (h->device < 64) configured[h->device] = true;
        }
        // a COOPERATIVE launch: the runtime refuses it when the grid can not be resident at once (the barrier
        // would never complete) -- then, and from then on, the per-step kernels do the work
        double *           qout = j + 1 < restart ? Q + static_cast<std::size_t>(j + 1) * n : nullptr;
        unsigned           a_n = un, a_j = static_cast<unsigned>(j), a_slice = pslice;
        const double *     a_Q = Q, *a_v = v;
        double *           a_coef = d_w2, *a_nrm = d_w2 + restart, *a_part = h->kr_mpart.p;
        unsigned long long *a_bar = h->kr_bar.p, a_base = h->kr_bar_base;
        void *args[] = {&a_n, &a_j, &a_slice, &a_Q, &a_v, &qout, &a_coef, &a_nrm, &a_part, &a_bar, &a_base};
        const cudaError_t e = cudaLaunchCooperativeKernel(reinterpret_cast<const void *>(mgs_persistent_kernel), dim3(pgrid),
                                                          dim3(kMT), args, psmem, h->stream);
        if (e == cudaSuccess) {
          h->kr_bar_base += static_cast<unsigned long long>(j + 2) * pgrid;
          ++h->launch_count;
          launched = true;
        } else if (e == cudaErrorCooperativeLaunchTooLarge || e == cudaErrorNotSupported || e == cudaErrorInvalidConfiguration) {
          cudaGetLastError();
          h->kr_no_coop = true;
        } else {
          HIF_CUDA(e);
        }
      }
      if (launched) {
      } else if (fused_mgs) {
        dot_to(h, n, v, Q, d_w2);
        for (int k = 0; k <= j; ++k) {
          const double *qk    = Q + static_cast<std::size_t>(k) * n;
          const double *qnext = k < j ? qk + n : v;
          mgs_step_kernel<<<nblk(n), kRT, 0, h->stream>>>(un, d_w2 + k, qk, qnext, v, h->kr_part.p, h->kr_count.p,
                                                          k < j ? d_w2 + k + 1 : d_w2 + restart);
          HIF_KERNEL_CHECK();
          ++h->launch_count;
        }
      } else {
        for (int k = 0; k <= j; ++k) {
          const double *qk = Q + static_cast<std::size_t>(k) * n;
          dot_to(h, n, v, qk, d_w2 + k);
          axpy_dev_kernel<<<kEW, kRT, 0, h->stream>>>(un, d_w2 + k, -1.0, qk, v);
          HIF_KERNEL_CHECK();
          ++h->launch_count;
        }
        dot_to(h, n, v, v, d_w2 + restart);
      }
      if (!launched && j + 1 < restart) {
        div_dev_kernel<<<kEW, kRT, 0, h->stream>>>(un, v, d_w2 + restart, true, Q + static_cast<std::size_t>(j + 1) * n);
        HIF_KERNEL_CHECK();
        ++h->launch_count;
      }
      HIF_CUDA(cudaMemcpyAsync(h->h_scal, d_w2, (restart + 1) * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
      HIF_CUDA(cudaStreamSynchronize(h->stream));
      for (int k = 0; k <= j; ++k) w2[k] = h->h_scal[k];
      const double v_norm2 = h->h_scal[restart], v_norm = std::sqrt(v_norm2);
      // Givens rotations (gmres.hpp:184-196), host scalars
      for (int c = 0; c + 1 <= j; ++c) {
        const double tmp = w2[c];
        w2[c]            = J[c] * tmp + J[restart + c] * w2[c + 1];
        w2[c + 1]        = -J[restart + c] * tmp + J[c] * w2[c + 1];
      }
      const double rho = std::sqrt(w2[j] * w2[j] + v_norm2);
      J[j]             = w2[j] / rho;
      J[restart + j]   = v_norm / rho;
      y[j + 1]         = -J[restart + j] * y[j];
      y[j]             = J[j] * y[j];
      w2[j]            = rho;
      for (int k = 0; k <= j; ++k) R[static_cast<std::size_t>(j) * restart + k] = w2[k];
      const double resid_prev = resid;
      resid                   = std::fabs(y[j + 1]) / beta0;
      if (resid >= resid_prev * (1.0 - 1e-8)) {
        flag = 1;  // STAGNATED
        break;
      } else if (iter >= maxit) {
        flag = 2;  // DIVERGED
        break;
      }
      ++iter;
      if (resid <= rtol || j + 1 >= restart) break;
      ++j;
    }
    for (int k = j; k > -1; --k) {
      y[k] /= R[static_cast<std::size_t>(k) * restart + k];
      const double tmp = y[k];
      for (int i = k - 1; i > -1; --i) y[i] -= tmp * R[static_cast<std::size_t>(k) * restart + i];
    }
    if (flexible) {  // x += Z(:,0:j) y  (gmres.hpp:223-226)
      for (int i = 0; i <= j; ++i) {
        axpy_kernel<<<kEW, kRT, 0, h->stream>>>(un, y[i], Z + static_cast<std::size_t>(i) * n, d_x);
        HIF_KERNEL_CHECK();
        ++h->launch_count;
      }
    } else {  // v = Q y ; x += M^{-1} v  (gmres.hpp:111-118)
      HIF_CUDA(cudaMemsetAsync(v, 0, n * sizeof(double), h->stream));
      for (int i = 0; i <= j; ++i) {
        axpy_kernel<<<kEW, kRT, 0, h->stream>>>(un, y[i], Q + static_cast<std::size_t>(i) * n, v);
        HIF_KERNEL_CHECK();
        ++h->launch_count;
      }
      apply_dev(h, v, w, rr);
      add_kernel<<<kEW, kRT, 0, h->stream>>>(un, w, d_x, d_x);
      HIF_KERNEL_CHECK();
      ++h->launch_count;
    }
    if (resid <= rtol || flag != 0) break;
  }
  check_sweep_error(h);
  *flag_out  = flag;
  *iters_out = iter;
  *nmv_out   = num_mv;
}

// ---------------------------------------------------------------------------------------------------------
// Block Krylov: nrhs independent gmres_hif / fgmres_hifir / hifir runs on row-interleaved blocks X[i*nc + c]
// (the layout of apply_mrhs_dev).  Every kernel below handles all columns in one launch.  Thread mapping: a
// warp covers cw consecutive columns (cw = the smallest power of two >= nc, at most 32) of 32 / cw
// consecutive rows, so every access of a row moves its cw values together; blockIdx.y selects a group of 32
// columns when nc > 32.  A column's arithmetic and fold order depend on n, cw and the number of column groups
// ceil(nc / 32) only -- never on the values of the other columns or on the position the column holds.  The
// groups enter through the row blocks of the reductions, nb_red = min(kRB / groups, ceil(n / rows_cta)) of
// col_shape: at n = 262 144 and cw = 32 that is 592, 296 or 197 blocks for 1, 2 or 3 groups, so the same
// column folds in another order in a block of another width.  mask[c] == 0 marks a retired column: the SpMV and
// the reductions give 0 for it and the divisions write 0, so its basis vectors stay exact zeros.
__device__ __forceinline__ void col_lane(unsigned cw, unsigned &c, unsigned &r0, unsigned &rstride) {
  const unsigned lane = threadIdx.x & 31u, rw = 32u / cw;
  c       = blockIdx.y * 32u + (lane & (cw - 1u));
  r0      = (blockIdx.x * (kRT / 32) + (threadIdx.x >> 5)) * rw + lane / cw;
  rstride = gridDim.x * (kRT / 32) * rw;
}
// per-column sum (MAX: max) over the block: the lanes of a warp that share a column, then the warps in
// order; valid in threads [0, cw) for column blockIdx.y * 32 + threadIdx.x
template <bool MAX>
__device__ __forceinline__ double block_col_fold(double v, unsigned cw, double *sm) {
  for (unsigned o = 16; o >= cw; o >>= 1) {
    const double t = __shfl_xor_sync(0xffffffffu, v, o);
    v              = MAX ? fmax(v, t) : v + t;
  }
  if ((threadIdx.x & 31u) < cw) sm[threadIdx.x] = v;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x < cw)
    for (unsigned w = 0; w < kRT / 32; ++w) t = MAX ? fmax(t, sm[w * 32 + threadIdx.x]) : t + sm[w * 32 + threadIdx.x];
  __syncthreads();
  return t;
}

// per-column reductions, stage 1 (mode as reduce_kernel: 0 dot, 1 max |a|, 2 sum (a / scal[c])^2); writes the
// block partials part[c * gridDim.x + blockIdx.x]
template <int MODE>
__global__ void __launch_bounds__(kRT) reduce_cols_kernel(const unsigned n, const unsigned nc, const unsigned cw,
                                                          const double *__restrict__ a, const double *__restrict__ b,
                                                          const double *__restrict__ scal, const int *__restrict__ mask,
                                                          double *__restrict__ part) {
  __shared__ double sm[kRT];
  unsigned          c, r0, rs;
  col_lane(cw, c, r0, rs);
  const bool on = c < nc && (!mask || mask[c]);
  double     alpha = 0.0;
  if (MODE == 2 && on) alpha = scal[c] > 0.0 ? 1.0 / scal[c] : 0.0;
  double acc = 0.0;
  if (on)
    for (unsigned i = r0; i < n; i += rs) {
      const std::size_t g = static_cast<std::size_t>(i) * nc + c;
      if (MODE == 0) acc = fma(a[g], b[g], acc);
      if (MODE == 1) acc = fmax(acc, fabs(a[g]));
      if (MODE == 2) {
        const double t = a[g] * alpha;
        acc            = fma(t, t, acc);
      }
    }
  acc = block_col_fold<MODE == 1>(acc, cw, sm);
  const unsigned cc = blockIdx.y * 32u + threadIdx.x;
  if (threadIdx.x < cw && cc < nc) part[static_cast<std::size_t>(cc) * gridDim.x + blockIdx.x] = acc;
}
// stage 2: one warp per column folds its nparts partials in fixed order
template <int MODE>
__global__ void __launch_bounds__(kRT) final_cols_kernel(const unsigned nparts, const unsigned nc,
                                                         const double *__restrict__ part, double *__restrict__ out) {
  const unsigned lane = threadIdx.x & 31u;
  for (unsigned c = blockIdx.x * (kRT / 32) + (threadIdx.x >> 5); c < nc; c += gridDim.x * (kRT / 32)) {
    double t = 0.0;
    for (unsigned b = lane; b < nparts; b += 32) {
      const double p = part[static_cast<std::size_t>(c) * nparts + b];
      t              = MODE == 1 ? fmax(t, p) : t + p;
    }
    t = MODE == 1 ? warp_max(t) : warp_sum(t);
    if (lane == 0) out[c] = t;
  }
}

// One modified Gram-Schmidt step for every column (mgs_step_kernel on blocks):
//   v_c <- v_c - h_{k,c} q_{k,c}   and, on the updated v,   out_c = <v_c, qnext_c>   (qnext = v: ||v_c||^2).
// The block that arrives last folds the partials of all columns, one warp per column in fixed order, and
// re-arms the arrival counter.
__global__ void __launch_bounds__(kRT) mgs_step_cols_kernel(const unsigned n, const unsigned nc, const unsigned cw,
                                                            const double *coef, const double *__restrict__ qk,
                                                            const double *qnext, double *v, const int *__restrict__ mask,
                                                            double *part, unsigned *counter, double *out) {
  __shared__ double sm[kRT];
  __shared__ bool   last;
  unsigned          c, r0, rs;
  col_lane(cw, c, r0, rs);
  const bool   on   = c < nc && mask[c];
  const double a    = on ? -coef[c] : 0.0;
  const bool   self = qnext == v;
  double       acc  = 0.0;
  if (on)
    for (unsigned i = r0; i < n; i += rs) {
      const std::size_t g  = static_cast<std::size_t>(i) * nc + c;
      const double      vi = fma(a, qk[g], v[g]);
      v[g]                 = vi;
      acc                  = fma(vi, self ? vi : qnext[g], acc);
    }
  acc               = block_col_fold<false>(acc, cw, sm);
  const unsigned cc = blockIdx.y * 32u + threadIdx.x;
  if (threadIdx.x < cw) {
    if (cc < nc) part[static_cast<std::size_t>(cc) * gridDim.x + blockIdx.x] = acc;
    __threadfence();
  }
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(counter, 1u) == gridDim.x * gridDim.y - 1u;
  __syncthreads();
  if (last) {
    __threadfence();
    const unsigned lane = threadIdx.x & 31u;
    for (unsigned col = threadIdx.x >> 5; col < nc; col += kRT / 32) {
      double t = 0.0;
      for (unsigned b = lane; b < gridDim.x; b += 32)
        t += reinterpret_cast<volatile double *>(part)[static_cast<std::size_t>(col) * gridDim.x + b];
      t = warp_sum(t);
      if (lane == 0) out[col] = t;
    }
    __syncthreads();
    if (threadIdx.x == 0) *counter = 0u;
  }
}

// Y = A X, or R = B - A X; zero in retired columns: the lanes of a warp run across cw columns of 32 / cw rows,
// so every gather of X moves whole rows of the block; the column groups of nc > 32 loop inside the warp, the
// row of A is fetched from memory once.  Per column the products are summed in row order, as spmv_kernel<1>.
template <bool RESID>
__global__ void __launch_bounds__(kRT) spmv_cols_kernel(const unsigned n, const unsigned nc, const unsigned cw,
                                                        const unsigned *__restrict__ ptr, const int *__restrict__ col,
                                                        const double *__restrict__ val, const double *__restrict__ x,
                                                        const double *__restrict__ b, const int *__restrict__ mask,
                                                        double *__restrict__ y) {
  const unsigned lane = threadIdx.x & 31u, rw = 32u / cw;
  const unsigned row  = ((blockIdx.x * kRT + threadIdx.x) >> 5) * rw + lane / cw;
  if (row >= n) return;
  const unsigned e0 = ptr[row], e1 = ptr[row + 1];
  for (unsigned c = lane & (cw - 1u); c < nc; c += 32) {
    const std::size_t g = static_cast<std::size_t>(row) * nc + c;
    if (mask && !mask[c]) {
      y[g] = 0.0;
      continue;
    }
    double acc = 0.0;
    for (unsigned k = e0; k < e1; ++k) acc = fma(val[k], x[static_cast<std::size_t>(col[k]) * nc + c], acc);
    y[g] = RESID ? b[g] - acc : acc;
  }
}

// out_c = x_c / d_c with d_c = sqrt(den[c]) or den[c] (true division, gmres.hpp:181); zero in retired columns
// and where d_c is not positive
__global__ void __launch_bounds__(kRT) div_cols_kernel(const unsigned n, const unsigned nc, const unsigned cw,
                                                       const double *__restrict__ x, const double *__restrict__ den,
                                                       const bool take_sqrt, const int *__restrict__ mask,
                                                       double *__restrict__ out) {
  unsigned c, r0, rs;
  col_lane(cw, c, r0, rs);
  if (c >= nc) return;
  const double d  = take_sqrt ? sqrt(den[c]) : den[c];
  const bool   on = mask[c] && d > 0.0;
  for (unsigned i = r0; i < n; i += rs) {
    const std::size_t g = static_cast<std::size_t>(i) * nc + c;
    out[g]              = on ? x[g] / d : 0.0;
  }
}

// x_c <- x_c + sum_{k < nterms} y[k][c] Z_k(:, c), one fma per term in the order k = 0 .. nterms-1 (the axpy
// loop of krylov_dev in one pass); Z = [nterms][n][nc]
__global__ void __launch_bounds__(kRT) axpy_cols_kernel(const unsigned n, const unsigned nc, const unsigned cw,
                                                        const unsigned nterms, const double *__restrict__ y,
                                                        const double *__restrict__ Z, double *__restrict__ x) {
  unsigned c, r0, rs;
  col_lane(cw, c, r0, rs);
  if (c >= nc) return;
  const std::size_t stride = static_cast<std::size_t>(n) * nc;
  for (unsigned i = r0; i < n; i += rs) {
    const std::size_t g   = static_cast<std::size_t>(i) * nc + c;
    double            acc = x[g];
    for (unsigned k = 0; k < nterms; ++k) acc = fma(y[static_cast<std::size_t>(k) * nc + c], Z[k * stride + g], acc);
    x[g] = acc;
  }
}

// x_c <- x_c + w_c in the columns that mask marks, x_c unchanged in the others (the batched apply of a zero
// column leaves the ready-bit tags of its sweeps behind: denormals, not exact zeros)
__global__ void __launch_bounds__(kRT) add_cols_kernel(const unsigned n, const unsigned nc, const unsigned cw,
                                                       const int *__restrict__ mask, const double *__restrict__ w,
                                                       double *__restrict__ x) {
  unsigned c, r0, rs;
  col_lane(cw, c, r0, rs);
  if (c >= nc || !mask[c]) return;
  for (unsigned i = r0; i < n; i += rs) {
    const std::size_t g = static_cast<std::size_t>(i) * nc + c;
    x[g]                = w[g] + x[g];
  }
}

// x_c <- 0 for the retired columns
__global__ void __launch_bounds__(kRT) zero_cols_kernel(const unsigned n, const unsigned nc, const unsigned cw,
                                                        const int *__restrict__ mask, double *__restrict__ x) {
  unsigned c, r0, rs;
  col_lane(cw, c, r0, rs);
  if (c >= nc || mask[c]) return;
  for (unsigned i = r0; i < n; i += rs) x[static_cast<std::size_t>(i) * nc + c] = 0.0;
}

namespace {

struct ColShape {  // launch shape of the block kernels for an n x nc block
  unsigned n = 0, nc = 0, cw = 1, groups = 1;
  unsigned nb_red = 1, nb_ew = 1;  // row blocks of the reductions (fixed: deterministic folds) / element-wise kernels
  dim3     red() const { return dim3(nb_red, groups); }
  dim3     ew() const { return dim3(nb_ew, groups); }
};
ColShape col_shape(std::size_t n, std::size_t nc) {
  ColShape s;
  s.n  = static_cast<unsigned>(n);
  s.nc = static_cast<unsigned>(nc);
  while (s.cw < 32u && s.cw < nc) s.cw <<= 1;
  s.groups               = cdiv(nc, 32);
  const unsigned rows_cta = (kRT / 32) * (32u / s.cw);
  s.nb_red = std::max(1u, std::min<unsigned>(kRB / s.groups, cdiv(n, rows_cta)));
  s.nb_ew  = std::max(1u, std::min<unsigned>(2 * kRB / s.groups, cdiv(n, rows_cta)));
  return s;
}

void check_block(Handle *h, std::size_t nrhs) {
  if (static_cast<unsigned long long>(h->n0()) * nrhs > 0xffffffffull) throw std::length_error("multi-rhs block too large");
}

void ensure_cols_scal(Handle *h, std::size_t nc) {
  ensure(h, h->kb_red, 4 * nc);
  ensure(h, h->kb_part, static_cast<std::size_t>(kRB) * nc);
  if (h->kb_mask.n < 2 * nc) h->kb_mask.alloc(2 * nc, &h->device_bytes);  // active columns, columns of the cycle
  if (!h->kb_count.n) h->kb_count.alloc(1, &h->device_bytes);  // zeroed: arrival counter of mgs_step_cols_kernel
}

// out[c] (device) = reduction MODE of column c
template <int MODE>
void reduce_cols(Handle *h, const ColShape &s, const double *a, const double *b, const double *scal, const int *mask,
                 double *d_out) {
  reduce_cols_kernel<MODE><<<s.red(), kRT, 0, h->stream>>>(s.n, s.nc, s.cw, a, b, scal, mask, h->kb_part.p);
  final_cols_kernel<MODE><<<cdiv(s.nc, kRT / 32), kRT, 0, h->stream>>>(s.nb_red, s.nc, h->kb_part.p, d_out);
  HIF_KERNEL_CHECK();
  h->launch_count += 2;
}

// per-column max-scaled two-pass 2-norm (utils/math.hpp:112-137), returned on the host
void norm2_cols(Handle *h, const ColShape &s, const double *d_v, const int *mask, double *out) {
  double *mx = h->kb_red.p, *ss = h->kb_red.p + s.nc;
  reduce_cols<1>(h, s, d_v, nullptr, nullptr, mask, mx);
  reduce_cols<2>(h, s, d_v, nullptr, mx, mask, ss);
  std::vector<double> t(2 * static_cast<std::size_t>(s.nc));
  HIF_CUDA(cudaMemcpyAsync(t.data(), mx, t.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  HIF_CUDA(cudaStreamSynchronize(h->stream));
  for (unsigned c = 0; c < s.nc; ++c) out[c] = t[c] == 0.0 ? 0.0 : t[c] * std::sqrt(t[s.nc + c]);
}

void spmv_cols(Handle *h, const ColShape &s, const double *d_x, const double *d_b, const int *mask, double *d_y) {
  if (!h->has_A) throw std::logic_error("no matrix attached: call lhfdGpuSetMatrix first");
  const DevCsr & A    = h->A.A;
  const unsigned rw   = 32u / s.cw;
  const unsigned grid = cdiv(static_cast<std::size_t>(cdiv(s.n, rw)) * 32u, kRT);
  if (d_b)
    spmv_cols_kernel<true><<<grid, kRT, 0, h->stream>>>(s.n, s.nc, s.cw, A.ptr.p, A.col.p, A.val.p, d_x, d_b, mask, d_y);
  else
    spmv_cols_kernel<false><<<grid, kRT, 0, h->stream>>>(s.n, s.nc, s.cw, A.ptr.p, A.col.p, A.val.p, d_x, nullptr, mask, d_y);
  HIF_KERNEL_CHECK();
  ++h->launch_count;
}

template <class T>
void upload(Handle *h, T *d_dst, const std::vector<T> &src) {  // pageable source: staged before the call returns
  HIF_CUDA(cudaMemcpyAsync(d_dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice, h->stream));
}

}  // namespace

void check_krylov_mrhs(Handle *h, std::size_t nrhs, int restart) {
  if (!h->has_A) throw std::logic_error("Krylov solve needs the matrix: call lhfdGpuSetMatrix first");
  if (restart < 1 || restart > 96) throw std::invalid_argument("restart must be in [1, 96]");
  check_block(h, nrhs);
}

// hifir_dev on a block: the first apply, then R = B - A X, M^{-1} R and X += ... for every column at once
void hifir_mrhs_dev(Handle *h, std::size_t nrhs, const double *d_B, std::size_t nirs, double *d_X, std::size_t rank) {
  if (nrhs == 1) {
    hifir_dev(h, d_B, nirs, d_X, rank);
    return;
  }
  check_block(h, nrhs);
  if (nirs <= 1) {
    apply_mrhs_dev(h, nrhs, d_B, d_X, rank);
    return;
  }
  if (!h->has_A) throw std::logic_error("iterative refinement needs the matrix: call lhfdGpuSetMatrix first");
  const std::size_t nn = h->n0() * nrhs;
  ensure(h, h->kb_r, nn);
  ensure(h, h->kb_t, nn);
  const ColShape s = col_shape(h->n0(), nrhs);
  apply_mrhs_dev(h, nrhs, d_B, d_X, rank);
  for (std::size_t i = 1; i < nirs; ++i) {
    spmv_cols(h, s, d_X, d_B, nullptr, h->kb_t.p);  // T = B - A X
    apply_mrhs_dev(h, nrhs, h->kb_t.p, h->kb_r.p, rank);
    add_kernel<<<kEW, kRT, 0, h->stream>>>(static_cast<unsigned>(nn), h->kb_r.p, d_X, d_X);
    HIF_KERNEL_CHECK();
    ++h->launch_count;
  }
}

// nrhs independent gmres_hif / fgmres_hifir runs in lockstep.  Every column starts the first cycle; a column
// leaves krylov_dev's inner loop before j + 1 == restart only when it terminates for good, so all columns still
// active share it_outer, j, iter and nirs = 2^it_outer: one step is one block apply (FGMRES: one block
// refinement), one block SpMV and one block Gram-Schmidt sweep, and the host runs the Givens rotations and the
// stopping tests per column with krylov_dev's arithmetic.  A column that terminates is retired in the device
// mask: its next basis vector is zeroed, it stays exact zeros in every later SpMV, reduction and division, and
// the solution updates of later cycles leave its x untouched.  No NaN or Inf is formed in a retired column.
void krylov_mrhs_dev(Handle *h, bool flexible, std::size_t nrhs, const double *d_B, int restart, double rtol, int maxit,
                     bool full_rank, double *d_X, int *flag_out, int *iters_out, int *nmv_out) {
  if (nrhs == 1) {
    krylov_dev(h, flexible, d_B, restart, rtol, maxit, full_rank, d_X, flag_out, iters_out, nmv_out);
    return;
  }
  check_krylov_mrhs(h, nrhs, restart);
  const std::size_t n = h->n0(), nc = nrhs, nn = n * nc, R1 = static_cast<std::size_t>(restart);
  const std::size_t rr = full_rank ? static_cast<std::size_t>(-1) : 0;
  const ColShape    s  = col_shape(n, nc);
  ensure_cols_scal(h, nc);
  ensure(h, h->kb_H, (R1 + 1) * nc);
  ensure(h, h->kb_y, R1 * nc);
  std::vector<double> beta0(nc), beta(nc);
  std::vector<int>    active(nc, 1);
  upload(h, h->kb_mask.p, active);
  norm2_cols(h, s, d_B, h->kb_mask.p, beta0.data());
  HIF_CUDA(cudaMemsetAsync(d_X, 0, nn * sizeof(double), h->stream));
  std::size_t nactive = 0;
  for (std::size_t c = 0; c < nc; ++c) {
    flag_out[c] = iters_out[c] = nmv_out[c] = 0;
    active[c]                               = beta0[c] != 0.0;  // b = 0: x = 0, nothing to iterate
    nactive += active[c];
  }
  if (!nactive) return;
  upload(h, h->kb_mask.p, active);
  ensure(h, h->kb_v, nn);
  ensure(h, h->kb_Q, nn * R1);
  if (flexible)
    ensure(h, h->kb_Z, nn * R1);
  else
    ensure(h, h->kb_w, nn);
  double *v = h->kb_v.p, *w = h->kb_w.p, *Q = h->kb_Q.p, *Z = h->kb_Z.p, *dH = h->kb_H.p;
  int *   mask = h->kb_mask.p;
  // per-column host state of krylov_dev: y, w2, R, J, resid; jc = the last step of the column in this cycle
  std::vector<double> y(nc * (R1 + 1), 0.0), w2(R1, 0.0), Rm(nc * R1 * R1, 0.0), J(nc * 2 * R1, 0.0), resid(nc, 1.0);
  std::vector<double> Hh((R1 + 1) * nc), yd(R1 * nc);
  std::vector<int>    jc(nc, -1), in_cycle(nc, 0);
  const int           max_outer = static_cast<int>(std::ceil(static_cast<double>(maxit) / restart));
  int                 iter      = 0;
  for (int it_outer = 0; it_outer < max_outer; ++it_outer) {
    if (iter)
      spmv_cols(h, s, d_X, d_B, mask, v);  // v = b - A x
    else
      HIF_CUDA(cudaMemcpyAsync(v, d_B, nn * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    norm2_cols(h, s, v, mask, beta.data());
    for (std::size_t c = 0; c < nc; ++c) {
      in_cycle[c] = active[c];
      jc[c]       = -1;
      y[c * (R1 + 1)] = beta[c];
    }
    upload(h, h->kb_red.p + 2 * nc, beta);  // Q(:,0) = v / beta
    div_cols_kernel<<<s.ew(), kRT, 0, h->stream>>>(s.n, s.nc, s.cw, v, h->kb_red.p + 2 * nc, false, mask, Q);
    HIF_KERNEL_CHECK();
    ++h->launch_count;
    int               j    = 0;
    const std::size_t nirs = static_cast<std::size_t>(1) << it_outer;
    for (;;) {
      const double *qj = Q + j * nn;
      if (flexible) {
        double *zj = Z + j * nn;
        hifir_mrhs_dev(h, nrhs, qj, nirs, zj, rr);
        spmv_cols(h, s, zj, nullptr, mask, v);
      } else {
        apply_mrhs_dev(h, nrhs, qj, w, rr);
        spmv_cols(h, s, w, nullptr, mask, v);
      }
      for (std::size_t c = 0; c < nc; ++c)
        if (active[c]) nmv_out[c] += flexible ? static_cast<int>(nirs) : 1;
      // modified Gram-Schmidt (gmres.hpp:174-177): H[0] = <v, q_0>, then per k one fused launch; ||v||^2 -> H[j+1]
      reduce_cols<0>(h, s, v, Q, nullptr, mask, dH);
      for (int k = 0; k <= j; ++k) {
        const double *qk    = Q + k * nn;
        const double *qnext = k < j ? qk + nn : v;
        mgs_step_cols_kernel<<<s.red(), kRT, 0, h->stream>>>(s.n, s.nc, s.cw, dH + k * nc, qk, qnext, v, mask,
                                                             h->kb_part.p, h->kb_count.p, dH + (k + 1) * nc);
        HIF_KERNEL_CHECK();
        ++h->launch_count;
      }
      if (j + 1 < restart) {
        div_cols_kernel<<<s.ew(), kRT, 0, h->stream>>>(s.n, s.nc, s.cw, v, dH + (j + 1) * nc, true, mask, Q + (j + 1) * nn);
        HIF_KERNEL_CHECK();
        ++h->launch_count;
      }
      HIF_CUDA(cudaMemcpyAsync(Hh.data(), dH, (j + 2) * nc * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
      HIF_CUDA(cudaStreamSynchronize(h->stream));
      bool retired = false, cont = false;
      for (std::size_t c = 0; c < nc; ++c) {
        if (!active[c]) continue;
        double *yc = &y[c * (R1 + 1)], *Jc = &J[c * 2 * R1], *Rc = &Rm[c * R1 * R1];
        for (int k = 0; k <= j; ++k) w2[k] = Hh[k * nc + c];
        const double v_norm2 = Hh[(j + 1) * nc + c], v_norm = std::sqrt(v_norm2);
        // Givens rotations (gmres.hpp:184-196), as krylov_dev
        for (int q = 0; q + 1 <= j; ++q) {
          const double tmp = w2[q];
          w2[q]            = Jc[q] * tmp + Jc[restart + q] * w2[q + 1];
          w2[q + 1]        = -Jc[restart + q] * tmp + Jc[q] * w2[q + 1];
        }
        const double rho = std::sqrt(w2[j] * w2[j] + v_norm2);
        Jc[j]            = w2[j] / rho;
        Jc[restart + j]  = v_norm / rho;
        yc[j + 1]        = -Jc[restart + j] * yc[j];
        yc[j]            = Jc[j] * yc[j];
        w2[j]            = rho;
        for (int k = 0; k <= j; ++k) Rc[static_cast<std::size_t>(j) * R1 + k] = w2[k];
        const double resid_prev = resid[c];
        resid[c]                = std::fabs(yc[j + 1]) / beta0[c];
        jc[c]                   = j;
        bool done               = true;
        if (resid[c] >= resid_prev * (1.0 - 1e-8)) {
          flag_out[c] = 1;  // STAGNATED
        } else if (iter >= maxit) {
          flag_out[c] = 2;  // DIVERGED
        } else {
          iters_out[c] = iter + 1;
          if (resid[c] > rtol) {
            done = false;
            if (j + 1 < restart) cont = true;
          }
        }
        if (done) {
          iters_out[c] = flag_out[c] ? iter : iter + 1;
          active[c]    = 0;
          retired      = true;
        }
      }
      ++iter;  // every column still active passed the tests: they share the count
      if (!cont) break;
      if (retired) {  // the retired columns' next basis vector was already formed: zero it
        upload(h, mask, active);
        zero_cols_kernel<<<s.ew(), kRT, 0, h->stream>>>(s.n, s.nc, s.cw, mask, Q + (j + 1) * nn);
        HIF_KERNEL_CHECK();
        ++h->launch_count;
      }
      ++j;
    }
    // back substitution per column with its own last step; y beyond it (and of columns outside the cycle) is 0
    std::fill(yd.begin(), yd.end(), 0.0);
    for (std::size_t c = 0; c < nc; ++c) {
      if (!in_cycle[c]) continue;
      double *yc = &y[c * (R1 + 1)], *Rc = &Rm[c * R1 * R1];
      for (int k = jc[c]; k > -1; --k) {
        yc[k] /= Rc[static_cast<std::size_t>(k) * R1 + k];
        const double tmp = yc[k];
        for (int i = k - 1; i > -1; --i) yc[i] -= tmp * Rc[static_cast<std::size_t>(k) * R1 + i];
      }
      for (int k = 0; k <= jc[c]; ++k) yd[k * nc + c] = yc[k];
    }
    upload(h, h->kb_y.p, yd);
    const unsigned nterms = static_cast<unsigned>(j + 1);
    if (flexible) {  // x += Z(:,0:j) y  (gmres.hpp:223-226)
      axpy_cols_kernel<<<s.ew(), kRT, 0, h->stream>>>(s.n, s.nc, s.cw, nterms, h->kb_y.p, Z, d_X);
      HIF_KERNEL_CHECK();
      ++h->launch_count;
    } else {  // v = Q y ; x += M^{-1} v  (gmres.hpp:111-118)
      HIF_CUDA(cudaMemsetAsync(v, 0, nn * sizeof(double), h->stream));
      axpy_cols_kernel<<<s.ew(), kRT, 0, h->stream>>>(s.n, s.nc, s.cw, nterms, h->kb_y.p, Q, v);
      HIF_KERNEL_CHECK();
      apply_mrhs_dev(h, nrhs, v, w, rr);
      upload(h, mask + nc, in_cycle);
      add_cols_kernel<<<s.ew(), kRT, 0, h->stream>>>(s.n, s.nc, s.cw, mask + nc, w, d_X);
      HIF_KERNEL_CHECK();
      h->launch_count += 2;
    }
    nactive = 0;
    for (std::size_t c = 0; c < nc; ++c) nactive += active[c];
    if (!nactive) break;
    upload(h, mask, active);
  }
  check_sweep_error(h);
}

}  // namespace hifgpu
