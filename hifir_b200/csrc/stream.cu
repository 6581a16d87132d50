// stream.cu -- level-major streaming triangular sweep.
//
// Replaces CCS::solve_as_strict_lower / solve_as_strict_upper of the reference
// (ds/CompressedStorage.hpp:2267-2279, 2356-2369) on the merged factors of merge.cu, whose
// dependency depth is ~50-150 instead of 700-2500.
//
// With so few level sets the factor can be laid out LEVEL-MAJOR and the sweep becomes a
// sequence of sparse matrix-vector products that overlap freely:
//   * rows are sorted by (level set, row length); 32 consecutive rows form a SLICE that one
//     warp solves (sliced ELL: entry k of the 32 rows is one coalesced 128 B + 256 B
//     transaction, rows of a slice have (nearly) equal length, a slice never straddles
//     two level sets);
//   * the factor is streamed straight from HBM with evict-first loads, exactly once;
//   * the solution lives in the tagged buffers of common.cuh (value + ready bit in one
//     word).  A lane gathers its dependencies OPTIMISTICALLY from L2 -- several in flight --
//     and re-polls only the ones that are not ready yet.  Entries are ordered by the level
//     of their producer, so all but the last are ready on the first try.  No flags, no
//     fences, no grid barriers, no per-level launches;
//   * slices are handed out through a ticket counter in level order: everything a warp can
//     wait for belongs to an earlier ticket, i.e. to a resident or finished warp (no
//     deadlock whatever the CTA placement).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <numeric>

#include "hifgpu.h"

namespace hifgpu {

constexpr unsigned kStreamWarps = 8;  // slices per ticket = warps per CTA
constexpr unsigned kPadCol      = 0xffffffffu;
constexpr unsigned kPadCode     = 0xffffffffu;
constexpr unsigned kEmptySlice  = 0xffffffffu;  // sdesc.z of a padding slice (its warp idles)

__device__ __forceinline__ unsigned ld_stream_u32(const unsigned *p) {
  unsigned v;
  asm volatile("ld.global.cs.u32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ double ld_stream_f64(const double *p) {
  double v;
  asm volatile("ld.global.cs.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ float ld_stream_f32(const float *p) {
  float v;
  asm volatile("ld.global.cs.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ double ld_stream_val(const double *p) { return ld_stream_f64(p); }
__device__ __forceinline__ float  ld_stream_val(const float *p) { return ld_stream_f32(p); }
__device__ __forceinline__ int ld_poll_i32(const int *p) {
  int v;
  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long stream_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void ld_poll_v2(const unsigned long long *p, unsigned long long &a, unsigned long long &b) {
  asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ void st_publish_v2(unsigned long long *p, unsigned long long a, unsigned long long b) {
  asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(a), "l"(b) : "memory");
}

// sync layout (ints, zeroed once per apply): [0] ticket counter, [16] frontier hint (highest
// completed level set + 1), [kSyncStride * (1 + l)] finished chunks of level set l (one 128-byte
// line per counter: the pollers of different levels hit different L2 slices).  The level counters
// only THROTTLE: the warps of a chunk of level l first pull their share of the factor from HBM
// into registers (it depends on nothing), then wait until level l - window is complete before
// they touch the solution buffer, so that at most `window` level sets poll it at any time
// (thousands of run-ahead warps spinning on L2 would starve the producers).  Correctness never
// depends on the counters -- readiness is carried by the tagged values -- so they need no fences.
//
// Slice s (one warp): 32 / lpr rows, lpr = 2^sd.z lanes per row (long rows are spread over
// several lanes and reduced with shuffles); entry k of lane j at cols/vals[(sd.x + k) * 32 + j].
// Chunk c (one CTA round) = slices [8c, 8c + 8), all of one level set (sd.w).
//
// NR right-hand sides per row (row-interleaved, X[i*NR + c], the Array<std::array<T,Nrhs>>
// layout of hif::HIF::solve_mrhs, builder.hpp:433-445; per-column arithmetic =
// CCS::solve_as_strict_lower/upper_mrhs, CompressedStorage.hpp:2286-2301, 2376-2393): a lane keeps
// NR accumulators, a dependency is ONE 64-byte gather (NR = 8) instead of eight 8-byte ones, and
// the factor is streamed once for all NR columns.  Same plan (sliced ELL) as for NR = 1.
//
// kU entries per lane are held in registers; their gathers go out kG at a time.  Measured at
// 128^3 (ms per apply): kU = 4 / 5 CTAs per SM 1.58, kU = 8 / kG = 4 / 4 CTAs 1.37 (the optimum:
// 2, 3, 5, 6 CTAs per SM, kU = 16 and shared-memory staging of the entries are all slower).
//
// VT = storage type of the factor values: double, or float for the factors of a single-precision
// hif::HIF<float> (lhfsGpu* / lhfsdGpu* entry points) -- 8 instead of 12 bytes per streamed entry;
// the arithmetic and the solution stay in double whatever VT.
template <bool UPPER, int kU, int NR, bool kTrace, class VT>
__global__ void __launch_bounds__(kStreamWarps * 32, NR > 1 ? 2 : (kU == 4 ? 5 : 4))
    sweep_stream_kernel(const unsigned nchunks, const uint4 *__restrict__ sdesc, const unsigned *__restrict__ lvl_need,
                        const unsigned *__restrict__ codes, const unsigned *__restrict__ cols,
                        const VT *__restrict__ vals, const unsigned m, const double *__restrict__ rhs_plain,
                        const unsigned long long *rhs_tagged, const double *__restrict__ diag, unsigned long long *x,
                        const unsigned parity, int *sync, int *error_flag, const unsigned window,
                        const unsigned adm_sleep, const int publish_st, unsigned long long *trace_buf) {
  unsigned long long *const trace = kTrace ? trace_buf : nullptr;  // the production variant carries no tracing code
  static_assert(NR == 1 || NR % 2 == 0, "NR must be 1 or even (128-bit transactions)");
  constexpr int kG = NR == 1 ? (kU > 4 ? 4 : kU) : 2;  // entries whose gathers are in flight together
  static_assert(kU % kG == 0, "kU must be a multiple of the gather group");
  __shared__ unsigned s_c[2];
  __shared__ int      s_last;
  const unsigned      warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  if (threadIdx.x == 0) {
    s_last = -1;
    s_c[0] = static_cast<unsigned>(atomicAdd(sync, 1));
  }
  unsigned f_seen = 0;  // thread 0: highest completed level + 1 it has reported
  for (unsigned round = 0;; ++round) {
    __syncthreads();  // every warp of the previous chunk has published; s_c[round & 1] is written
    if (threadIdx.x == 0 && s_last >= 0) atomicAdd(sync + kSyncStride * (1 + s_last), 1);  // fire and forget
    const unsigned c = s_c[round & 1u];
    if (c >= nchunks) break;
    if (trace && threadIdx.x == 0) trace[8 * c + 0] = stream_timer_ns();
    const unsigned s    = c * kStreamWarps + warp;
    const uint4    sd   = sdesc[s];  // x: offset (units of 32 entries), y: entries per lane, z: log2 lanes per row, w: level
    const bool     idle = sd.z == kEmptySlice;  // padding slice of a spread-out thin level set
    const unsigned code = idle ? kPadCode : codes[static_cast<std::size_t>(s) * 32u + lane];
    const unsigned lpr  = idle ? 1u : 1u << sd.z;
    const bool     act  = code != kPadCode && (lane & (lpr - 1u)) == 0u;  // the lane that owns the row
    const std::size_t slot = static_cast<std::size_t>(code & kCodeSlotMask);
    const std::size_t base = static_cast<std::size_t>(sd.x) * 32u + lane;
    const unsigned    len  = sd.y;
    // ---- everything that does not depend on other rows: factor entries, right-hand side
    unsigned cc[kU];
    VT       vv[kU];
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      cc[u] = kPadCol;
      if (static_cast<unsigned>(u) < len) {
        cc[u] = ld_stream_u32(cols + base + static_cast<std::size_t>(u) * 32u);
        vv[u] = ld_stream_val(vals + base + static_cast<std::size_t>(u) * 32u);
      }
    }
    double acc[NR];
#pragma unroll
    for (int q = 0; q < NR; ++q) acc[q] = 0.0;
    if (act && !(code & kCodeZeroRhs)) {
      // b_i (L sweep) or (L^{-1} b)_i / d_i with a true division (prec_solve.hpp:219, :256-259)
      // for the U sweep; slots >= m are the auxiliary unknowns of merge.cu
      const std::size_t ri = slot >= m ? slot - m : slot;
      if (UPPER) {
        const double d = diag[ri];
#pragma unroll
        for (int q = 0; q < NR; ++q) acc[q] = tag_value(rhs_tagged[ri * NR + q]) / d;
      } else {
#pragma unroll
        for (int q = 0; q < NR; ++q) acc[q] = rhs_plain[ri * NR + q];
      }
    }
    // ---- admission: level sd.w - window complete (thread 0 polls for the CTA).  Far-away
    // waiters sleep in proportion to their distance from the frontier hint and only look at
    // that one word, the waiters of the next levels spin on their counter
    if (threadIdx.x == 0) {
      s_last = static_cast<int>(sd.w);
      if (trace) {
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        trace[8 * c + 1] = stream_timer_ns();  // factor entries requested
        trace[8 * c + 4] = sd.w;
        trace[8 * c + 5] = smid;
      }
      if (sd.w >= window) {
        const unsigned t     = sd.w - window;
        const unsigned need  = lvl_need[t];
        const int *    ctr   = sync + kSyncStride * (1 + t);
        unsigned       spins = 0;
        // common case (wide level sets): the level is complete already -- one load
        while (static_cast<unsigned>(ld_poll_i32(ctr)) < need) {
          const unsigned f = static_cast<unsigned>(ld_poll_i32(sync + 16));  // levels [0, f) are known to be done
          if (t < f + 2u) {
            while (static_cast<unsigned>(ld_poll_i32(ctr)) < need) {
              if (++spins > (kSpinLimit >> 4)) {
                *error_flag = 1;
                break;
              }
            }
            break;
          }
          __nanosleep(min((t - f) * adm_sleep, 20000u));
          if (++spins > (kSpinLimit >> 4)) {
            *error_flag = 1;
            break;
          }
        }
        if (t + 1u > f_seen) {  // advance the hint
          f_seen = t + 1u;
          atomicMax(sync + 16, static_cast<int>(f_seen));
        }
      }
      if (trace) trace[8 * c + 2] = stream_timer_ns();  // admitted
    }
    __syncthreads();
    // the next ticket is fetched behind the gathers of this chunk (off the critical path); it is
    // held for the ~1 us this chunk still needs, which delays nobody
    unsigned   next_ticket = 0;
    const bool ticket_lane = threadIdx.x == 32u;
    // ---- gather the dependencies optimistically, re-poll the ones that are not ready
    auto gather = [&](unsigned col, unsigned long long(&g)[NR]) {
      const unsigned long long *src = x + static_cast<std::size_t>(col) * NR;
      if (NR == 1) {
        g[0] = ld_poll(src);
      } else {
#pragma unroll
        for (int q = 0; q < NR; q += 2) ld_poll_v2(src + q, g[q], g[q + 1]);
      }
    };
    auto ready = [&](const unsigned long long(&g)[NR]) {
      bool ok = true;
#pragma unroll
      for (int q = 0; q < NR; ++q) ok &= tag_ready(g[q], parity);
      return ok;
    };
    for (unsigned k = 0;;) {
#pragma unroll
      for (int u0 = 0; u0 < kU; u0 += kG) {
        unsigned long long g[kG][NR];
#pragma unroll
        for (int j = 0; j < kG; ++j)
          if (cc[u0 + j] != kPadCol) gather(cc[u0 + j], g[j]);
        if (ticket_lane && k == 0 && u0 == 0) next_ticket = static_cast<unsigned>(atomicAdd(sync, 1));
        if (trace && threadIdx.x == 0 && k == 0 && u0 == 0) {  // warp 0: first gather round trip
          unsigned long long any = 0;
#pragma unroll
          for (int j = 0; j < kG; ++j)
            if (cc[j] != kPadCol) any |= g[j][0];
          trace[8 * c + 6] = stream_timer_ns() + (any == 0x7ff8dead00000001ull ? 1u : 0u);
        }
        // entries that were not ready on the first try (padding counts as ready) are re-polled
        // TOGETHER, round by round: one L2 round trip per round whatever their number
        unsigned pend = 0;
#pragma unroll
        for (int j = 0; j < kG; ++j)
          if (cc[u0 + j] != kPadCol && !ready(g[j])) pend |= 1u << j;
        for (unsigned rounds = 0; __any_sync(0xffffffffu, pend != 0u);) {
#pragma unroll
          for (int j = 0; j < kG; ++j)
            if (pend & (1u << j)) gather(cc[u0 + j], g[j]);
#pragma unroll
          for (int j = 0; j < kG; ++j)
            if ((pend & (1u << j)) && ready(g[j])) pend &= ~(1u << j);
          if (++rounds > (kSpinLimit >> 3)) {  // hang guard: flag the error, go on with garbage
            *error_flag = 1;
            break;
          }
        }
#pragma unroll
        for (int j = 0; j < kG; ++j)
          if (cc[u0 + j] != kPadCol) {
#pragma unroll
            for (int q = 0; q < NR; ++q) acc[q] = fma(-static_cast<double>(vv[u0 + j]), tag_value(g[j][q]), acc[q]);
          }
      }
      k += kU;
      if (k >= len) break;
#pragma unroll
      for (int u = 0; u < kU; ++u) {  // rows longer than kU * lpr entries (rare)
        cc[u] = kPadCol;
        if (k + u < len) {
          cc[u] = ld_stream_u32(cols + base + static_cast<std::size_t>(k + u) * 32u);
          vv[u] = ld_stream_val(vals + base + static_cast<std::size_t>(k + u) * 32u);
        }
      }
    }
    if (trace && threadIdx.x == 0) trace[8 * c + 7] = stream_timer_ns();  // warp 0: all dependencies consumed
    for (unsigned o = lpr >> 1; o > 0; o >>= 1) {
#pragma unroll
      for (int q = 0; q < NR; ++q) acc[q] += __shfl_xor_sync(0xffffffffu, acc[q], o);
    }
    if (act) {
      if (NR == 1) {
        if (!publish_st) {
          // publish through the L2 atomic unit: an exchange is visible to the pollers ~0.2 us
          // earlier than a plain store (measured: 1.81 -> 1.64 ms per apply at 128^3)
          unsigned long long old;
          asm volatile("atom.relaxed.gpu.global.exch.b64 %0, [%1], %2;"
                       : "=l"(old)
                       : "l"(x + slot), "l"(tag_set(acc[0], parity))
                       : "memory");
        } else {
          st_publish(x + slot, tag_set(acc[0], parity));
        }
      } else {
#pragma unroll
        for (int q = 0; q < NR; q += 2)
          st_publish_v2(x + slot * NR + q, tag_set(acc[q], parity), tag_set(acc[q + 1 < NR ? q + 1 : q], parity));
      }
    }
    if (trace && lane == 0) atomicMax(trace + 8 * c + 3, stream_timer_ns());  // last warp published
    if (ticket_lane) s_c[(round + 1u) & 1u] = next_ticket;
  }
}

// ---- host: sweep form -> level-major sliced ELL ------------------------------------
namespace {
struct StreamHost {
  std::vector<unsigned> lvl_need;  // chunks per level set
  std::vector<uint4>    sdesc;     // slices, 8 per chunk
  std::vector<unsigned> codes, cols;
  std::vector<double>   vals;
  std::size_t           padded = 0;
  unsigned              depth = 0;
};

// lanes per row (2^z <= R) so that a lane holds <= U entries if possible
unsigned lanes_log2_for(unsigned len, unsigned U, unsigned R) {
  unsigned z = 0;
  while ((2u << z) <= R && ((len + (1u << z) - 1u) >> z) > U) ++z;
  return z;
}
unsigned stream_unroll() {
  const char *e = std::getenv("HIFIR_B200_STREAM_U");
  return e && std::atoi(e) == 4 ? 4u : 8u;  // measured at 128^3: 4 -> 1.58 ms, 8 -> 1.37 ms per apply
}

void pack_stream(const HostCsr &S, StreamHost &H, unsigned U, unsigned R = 32u) {
  const unsigned m = static_cast<unsigned>(S.nrows);
  if (!m) return;
  if (S.gid.size() != m) throw std::logic_error("build_stream_plan: factor is not in sweep form");
  validate_sweep_form(S);
  std::vector<uint4> &   sdesc = H.sdesc;
  std::vector<unsigned> &codes = H.codes, &cols = H.cols;
  std::vector<double> &  vals = H.vals;
  std::vector<unsigned> lev(m, 0u);
  unsigned              depth = 0;
  for (unsigned i = 0; i < m; ++i) {
    unsigned l = 0;
    for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k) l = std::max(l, lev[S.col[k]] + 1u);
    lev[i] = l;
    depth  = std::max(depth, l + 1u);
  }
  auto rowlen = [&](unsigned i) { return S.ptr[i + 1] - S.ptr[i]; };
  std::vector<unsigned> ord(m);
  std::iota(ord.begin(), ord.end(), 0u);
  std::stable_sort(ord.begin(), ord.end(), [&](unsigned a, unsigned b) {
    if (lev[a] != lev[b]) return lev[a] < lev[b];
    return rowlen(a) > rowlen(b);
  });
  std::vector<unsigned> ent;
  cols.reserve(S.col.size() + S.col.size() / 8);
  vals.reserve(S.col.size() + S.col.size() / 8);
  H.lvl_need.assign(depth, 0u);
  std::size_t padded = 0;
  for (unsigned p = 0; p < m;) {
    // one slice: rows of one level set with the same lanes-per-row class
    const unsigned l = lev[ord[p]], z = lanes_log2_for(rowlen(ord[p]), U, R), lpr = 1u << z, cap = R >> z;
    unsigned       cnt = 1;
    while (cnt < cap && p + cnt < m && lev[ord[p + cnt]] == l && lanes_log2_for(rowlen(ord[p + cnt]), U, R) == z) ++cnt;
    const unsigned width = (rowlen(ord[p]) + lpr - 1u) >> z;  // rows are sorted by length: the first is the longest
    sdesc.push_back(make_uint4(static_cast<unsigned>(cols.size() / R), width, z, l));
    const std::size_t c0 = cols.size();
    cols.resize(c0 + static_cast<std::size_t>(width) * R, kPadCol);
    vals.resize(c0 + static_cast<std::size_t>(width) * R, 0.0);
    for (unsigned r = 0; r < cap; ++r) {
      if (r >= cnt) {
        for (unsigned j = 0; j < lpr; ++j) codes.push_back(kPadCode);
        continue;
      }
      const unsigned i = ord[p + r];
      for (unsigned j = 0; j < lpr; ++j) codes.push_back(S.gid[i]);
      const unsigned b = S.ptr[i], e = S.ptr[i + 1];
      // entries in the order their producers finish (level set); ties: the reference's order
      ent.resize(e - b);
      std::iota(ent.begin(), ent.end(), b);
      std::stable_sort(ent.begin(), ent.end(), [&](unsigned x, unsigned y) { return lev[S.col[x]] < lev[S.col[y]]; });
      for (unsigned q = 0; q < e - b; ++q) {  // entry q of the row -> lane r*lpr + q%lpr, position q/lpr
        const std::size_t at = c0 + static_cast<std::size_t>(q >> z) * R + r * lpr + (q & (lpr - 1u));
        cols[at]             = S.gid[S.col[ent[q]]] & kCodeSlotMask;
        vals[at]             = S.val[ent[q]];
      }
      padded += static_cast<std::size_t>(width) * lpr - (e - b);
    }
    p += cnt;
  }
  // ---- chunks: 8 slice descriptors each (one per warp of a CTA), all of one level set.  A
  // thin level set is spread over as many CTAs (SMs) as possible -- an SM serves one L2 request
  // per clock, so the gathers of a full chunk alone take ~1 us -- a wide one uses full chunks.
  {
    const char *          es          = std::getenv("HIFIR_B200_STREAM_SPREAD");
    const bool            spread_thin = !es || std::atoi(es) != 0;
    std::vector<uint4>    sd2;
    std::vector<unsigned> cd2;
    const std::size_t     ns = sdesc.size();
    sd2.reserve(ns + ns / 4);
    cd2.reserve(codes.size() + codes.size() / 4);
    for (std::size_t s0 = 0; s0 < ns;) {
      const unsigned l  = sdesc[s0].w;
      std::size_t    s1 = s0;
      while (s1 < ns && sdesc[s1].w == l) ++s1;
      const std::size_t S = s1 - s0;
      // up to 4 SMs' worth of slices: one chunk per SM, beyond: full chunks (throughput matters)
      const unsigned spc = (S > 4u * kNumSMs || !spread_thin) ? kStreamWarps
                                            : static_cast<unsigned>(std::max<std::size_t>(1, (S + kNumSMs - 1) / kNumSMs));
      for (std::size_t s = s0; s < s1; s += spc) {
        for (unsigned w = 0; w < kStreamWarps; ++w) {
          if (w < spc && s + w < s1) {
            sd2.push_back(sdesc[s + w]);
            cd2.insert(cd2.end(), codes.begin() + (s + w) * R, codes.begin() + (s + w + 1) * R);
          } else {
            sd2.push_back(make_uint4(0u, 0u, kEmptySlice, l));
            cd2.insert(cd2.end(), R, kPadCode);
          }
        }
        ++H.lvl_need[l];
      }
      s0 = s1;
    }
    sdesc.swap(sd2);
    codes.swap(cd2);
  }
  if (cols.size() / R > 0xffffffffull) throw std::length_error("stream plan too large");
  H.padded = padded;
  H.depth  = depth;
}
}  // namespace

void build_stream_plan(const HostCsr &S, bool upper, SweepPlan &plan, std::size_t *tally) {
  plan.stream  = true;
  plan.upper   = upper;
  plan.nr      = 1;  // the same plan serves the multi-rhs kernel (launch_stream_sweep, nr = kMrhsWidth)
  plan.m       = static_cast<unsigned>(S.orig_rows);
  plan.nblocks = 0;
  if (!S.nrows) return;
  StreamHost H;
  plan.st_u = stream_unroll();
  pack_stream(S, H, plan.st_u);
  plan.nblocks    = static_cast<unsigned>(H.sdesc.size());  // slices
  plan.slab_bytes = H.cols.size() * (plan.f32 ? 8u : 12u) + H.codes.size() * 4u + H.sdesc.size() * 16u;
  plan.st_depth   = H.depth;
  plan.st_padded  = H.padded;
  plan.st_chunks  = static_cast<unsigned>(H.sdesc.size() / kStreamWarps);
  plan.st_need.upload(H.lvl_need, tally);
  plan.st_sdesc.upload(reinterpret_cast<const unsigned *>(H.sdesc.data()), H.sdesc.size() * 4u, tally);
  plan.st_codes.upload(H.codes, tally);
  plan.st_cols.upload(H.cols, tally);
  if (plan.f32) {  // single-precision factors: the merged values are rounded to float once, here
    std::vector<float> v32(H.vals.begin(), H.vals.end());
    plan.st_vals32.upload(v32, tally);
  } else {
    plan.st_vals.upload(H.vals, tally);
  }
}

namespace {
// CPU emulation of the streaming sweep on packed arrays (slices in ticket order = level order, rows of a slice
// one after the other), in the device's arithmetic order: per-lane fma over the entries, then the shfl_xor
// tree.  `x` has 2 * m slots.  parity < 0: plain values; 0 / 1: every published value goes through tag_set
// before any consumer reads it, and the right-hand side of an upper sweep (on the device the L sweep's
// tagged result) is tagged as well.
void stream_emulate_packed(const uint4 *sdesc, std::size_t nslices, const unsigned *codes, const unsigned *cols,
                           const double *vals, unsigned m, bool upper, const double *rhs, const double *diag, double *x,
                           int parity) {
  auto pub = [&](double v) { return parity < 0 ? v : tag_set_host(v, static_cast<unsigned>(parity)); };
  for (std::size_t s = 0; s < nslices; ++s) {
    const uint4 sd = sdesc[s];
    if (sd.z == kEmptySlice) continue;
    const std::size_t base = static_cast<std::size_t>(sd.x) * 32u;
    const unsigned    lpr  = 1u << sd.z;
    for (unsigned lane = 0; lane < 32u; lane += lpr) {
      const unsigned code = codes[s * 32u + lane];
      if (code == kPadCode) continue;
      const unsigned slot = code & kCodeSlotMask, ri = slot >= m ? slot - m : slot;
      double         part[32];
      for (unsigned j = 0; j < lpr; ++j) {  // per-lane partial sums, then the shuffle tree
        double acc = (j == 0 && !(code & kCodeZeroRhs)) ? (upper ? pub(rhs[ri]) / diag[ri] : rhs[ri]) : 0.0;
        for (unsigned k = 0; k < sd.y; ++k) {
          const unsigned c = cols[base + static_cast<std::size_t>(k) * 32u + lane + j];
          if (c != kPadCol) acc = std::fma(-vals[base + static_cast<std::size_t>(k) * 32u + lane + j], x[c], acc);
        }
        part[j] = acc;
      }
      for (unsigned o = lpr >> 1; o > 0; o >>= 1)
        for (unsigned j = 0; j < o; ++j) part[j] += part[j + o];
      x[slot] = pub(part[0]);
    }
  }
}
}  // namespace

// CPU emulation of the streaming sweep on the packed data: lets tests check merge + packing without a GPU.
// `x` has 2 * orig_rows slots.  stats = {slices, padded entries, bytes, depth}
void stream_host_emulate(const HostCsr &S, bool upper, const double *rhs, const double *diag, double *x,
                         std::size_t stats[4], bool f32, int parity) {
  StreamHost H;
  pack_stream(S, H, stream_unroll());
  if (f32)  // single-precision factors: the packed values are rounded to float (build_stream_plan)
    for (double &v : H.vals) v = static_cast<double>(static_cast<float>(v));
  stream_emulate_packed(H.sdesc.data(), H.sdesc.size(), H.codes.data(), H.cols.data(), H.vals.data(),
                        static_cast<unsigned>(S.orig_rows), upper, rhs, diag, x, parity);
  stats[0] = H.sdesc.size();
  stats[1] = H.padded;
  stats[2] = H.cols.size() * 12u + H.codes.size() * 4u + H.sdesc.size() * 16u;
  stats[3] = H.depth;
}

// the same on the arrays of a plan copied back from the device (float values widened, as the kernel does)
void stream_emulate_device_plan(const SweepPlan &plan, const double *rhs, const double *diag, double *x, unsigned parity) {
  if (!plan.nblocks) return;
  std::vector<uint4>    sdesc(plan.st_sdesc.n / 4u);
  std::vector<unsigned> codes(plan.st_codes.n), cols(plan.st_cols.n);
  std::vector<double>   vals(plan.f32 ? plan.st_vals32.n : plan.st_vals.n);
  if (codes.size() < sdesc.size() * 32u || vals.size() != cols.size()) throw std::logic_error("streaming plan: array sizes");
  HIF_CUDA(cudaMemcpy(sdesc.data(), plan.st_sdesc.p, sdesc.size() * sizeof(uint4), cudaMemcpyDeviceToHost));
  HIF_CUDA(cudaMemcpy(codes.data(), plan.st_codes.p, codes.size() * 4u, cudaMemcpyDeviceToHost));
  HIF_CUDA(cudaMemcpy(cols.data(), plan.st_cols.p, cols.size() * 4u, cudaMemcpyDeviceToHost));
  if (plan.f32) {
    std::vector<float> v32(vals.size());
    HIF_CUDA(cudaMemcpy(v32.data(), plan.st_vals32.p, v32.size() * 4u, cudaMemcpyDeviceToHost));
    std::copy(v32.begin(), v32.end(), vals.begin());
  } else {
    HIF_CUDA(cudaMemcpy(vals.data(), plan.st_vals.p, vals.size() * 8u, cudaMemcpyDeviceToHost));
  }
  stream_emulate_packed(sdesc.data(), sdesc.size(), codes.data(), cols.data(), vals.data(), plan.m, plan.upper, rhs, diag, x,
                        static_cast<int>(parity));
}

namespace {
int stream_env(const char *name, int dflt) {
  const char *e = std::getenv(name);
  return e ? std::atoi(e) : dflt;
}
template <bool UPPER, int kU, int NR, class VT>
void launch_stream_V(Handle *h, const SweepPlan &plan, const VT *vals, const double *rhs_plain,
                     const unsigned long long *rhs_tagged, const double *diag, unsigned long long *x, unsigned parity,
                     int *sync, unsigned long long *trace) {
  static int ctas_per_sm = 0;
  if (!ctas_per_sm) {
    HIF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, sweep_stream_kernel<UPPER, kU, NR, false, VT>,
                                                           static_cast<int>(kStreamWarps * 32), 0));
    if (ctas_per_sm < 1) ctas_per_sm = 1;
  }
  const unsigned window = static_cast<unsigned>(std::max(1, stream_env("HIFIR_B200_STREAM_WINDOW", 3)));
  const unsigned sleep  = static_cast<unsigned>(std::max(20, stream_env("HIFIR_B200_STREAM_SLEEP", 300)));
  const int      pub_st = stream_env("HIFIR_B200_STREAM_PUBLISH_ST", 0);
  const unsigned grid   = std::min<unsigned>(plan.st_chunks + 1u, static_cast<unsigned>(kNumSMs * ctas_per_sm));
  const uint4 *  sdesc  = reinterpret_cast<const uint4 *>(plan.st_sdesc.p);
  if (trace)
    sweep_stream_kernel<UPPER, kU, NR, true, VT><<<grid, kStreamWarps * 32, 0, h->stream>>>(
        plan.st_chunks, sdesc, plan.st_need.p, plan.st_codes.p, plan.st_cols.p, vals, plan.m, rhs_plain, rhs_tagged,
        diag, x, parity, sync, h->error_flag.p, window, sleep, pub_st, trace);
  else
    sweep_stream_kernel<UPPER, kU, NR, false, VT><<<grid, kStreamWarps * 32, 0, h->stream>>>(
        plan.st_chunks, sdesc, plan.st_need.p, plan.st_codes.p, plan.st_cols.p, vals, plan.m, rhs_plain, rhs_tagged,
        diag, x, parity, sync, h->error_flag.p, window, sleep, pub_st, nullptr);
}
template <bool UPPER, int kU, int NR>
void launch_stream_T(Handle *h, const SweepPlan &plan, const double *rhs_plain, const unsigned long long *rhs_tagged,
                     const double *diag, unsigned long long *x, unsigned parity, int *sync, unsigned long long *trace) {
  if (plan.f32)
    launch_stream_V<UPPER, kU, NR, float>(h, plan, plan.st_vals32.p, rhs_plain, rhs_tagged, diag, x, parity, sync, trace);
  else
    launch_stream_V<UPPER, kU, NR, double>(h, plan, plan.st_vals.p, rhs_plain, rhs_tagged, diag, x, parity, sync, trace);
}
template <bool UPPER>
void launch_stream_U(Handle *h, const SweepPlan &plan, const double *rhs_plain, const unsigned long long *rhs_tagged,
                     const double *diag, unsigned long long *x, unsigned parity, int *sync, unsigned long long *trace,
                     unsigned nr) {
  if (nr != 1u && nr != kMrhsWidth) throw std::logic_error("unsupported multi-rhs width");
  constexpr int W = static_cast<int>(kMrhsWidth);
  if (nr == kMrhsWidth && plan.st_u == 4)
    launch_stream_T<UPPER, 4, W>(h, plan, rhs_plain, rhs_tagged, diag, x, parity, sync, trace);
  else if (nr == kMrhsWidth)
    launch_stream_T<UPPER, 8, W>(h, plan, rhs_plain, rhs_tagged, diag, x, parity, sync, trace);
  else if (plan.st_u == 4)
    launch_stream_T<UPPER, 4, 1>(h, plan, rhs_plain, rhs_tagged, diag, x, parity, sync, trace);
  else
    launch_stream_T<UPPER, 8, 1>(h, plan, rhs_plain, rhs_tagged, diag, x, parity, sync, trace);
}
}  // namespace

void launch_stream_sweep(Handle *h, const SweepPlan &plan, const double *rhs_plain,
                         const unsigned long long *rhs_tagged, const double *diag, unsigned long long *x,
                         unsigned parity, int *ticket, unsigned long long *trace, unsigned nr) {
  if (!plan.nblocks) return;
  if (plan.upper)
    launch_stream_U<true>(h, plan, rhs_plain, rhs_tagged, diag, x, parity, ticket, trace, nr);
  else
    launch_stream_U<false>(h, plan, rhs_plain, rhs_tagged, diag, x, parity, ticket, trace, nr);
  HIF_KERNEL_CHECK();
  ++h->launch_count;
}

}  // namespace hifgpu
