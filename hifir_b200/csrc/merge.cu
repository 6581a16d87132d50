// merge.cu -- algebraic level merging of a triangular factor (attach time, host only).
//
// The factors of the reference have dependency depth 700-2500 (SURVEY.md App. A) while a
// sweep moves only ~200 MB: executed row by row, CCS::solve_as_strict_lower / _upper
// (ds/CompressedStorage.hpp:2267-2279, 2356-2369) are bound by the LATENCY of that chain on
// any parallel machine.  The chain is shortened here by an exact reformulation:
//
//   * level sets are grouped into SUPER LEVELS [l0, l1].  Split T = I + N + X with N = the
//     entries that connect two rows of the same super level, X = the rest (they reference
//     earlier super levels).  W = I + N is block diagonal over the super levels and
//       T x = b   <=>   t = b - X x ,  x = W^{-1} t .
//   * W^{-1} = sum_k (-N)^k is formed explicitly, row by row (N is nilpotent of order
//     <= levels per super level).  Its rows stay short because a super level is closed as soon
//     as the fill of the next level set would cost more than the dependent step it saves.
//   * The result is again a unit lower triangular system ("sweep form") in the unknowns
//     [.., t_i, x_i, ..]: a row with in-level dependencies becomes two rows (t_i: the
//     cross-level part, x_i: -t_i - sum_j Winv_ij t_j with zero right-hand side), any other
//     row is unchanged.  The sweep kernels of sptrsv.cu run it as they run the original; its
//     depth is <= 2 per super level instead of one per level set.
//
// Nothing is approximated: the difference to the reference's substitution is rounding only
// (the inverse-based dropping of HIF bounds ||L^{-1}||, ||U^{-1}|| by kappa, so the diagonal
// blocks W are well conditioned).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <stdexcept>
#include <string>

#include "hifgpu.h"

namespace hifgpu {

MergeParams MergeParams::from_env() {
  MergeParams p;
  if (const char *e = std::getenv("HIFIR_B200_MERGE")) p.enabled = std::atoi(e) != 0;
  if (const char *e = std::getenv("HIFIR_B200_MERGE_GAIN")) p.gain = std::atof(e), p.auto_caps = false;
  if (const char *e = std::getenv("HIFIR_B200_MERGE_ROWCAP")) p.row_cap = static_cast<unsigned>(std::atoi(e));
  if (const char *e = std::getenv("HIFIR_B200_MERGE_BMAX")) p.bmax = static_cast<unsigned>(std::atoi(e));
  if (const char *e = std::getenv("HIFIR_B200_MERGE_ROWCOST")) p.row_cost = std::atof(e);
  if (const char *e = std::getenv("HIFIR_B200_MERGE_SLCAP")) p.sl_cap = std::atof(e), p.auto_caps = false;
  if (const char *e = std::getenv("HIFIR_B200_MERGE_ALAP")) p.alap = std::atoi(e);
  if (const char *e = std::getenv("HIFIR_B200_MERGE_CHAIN")) p.chain = std::atoi(e) != 0;
  if (const char *e = std::getenv("HIFIR_B200_MERGE_SLACK")) p.slack = std::atoi(e) != 0;
  if (const char *e = std::getenv("HIFIR_B200_MERGE_CHAINALL")) p.chain_all = std::atoi(e) != 0;
  if (const char *e = std::getenv("HIFIR_B200_MERGE_STEPS")) p.steps = static_cast<unsigned>(std::atoi(e));
  return p;
}

double MergeParams::plan_cost(std::size_t steps, std::size_t entries, std::size_t rows) const {
  const double e = static_cast<double>(entries), r = static_cast<double>(rows);
  const int    k = 12.0 * e + 8.0 * r <= l2_bytes ? 1 : 0;
  return tau_step[k] * static_cast<double>(steps) + c_entry[k] * e;
}

// Rows in sweep order (forward for L, backward for U), every entry references an EARLIER row,
// entries of a row in the order the reference's column sweep applies them.
HostCsr to_sweep_form(const HostCsr &T, bool upper) {
  const unsigned m = static_cast<unsigned>(T.nrows);
  HostCsr        S;
  S.nrows = S.ncols = m;
  S.orig_rows       = m;
  S.gid.resize(m);
  if (!upper) {
    S.ptr = T.ptr;
    S.col = T.col;
    S.val = T.val;
    S.ptr.resize(m + 1, S.ptr.empty() ? 0u : S.ptr.back());
    for (unsigned i = 0; i < m; ++i) S.gid[i] = i;
    return S;
  }
  S.ptr.assign(m + 1, 0u);
  S.col.resize(T.col.size());
  S.val.resize(T.val.size());
  unsigned w = 0;
  for (unsigned s = 0; s < m; ++s) {
    const unsigned i = m - 1u - s;
    S.ptr[s]         = w;
    for (unsigned k = T.ptr[i + 1]; k-- > T.ptr[i];) {
      S.col[w] = static_cast<int>(m - 1u - static_cast<unsigned>(T.col[k]));
      S.val[w] = T.val[k];
      ++w;
    }
    S.gid[s] = i;
  }
  S.ptr[m] = w;
  return S;
}

// A factor in sweep form as the packers need it: row pointers start at 0 and never decrease, every
// entry references an EARLIER row, every row code addresses one of the 2 * orig_rows solution slots
// and no slot is written twice.  (The device sweeps index the solution buffers with these numbers.)
void validate_sweep_form(const HostCsr &S) {
  const std::size_t n = S.nrows;
  if (S.ptr.size() != n + 1 || S.gid.size() != n || S.col.size() != S.val.size())
    throw std::invalid_argument("sweep form: array sizes do not match");
  if (n == 0) return;
  if (S.ptr[0] != 0u || S.ptr[n] != S.col.size()) throw std::invalid_argument("sweep form: bad row pointers");
  std::vector<char> seen(2 * S.orig_rows, 0);
  for (std::size_t i = 0; i < n; ++i) {
    if (S.ptr[i + 1] < S.ptr[i]) throw std::invalid_argument("sweep form: row pointers decrease");
    for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k)
      if (S.col[k] < 0 || static_cast<std::size_t>(S.col[k]) >= i)
        throw std::invalid_argument("sweep form: an entry does not reference an earlier row");
    const std::size_t slot = S.gid[i] & kCodeSlotMask;
    if (slot >= seen.size() || seen[slot]) throw std::invalid_argument("sweep form: bad or repeated solution slot");
    seen[slot] = 1;
  }
}

static unsigned depth_of(const HostCsr &S, std::vector<unsigned> &lev) {
  const unsigned m = static_cast<unsigned>(S.nrows);
  lev.assign(m, 0u);
  unsigned depth = 0;
  for (unsigned i = 0; i < m; ++i) {
    unsigned l = 0;
    for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k) l = std::max(l, lev[S.col[k]] + 1u);
    lev[i] = l;
    depth  = std::max(depth, l + 1u);
  }
  return depth;
}

// as-late-as-possible level sets: a row sits as many steps before the end as its longest chain
// of dependents is long.  In a fan-out sweep (U: root first) this puts ALL leaves of the
// elimination tree into the last level set -- the mirror image of the forward sweep, where
// they are the first one -- instead of scattering them over every level: a leaf whose parent
// falls into the same super level would otherwise be split into two rows.
static unsigned depth_alap(const HostCsr &S, std::vector<unsigned> &lev) {
  const unsigned        m = static_cast<unsigned>(S.nrows);
  std::vector<unsigned> h(m, 0u);
  unsigned              depth = 0;
  for (unsigned i = m; i-- > 0;) {
    for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k) {
      const unsigned j = static_cast<unsigned>(S.col[k]);
      h[j]             = std::max(h[j], h[i] + 1u);
    }
    depth = std::max(depth, h[i] + 1u);
  }
  lev.resize(m);
  for (unsigned i = 0; i < m; ++i) lev[i] = depth - 1u - h[i];
  return depth;
}

// The merged system for a given step assignment: rows interleaved [.., t_i, x_i, ..] in the original
// sweep order.  step[] is monotone along dependencies; a row with wlen > 0 is PINNED (it has producers
// in its own step and carries the row wcol/wval of W^{-1} - I over the t unknowns of its step).
static HostCsr emit_merged(const HostCsr &S, const MergeParams &prm, MergeStats *st, const std::vector<unsigned> &step,
                           const std::vector<char> &pinned, const std::vector<std::size_t> &wbeg,
                           const std::vector<unsigned> &wlen, const std::vector<unsigned> &wcol,
                           const std::vector<double> &wval, unsigned nsteps) {
  const unsigned m = static_cast<unsigned>(S.nrows);
  // ---- the merged system, rows interleaved [.., t_i, x_i, ..] in the original sweep order
  HostCsr E;
  E.orig_rows = m;
  E.ptr.push_back(0u);
  std::vector<unsigned> xpos(m), tpos(m);
  std::vector<double>   cacc;
  std::vector<unsigned> cstamp, ctouched;
  unsigned              ccur = 0;
  if (prm.chain) {
    cacc.assign(2 * static_cast<std::size_t>(m), 0.0);
    cstamp.assign(2 * static_cast<std::size_t>(m), 0u);
  }
  auto emit_cross = [&](unsigned i) {  // entries of row i that reference earlier steps
    if (!prm.chain) {
      for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k) {
        const unsigned j = static_cast<unsigned>(S.col[k]);
        if (step[j] == step[i]) continue;
        E.col.push_back(static_cast<int>(xpos[j]));
        E.val.push_back(S.val[k]);
      }
      return;
    }
    ++ccur;
    ctouched.clear();
    auto add = [&](unsigned pos, double v) {
      if (cstamp[pos] != ccur) {
        cstamp[pos] = ccur;
        cacc[pos]   = 0.0;
        ctouched.push_back(pos);
      }
      cacc[pos] += v;
    };
    for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k) {
      const unsigned j = static_cast<unsigned>(S.col[k]);
      if (step[j] == step[i]) continue;
      // chaining: x_j of a PINNED row of the immediately preceding step is replaced by its
      // expansion in t, so that the critical rows of consecutive steps depend on each other's t
      if ((prm.chain_all || pinned[i]) && wlen[j] && step[j] + 1u == step[i]) {
        add(tpos[j], S.val[k]);
        for (std::size_t w = wbeg[j], we = wbeg[j] + wlen[j]; w < we; ++w) add(tpos[wcol[w]], S.val[k] * wval[w]);
      } else {
        add(xpos[j], S.val[k]);
      }
    }
    std::sort(ctouched.begin(), ctouched.end());
    for (unsigned pos : ctouched) {
      E.col.push_back(static_cast<int>(pos));
      E.val.push_back(cacc[pos]);
    }
  };
  for (unsigned i = 0; i < m; ++i) {
    if (!wlen[i]) {
      for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k)
        if (step[S.col[k]] >= step[i]) throw std::logic_error("merge_slack: in-step entry on an unsplit row");
      emit_cross(i);
      xpos[i] = tpos[i] = static_cast<unsigned>(E.gid.size());
      E.gid.push_back(S.gid[i]);
      E.ptr.push_back(static_cast<unsigned>(E.col.size()));
      continue;
    }
    emit_cross(i);  // t_i = b_i - sum_{j in earlier steps} T_ij x_j
    tpos[i] = static_cast<unsigned>(E.gid.size());
    E.gid.push_back(m + S.gid[i]);
    E.ptr.push_back(static_cast<unsigned>(E.col.size()));
    for (std::size_t w = wbeg[i], we = wbeg[i] + wlen[i]; w < we; ++w) {  // x_i = t_i + sum_j Winv_ij t_j
      E.col.push_back(static_cast<int>(tpos[wcol[w]]));
      E.val.push_back(-wval[w]);
    }
    E.col.push_back(static_cast<int>(tpos[i]));
    E.val.push_back(-1.0);
    xpos[i] = static_cast<unsigned>(E.gid.size());
    E.gid.push_back(S.gid[i] | kCodeZeroRhs);
    E.ptr.push_back(static_cast<unsigned>(E.col.size()));
  }
  E.nrows = E.ncols = E.gid.size();
  if (E.nrows > 0x7fffffffull || E.col.size() > 0xfffffff0ull) throw std::length_error("merged factor too large");
  if (st) {
    std::vector<unsigned> elev;
    st->ext_rows     = E.nrows;
    st->ext_nnz      = E.col.size();
    st->ext_depth    = depth_of(E, elev);
    st->super_levels = nsteps;
  }
  return E;
}

// ---- slack-aware merging ------------------------------------------------------------------
// The dependency DAG of an incomplete factor is a thin critical core inside a mass of rows with
// slack (Poisson 128^3, L_0: depth 715, but only 2 % of the rows -- 6 % of the entries -- lie
// within 64 levels of the critical path; SURVEY.md App. A).  merge_levels() above groups LEVEL
// SETS, so every row of a merged level set pays fill, critical or not.  Here a row is handled
// when it is DUE (its as-late-as-possible time z = depth - 1 - height) and placed into the
// earliest STEP its producers allow:
//     step(i) = min(current step, 1 + max_j step(j)).
// Only a row whose producer sits in the still-open current step is PINNED: it is the only kind
// of row that is split into (t_i, x_i) and receives a row of W^{-1}.  A row with slack lands in
// an earlier, already closed step and keeps its original entries.  The current step is closed
// (greedily, in due-time order) when the fill of the pinned rows due next would exceed `gain`,
// a W^{-1} row would exceed `row_cap`, or the step holds more than `sl_cap` entries.
// Result: the same exact reformulation T x = b <=> t = b - X x, x = W^{-1} t (W block diagonal
// over the steps), with fill proportional to the critical core instead of to the factor.
static unsigned height_of(const HostCsr &S, std::vector<unsigned> &h) {
  const unsigned m = static_cast<unsigned>(S.nrows);
  h.assign(m, 0u);
  unsigned depth = 0;
  for (unsigned i = m; i-- > 0;) {
    for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k) {
      const unsigned j = static_cast<unsigned>(S.col[k]);
      h[j]             = std::max(h[j], h[i] + 1u);
    }
    depth = std::max(depth, h[i] + 1u);
  }
  return depth;
}

HostCsr merge_slack(const HostCsr &S, const MergeParams &prm, MergeStats *st) {
  const unsigned m = static_cast<unsigned>(S.nrows);
  if (S.gid.size() != m || S.orig_rows != m) throw std::logic_error("merge_slack: input is not in sweep form");
  std::vector<unsigned> h;
  const unsigned        depth = height_of(S, h);
  if (st) {
    st->rows  = m;
    st->nnz   = S.col.size();
    st->depth = depth;
  }
  // rows bucketed by due time z = depth - 1 - h, index order inside a bucket (topological: a
  // producer is due strictly earlier than its consumers)
  std::vector<unsigned> dptr(depth + 1u, 0u), drows(m);
  for (unsigned i = 0; i < m; ++i) ++dptr[depth - h[i]];
  for (unsigned t = 0; t < depth; ++t) dptr[t + 1] += dptr[t];
  {
    std::vector<unsigned> next(dptr.begin(), dptr.end() - 1);
    for (unsigned i = 0; i < m; ++i) drows[next[depth - 1u - h[i]]++] = i;
  }
  std::vector<unsigned>    step(m, 0u);
  std::vector<std::size_t> wbeg(m, 0);
  std::vector<unsigned>    wlen(m, 0u);
  std::vector<char>        pinned(m, 0);
  std::vector<unsigned>    wcol;
  std::vector<double>      wval;
  std::vector<double>      acc(m, 0.0);
  std::vector<unsigned>    stamp(m, 0u), touched, tcol, tlen, trow, smax_of, cur_pinned;
  std::vector<double>      tval;
  unsigned                 cur = 0, t0 = 0, mark = 0;
  double                   step_entries = 0.0;
  std::vector<unsigned char> idepth(m, 0);  // length of the chain of pinned rows below a row, inside its step
  unsigned                 step_idepth = 0;
  // a step whose pinned rows only depend on unpinned rows of the step saved nothing (a t and an x
  // phase instead of two plain steps): undo its fill, its pinned rows open a step of their own
  auto close_step = [&] {
    if (step_idepth == 1u) {
      ++cur;
      for (unsigned i : cur_pinned) {
        wlen[i]   = 0;
        pinned[i] = 0;
        idepth[i] = 0;
        step[i]   = cur;
      }
    }
    cur_pinned.clear();
    step_idepth = 0;
  };
  for (unsigned t = 0; t < depth; ++t) {
    const unsigned rb = dptr[t], re = dptr[t + 1];
    smax_of.assign(re - rb, 0u);
    auto smax_plus1 = [&](unsigned i) {  // 1 + highest step of a producer (0: no producers)
      unsigned s = 0;
      for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k) s = std::max(s, step[S.col[k]] + 1u);
      return s;
    };
    for (unsigned q = rb; q < re; ++q) smax_of[q - rb] = smax_plus1(drows[q]);
    // tentative W^{-1} rows of the rows that would be pinned to the current step
    bool accept = false;
    tcol.clear(), tval.clear(), tlen.clear(), trow.clear();
    double   cost = 0.0, entries = 0.0;
    unsigned maxlen = 0;
    bool     any_pinned = false;
    for (unsigned q = rb; q < re; ++q) {
      const unsigned i = drows[q];
      if (smax_of[q - rb] <= cur) {
        if (smax_of[q - rb] == cur) entries += static_cast<double>(S.ptr[i + 1] - S.ptr[i]);
        continue;
      }
      any_pinned = true;
      if (!prm.enabled || t == t0 || t - t0 >= prm.bmax || maxlen > prm.row_cap) continue;
      ++mark;
      touched.clear();
      unsigned nwithin = 0;
      auto     add = [&](unsigned j, double v) {
        if (stamp[j] != mark) {
          stamp[j] = mark;
          acc[j]   = 0.0;
          touched.push_back(j);
        }
        acc[j] += v;
      };
      for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k) {
        const unsigned j = static_cast<unsigned>(S.col[k]);
        if (step[j] != cur) continue;
        ++nwithin;
        const double v = -S.val[k];  // row i of -N times (I + (W^{-1} - I))
        add(j, v);
        for (std::size_t w = wbeg[j], we = wbeg[j] + wlen[j]; w < we; ++w) add(wcol[w], v * wval[w]);
      }
      std::sort(touched.begin(), touched.end());
      for (unsigned j : touched) {
        tcol.push_back(j);
        tval.push_back(acc[j]);
      }
      trow.push_back(i);
      tlen.push_back(static_cast<unsigned>(touched.size()));
      cost += static_cast<double>(touched.size()) - nwithin + 1.0 + prm.row_cost;
      entries += static_cast<double>(S.ptr[i + 1] - S.ptr[i] - nwithin + touched.size()) + 1.0;
      maxlen = std::max<unsigned>(maxlen, static_cast<unsigned>(touched.size()) + 1u);
    }
    if (!any_pinned)
      accept = true;  // nothing due now depends on the open step: it simply stays open
    else
      accept = prm.enabled && t > t0 && t - t0 < prm.bmax && maxlen <= prm.row_cap && cost <= prm.gain &&
               step_entries + entries <= prm.sl_cap;
    if (!accept) {
      close_step();
      for (unsigned q = rb; q < re; ++q) smax_of[q - rb] = smax_plus1(drows[q]);
      ++cur;
      t0           = t;
      step_entries = 0.0;
      for (unsigned q = rb; q < re; ++q) {
        const unsigned i = drows[q];
        step[i]          = std::min(cur, smax_of[q - rb]);
        if (step[i] == cur) step_entries += static_cast<double>(S.ptr[i + 1] - S.ptr[i]);
      }
      continue;
    }
    step_entries += entries;
    std::size_t tp = 0, tr = 0;
    for (unsigned q = rb; q < re; ++q) {
      const unsigned i = drows[q];
      if (smax_of[q - rb] <= cur) {
        step[i] = smax_of[q - rb];
        continue;
      }
      // pinned
      if (trow[tr] != i) throw std::logic_error("merge_slack: tentative rows out of order");
      step[i]   = cur;
      pinned[i] = 1;
      {
        unsigned d = 0;
        for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k)
          if (step[S.col[k]] == cur) d = std::max<unsigned>(d, idepth[S.col[k]]);
        idepth[i]   = static_cast<unsigned char>(std::min(255u, d + 1u));
        step_idepth = std::max<unsigned>(step_idepth, idepth[i]);
      }
      wbeg[i]   = wcol.size();
      wlen[i]   = tlen[tr];
      wcol.insert(wcol.end(), tcol.begin() + tp, tcol.begin() + tp + wlen[i]);
      wval.insert(wval.end(), tval.begin() + tp, tval.begin() + tp + wlen[i]);
      tp += wlen[i];
      ++tr;
      cur_pinned.push_back(i);
    }
  }
  close_step();
  if (std::getenv("HIFIR_B200_MERGE_DEBUG")) {
    std::vector<unsigned> rows_in(cur + 1u, 0u), pin_in(cur + 1u, 0u), tmin(cur + 1u, depth), tmax(cur + 1u, 0u);
    std::vector<double>   fill_in(cur + 1u, 0.0);
    for (unsigned i = 0; i < m; ++i) {
      ++rows_in[step[i]];
      if (pinned[i]) {
        ++pin_in[step[i]];
        fill_in[step[i]] += wlen[i];
        const unsigned z = depth - 1u - h[i];
        tmin[step[i]] = std::min(tmin[step[i]], z), tmax[step[i]] = std::max(tmax[step[i]], z);
      }
    }
    for (unsigned s = 0; s <= cur; ++s)
      std::fprintf(stderr, "  step %u: rows %u pinned %u fill %.0f due-times of pinned [%u, %u]\n", s, rows_in[s], pin_in[s],
                   fill_in[s], tmin[s], tmax[s]);
  }
  return emit_merged(S, prm, st, step, pinned, wbeg, wlen, wcol, wval, cur + 1u);
}

// ---- proportional scheduling ----------------------------------------------------------------
// Every row sits at the relative position u = a / (a + h) of the longest path through it
// (a = as-soon-as-possible level, h = height = longest chain of dependents); u increases strictly
// along every dependency.  K steps cut [0, 1] uniformly: a path of P rows is compressed by P / K,
// a path with P <= K is not compressed at all (no fill) -- level-set bucketing compresses every
// path by depth / K, whatever its length.  Rows whose W^{-1} row would exceed row_cap are moved to
// the next step (the shift propagates to their dependents).
HostCsr merge_prop(const HostCsr &S, const MergeParams &prm, MergeStats *st) {
  const unsigned m = static_cast<unsigned>(S.nrows);
  std::vector<unsigned> a, h;
  const unsigned        depth = depth_of(S, a);
  height_of(S, h);
  if (st) {
    st->rows  = m;
    st->nnz   = S.col.size();
    st->depth = depth;
  }
  const unsigned K = std::max(1u, std::min(prm.steps, depth));
  std::vector<unsigned>    step(m, 0u);
  std::vector<std::size_t> wbeg(m, 0);
  std::vector<unsigned>    wlen(m, 0u);
  std::vector<char>        pinned(m, 0);
  std::vector<unsigned>    wcol;
  std::vector<double>      wval;
  std::vector<double>      acc(m, 0.0);
  std::vector<unsigned>    stamp(m, 0u), touched;
  unsigned                 mark = 0, nsteps = 1;
  for (unsigned i = 0; i < m; ++i) {
    const unsigned P  = a[i] + h[i];
    unsigned       s0 = P ? static_cast<unsigned>((static_cast<unsigned long long>(a[i]) * K) / (P + 1u)) : 0u;
    unsigned       smax = 0;
    bool           any = false;
    for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k) {
      smax = std::max(smax, step[S.col[k]]);
      any  = true;
    }
    unsigned s = any ? std::max(s0, smax) : s0;
    if (!prm.enabled && any) s = std::max(s, smax + 1u);  // no merging: one step per dependent row
    for (;;) {
      // row of W^{-1} - I if the row stays in step s
      ++mark;
      touched.clear();
      unsigned nwithin = 0;
      auto     add = [&](unsigned j, double v) {
        if (stamp[j] != mark) {
          stamp[j] = mark;
          acc[j]   = 0.0;
          touched.push_back(j);
        }
        acc[j] += v;
      };
      for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k) {
        const unsigned j = static_cast<unsigned>(S.col[k]);
        if (step[j] != s) continue;
        ++nwithin;
        const double v = -S.val[k];
        add(j, v);
        for (std::size_t w = wbeg[j], we = wbeg[j] + wlen[j]; w < we; ++w) add(wcol[w], v * wval[w]);
      }
      if (!nwithin) break;
      if (touched.size() + 1u > prm.row_cap) {  // too long: the row opens the next step for its paths
        ++s;
        continue;
      }
      std::sort(touched.begin(), touched.end());
      pinned[i] = 1;
      wbeg[i]   = wcol.size();
      wlen[i]   = static_cast<unsigned>(touched.size());
      for (unsigned j : touched) {
        wcol.push_back(j);
        wval.push_back(acc[j]);
      }
      break;
    }
    step[i] = s;
    nsteps  = std::max(nsteps, s + 1u);
  }
  return emit_merged(S, prm, st, step, pinned, wbeg, wlen, wcol, wval, nsteps);
}

HostCsr merge_levels(const HostCsr &S, const MergeParams &prm, MergeStats *st, bool fan_out) {
  const unsigned m = static_cast<unsigned>(S.nrows);
  if (S.gid.size() != m || S.orig_rows != m) throw std::logic_error("merge_levels: input is not in sweep form");
  if (prm.auto_caps && prm.enabled && !prm.steps && !prm.slack) {
    // Per-factor caps chosen by the cost model (MergeParams::plan_cost).  A super level that grows by
    // k level sets fills every row with its dependency cone inside the super level (~k^3 entries for
    // a stencil wavefront), so how much fill a saved step is worth depends on how the factor's
    // entries and steps price on the device.  The candidates are tried from the most fill down:
    // first the former fixed rule, sl_cap = clamp(nnz / 14, 3e5, 1.2e6) with gain = 3 sl_cap (fitted
    // on factors with 3x more entries), then smaller caps, then the unmerged factor.  The first one
    // that predicts a longer sweep than its predecessor ends the search (the curve has one minimum)
    // and the cheapest plan seen is kept: deterministic, and a large factor -- whose minimum is near
    // the top -- pays for two or three plans at attach, the cheaper ones to build.
    const double kCaps[] = {std::min(1.2e6, std::max(3.0e5, static_cast<double>(S.col.size()) / 14.0)), 1e5, 3e4,
                            1e4, 3e3, 1e3};
    double       best = 0.0, prev = 0.0;
    HostCsr      E;
    MergeStats   est;
    bool         turned = false;
    for (double cap : kCaps) {
      MergeParams q = prm;
      q.auto_caps   = false;
      q.sl_cap      = cap;
      q.gain        = std::max(prm.gain, 3.0 * cap);  // the super level's size binds, not one level set's fill
      MergeStats    qs;
      HostCsr       Q = merge_levels(S, q, &qs, fan_out);
      const double  c = prm.plan_cost(qs);
      if (cap == kCaps[0] || c < best) best = c, E = std::move(Q), est = qs;
      if (cap != kCaps[0] && c > prev) {
        turned = true;
        break;
      }
      prev = c;
    }
    if (!turned) {  // still falling: the unmerged factor
      std::vector<unsigned> lev;
      const std::size_t     depth0 = depth_of(S, lev);
      if (prm.plan_cost(depth0, S.col.size(), m) < best) {
        E        = S;
        est.rows = est.ext_rows = m;
        est.nnz = est.ext_nnz = S.col.size();
        est.depth = est.ext_depth = est.super_levels = depth0;
      }
    }
    if (st) *st = est;
    return E;
  }
  if (prm.steps) return merge_prop(S, prm, st);
  if (prm.slack) return merge_slack(S, prm, st);
  std::vector<unsigned> lev;
  const bool            alap  = prm.alap == 2 || (prm.alap == 1 && fan_out) || (prm.alap == 3 && !fan_out);
  const unsigned        depth = alap ? depth_alap(S, lev) : depth_of(S, lev);
  if (st) {
    st->rows  = m;
    st->nnz   = S.col.size();
    st->depth = depth;
  }
  // rows bucketed by level set
  std::vector<unsigned> lptr(depth + 1u, 0u), lrows(m);
  for (unsigned i = 0; i < m; ++i) ++lptr[lev[i] + 1u];
  for (unsigned l = 0; l < depth; ++l) lptr[l + 1] += lptr[l];
  {
    std::vector<unsigned> next(lptr.begin(), lptr.end() - 1);
    for (unsigned i = 0; i < m; ++i) lrows[next[lev[i]]++] = i;
  }
  // ---- greedy super levels; rows of W^{-1} - I (strictly lower part) per row
  std::vector<unsigned>    sl0(m, 0u);  // first level set of the row's super level
  std::vector<std::size_t> wbeg(m, 0);
  std::vector<unsigned>    wlen(m, 0u);
  std::vector<unsigned>    wcol;
  std::vector<double>      wval;
  wcol.reserve(S.col.size());
  wval.reserve(S.col.size());
  std::vector<double>   acc(m, 0.0);
  std::vector<unsigned> stamp(m, 0u), touched, tcol, tlen;
  std::vector<double>   tval;
  unsigned              cur = 0, l0 = 0;
  double                sl_entries = 0.0;  // entries of the current super level (both of its phases)
  auto close_super = [&](unsigned lend) {  // super level [l0, lend) ends
    // two merged level sets save nothing (t and x steps instead of two x steps): undo
    if (lend - l0 == 2u)
      for (unsigned q = lptr[l0 + 1]; q < lptr[l0 + 2]; ++q) {
        const unsigned i = lrows[q];
        wlen[i]          = 0;
        sl0[i]           = l0 + 1u;
      }
  };
  for (unsigned l = 0; l < depth; ++l) {
    const unsigned rb = lptr[l], re = lptr[l + 1];
    bool           accept = false;
    if (prm.enabled && l > l0 && l - l0 < prm.bmax) {
      tcol.clear();
      tval.clear();
      tlen.assign(re - rb, 0u);
      double   cost = 0.0, entries = 0.0;
      unsigned maxlen = 0;
      for (unsigned q = rb; q < re && maxlen <= prm.row_cap; ++q) {
        const unsigned i = lrows[q];
        ++cur;
        touched.clear();
        unsigned nwithin = 0;
        auto     add = [&](unsigned j, double v) {
          if (stamp[j] != cur) {
            stamp[j] = cur;
            acc[j]   = 0.0;
            touched.push_back(j);
          }
          acc[j] += v;
        };
        for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k) {
          const unsigned j = static_cast<unsigned>(S.col[k]);
          if (lev[j] < l0) continue;
          ++nwithin;
          const double v = -S.val[k];  // row i of -N times (I + (W^{-1} - I))
          add(j, v);
          for (std::size_t w = wbeg[j], we = wbeg[j] + wlen[j]; w < we; ++w) add(wcol[w], v * wval[w]);
        }
        std::sort(touched.begin(), touched.end());
        for (unsigned j : touched) {
          tcol.push_back(j);
          tval.push_back(acc[j]);
        }
        tlen[q - rb] = static_cast<unsigned>(touched.size());
        if (nwithin) cost += static_cast<double>(touched.size()) - nwithin + 1.0 + prm.row_cost;
        entries += static_cast<double>(S.ptr[i + 1] - S.ptr[i] - nwithin + touched.size()) + (nwithin ? 1.0 : 0.0);
        maxlen = std::max<unsigned>(maxlen, static_cast<unsigned>(touched.size()) + 1u);
      }
      // a super level whose phases already saturate the machine gains nothing from growing:
      // merging only pays while its steps are bound by the latency of a dependent hop
      accept = maxlen <= prm.row_cap && cost <= prm.gain && sl_entries + entries <= prm.sl_cap;
      if (accept) sl_entries += entries;
    }
    if (accept) {
      std::size_t tp = 0;
      for (unsigned q = rb; q < re; ++q) {
        const unsigned i = lrows[q];
        wbeg[i]          = wcol.size();
        wlen[i]          = tlen[q - rb];
        wcol.insert(wcol.end(), tcol.begin() + tp, tcol.begin() + tp + wlen[i]);
        wval.insert(wval.end(), tval.begin() + tp, tval.begin() + tp + wlen[i]);
        tp += wlen[i];
        sl0[i] = l0;
      }
    } else {
      if (l > 0) close_super(l);
      l0         = l;
      sl_entries = 0.0;
      for (unsigned q = rb; q < re; ++q) {
        sl0[lrows[q]] = l0;
        sl_entries += static_cast<double>(S.ptr[lrows[q] + 1] - S.ptr[lrows[q]]);
      }
    }
  }
  if (depth) close_super(depth);
  // ---- the merged system, rows interleaved [.., t_i, x_i, ..] in the original sweep order
  HostCsr E;
  E.orig_rows = m;
  E.ptr.push_back(0u);
  std::vector<unsigned> xpos(m), tpos(m);
  // ordinal of the super level of every level set
  std::vector<unsigned> sl_ord(depth, 0u);
  {
    std::vector<unsigned> first(depth, 0u);
    for (unsigned i = 0; i < m; ++i) first[lev[i]] = sl0[i];
    unsigned ordn = 0;
    for (unsigned l = 0; l < depth; ++l) {
      if (l > 0 && first[l] != first[l - 1]) ++ordn;
      sl_ord[l] = ordn;
    }
  }
  // Chaining (prm.chain): an entry that references x_j of the IMMEDIATELY preceding super level is
  // replaced by x_j = t_j + sum_l Winv_jl t_l.  The t rows of consecutive super levels then depend
  // on each other directly -- one dependent step per super level instead of two -- and the x
  // rows leave the critical path (they are computed beside the next super level's t rows).
  std::vector<double>   cacc;
  std::vector<unsigned> cstamp, ctouched;
  unsigned              ccur = 0;
  if (prm.chain) {
    cacc.assign(2 * static_cast<std::size_t>(m), 0.0);
    cstamp.assign(2 * static_cast<std::size_t>(m), 0u);
  }
  auto emit_cross = [&](unsigned i) {  // entries of row i that reference earlier super levels
    if (!prm.chain) {
      for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k) {
        const unsigned j = static_cast<unsigned>(S.col[k]);
        if (lev[j] >= sl0[i]) continue;
        E.col.push_back(static_cast<int>(xpos[j]));
        E.val.push_back(S.val[k]);
      }
      return;
    }
    ++ccur;
    ctouched.clear();
    auto add = [&](unsigned pos, double v) {
      if (cstamp[pos] != ccur) {
        cstamp[pos] = ccur;
        cacc[pos]   = 0.0;
        ctouched.push_back(pos);
      }
      cacc[pos] += v;
    };
    const unsigned my = sl_ord[lev[i]];
    for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k) {
      const unsigned j = static_cast<unsigned>(S.col[k]);
      if (lev[j] >= sl0[i]) continue;
      if (wlen[j] && sl_ord[lev[j]] + 1u == my) {
        add(tpos[j], S.val[k]);
        for (std::size_t w = wbeg[j], we = wbeg[j] + wlen[j]; w < we; ++w) add(tpos[wcol[w]], S.val[k] * wval[w]);
      } else {
        add(xpos[j], S.val[k]);
      }
    }
    std::sort(ctouched.begin(), ctouched.end());
    for (unsigned pos : ctouched) {
      E.col.push_back(static_cast<int>(pos));
      E.val.push_back(cacc[pos]);
    }
  };
  for (unsigned i = 0; i < m; ++i) {
    if (!wlen[i]) {
      for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k)
        if (lev[S.col[k]] >= sl0[i]) throw std::logic_error("merge_levels: in-level entry on an unsplit row");
      emit_cross(i);
      xpos[i] = tpos[i] = static_cast<unsigned>(E.gid.size());
      E.gid.push_back(S.gid[i]);
      E.ptr.push_back(static_cast<unsigned>(E.col.size()));
      continue;
    }
    // t_i = b_i - sum_{j in earlier super levels} T_ij x_j
    emit_cross(i);
    tpos[i] = static_cast<unsigned>(E.gid.size());
    E.gid.push_back(m + S.gid[i]);
    E.ptr.push_back(static_cast<unsigned>(E.col.size()));
    // x_i = t_i + sum_j Winv_ij t_j   (a sweep row computes rhs - sum val * x)
    for (std::size_t w = wbeg[i], we = wbeg[i] + wlen[i]; w < we; ++w) {
      E.col.push_back(static_cast<int>(tpos[wcol[w]]));
      E.val.push_back(-wval[w]);
    }
    E.col.push_back(static_cast<int>(tpos[i]));
    E.val.push_back(-1.0);
    xpos[i] = static_cast<unsigned>(E.gid.size());
    E.gid.push_back(S.gid[i] | kCodeZeroRhs);
    E.ptr.push_back(static_cast<unsigned>(E.col.size()));
  }
  E.nrows = E.ncols = E.gid.size();
  if (E.nrows > 0x7fffffffull || E.col.size() > 0xfffffff0ull) throw std::length_error("merged factor too large");
  if (st) {
    std::vector<unsigned> elev;
    st->ext_rows     = E.nrows;
    st->ext_nnz      = E.col.size();
    st->ext_depth    = depth_of(E, elev);
    std::vector<char> seen(depth + 1u, 0);
    for (unsigned i = 0; i < m; ++i) seen[sl0[i]] = 1;
    st->super_levels = static_cast<std::size_t>(std::count(seen.begin(), seen.end(), 1));
  }
  return E;
}

}  // namespace hifgpu
