// wsweep.cu -- statically scheduled, warp-autonomous triangular sweep ("warp streams").
//
// Replaces CCS::solve_as_strict_lower / solve_as_strict_upper of the reference
// (ds/CompressedStorage.hpp:2267-2279, 2356-2369) on the merged factors of merge.cu.
//
// Round 1's streaming kernel handed out chunks of 8 slices through a ticket counter and ran every
// chunk through a dependent chain ticket -> descriptor -> factor entries -> admission -> gathers
// -> publish, two CTA barriers per chunk: 2.1-2.8 us per level set although the hardware hand-off
// is 0.3-0.5 us.  Here nothing is dynamic:
//   * the slices of every level set are dealt round-robin to the warps of ONE persistent CTA per SM
//     at attach time; a warp owns a private, contiguous STREAM of segments (header, row codes,
//     publish slots, slot indices and values of <= 8 entries per lane) in level order;
//   * the stream is staged through shared memory by 1-D TMA bulk copies (cp.async.bulk + mbarrier)
//     into a per-warp ring several segments ahead -- the factor data never sits on the dependent
//     path of a level, costs no registers and is read from HBM exactly once;
//   * warps never synchronize with each other: no tickets, no CTA barriers, no level counters.
//     Readiness travels with the value (tagged words, common.cuh).  A warp gathers all entries of
//     a segment at once and re-polls only what was not ready;
//   * run-ahead warps do not hammer L2: before touching the solution a warp waits (sleeping in
//     proportion to its distance from a frontier hint) until a SENTINEL row -- the last row of
//     level l - window -- carries the current tag.  The sentinel only throttles; correctness
//     rests on the tags alone;
//   * solution slots are renumbered level-major and, inside a level set, in sweep order, rows of a
//     level are ordered by (lanes per row, length bucket, sweep order): the 32 gathers of a warp
//     instruction share 32-byte sectors (0.6-0.7 sector requests per entry instead of 0.7-0.8; an
//     SM issues one L2 sector request per clock, the throughput ceiling of the wide level sets).
//   * rows without entries (55 % of L_0: the leaves of the elimination tree) are copied 8 per
//     lane by COPY segments.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <string>
#include <type_traits>

#include "hifgpu.h"

namespace hifgpu {

namespace {
constexpr unsigned kWsU        = 8;            // entries per lane and segment
constexpr unsigned kWsNone     = 0xffffffffu;  // padding column / no sentinel
constexpr unsigned kSegFirst   = 1u, kSegLast = 2u, kSegCopy = 4u, kSegUpper = 8u;
constexpr unsigned kWsHdrWords = 4;

inline unsigned seg_words(unsigned width, bool copy, bool f32) {
  if (copy) return kWsHdrWords + width * 32u * 2u;
  return kWsHdrWords + 64u + width * 32u * (f32 ? 2u : 3u);
}
}  // namespace

unsigned ws_stage_bytes(bool f32) { return seg_words(kWsU, false, f32) * 4u; }

int ws_env(const char *name, int dflt) {
  const char *e = std::getenv(name);
  return e ? std::atoi(e) : dflt;
}

// ---- host: merged sweep form -> warp streams ------------------------------------------
// slot_of (out): solution slot of every ORIGINAL row.  rhs_index (nullable): position of original
// row r in the right-hand side array of this sweep (identity when null) -- the U sweep reads the L
// sweep's tagged result, which lives at the L plan's slots.
void pack_warp_streams(const HostCsr &S, WsHost &H, unsigned nwarps, unsigned window, bool f32,
                       const unsigned *rhs_index, unsigned umin_force) {
  const unsigned n = static_cast<unsigned>(S.nrows), m = static_cast<unsigned>(S.orig_rows);
  H = WsHost();
  H.nwarps = nwarps;
  H.wdesc.assign(static_cast<std::size_t>(nwarps) * 8u, 0u);
  H.slot_of.assign(m, 0u);
  H.nslots = n;
  if (!n) return;
  if (S.gid.size() != n) throw std::logic_error("pack_warp_streams: factor is not in sweep form");
  validate_sweep_form(S);  // the device indexes the solution buffers with these numbers
  std::vector<unsigned> lev(n, 0u);
  unsigned              depth = 0;
  for (unsigned i = 0; i < n; ++i) {
    unsigned l = 0;
    for (unsigned k = S.ptr[i]; k < S.ptr[i + 1]; ++k) l = std::max(l, lev[S.col[k]] + 1u);
    lev[i] = l;
    depth  = std::max(depth, l + 1u);
  }
  auto rowlen = [&](unsigned i) { return S.ptr[i + 1] - S.ptr[i]; };
  // Entries per lane, chosen per level set: a thin level set is bound by the latency of one warp's
  // round of scattered gathers (~1 us for 8 x 32 of them: an SM accepts one sector request per
  // clock, a single warp one every ~5), so its rows are spread over as many lanes -- and warps --
  // as there are: U_l = entries of the level / lanes of one warp group, clamped to [umin, 8].
  const unsigned groups = static_cast<unsigned>(std::max(1, ws_env("HIFIR_B200_WS_GROUPS", 2)));
  const unsigned umin   = umin_force ? umin_force : static_cast<unsigned>(std::min(8, std::max(1, ws_env("HIFIR_B200_WS_UMIN", 1))));
  const unsigned gwarps = std::max(1u, nwarps / groups);  // warps that serve one level set of a thin stretch
  std::vector<unsigned> ulev(depth, kWsU);
  {
    std::vector<double> ent_l(depth, 0.0);
    for (unsigned i = 0; i < n; ++i) ent_l[lev[i]] += rowlen(i);
    for (unsigned l = 0; l < depth; ++l) {
      const double u = std::ceil(ent_l[l] / (32.0 * gwarps));
      ulev[l]        = static_cast<unsigned>(std::min<double>(kWsU, std::max<double>(umin, u)));
    }
  }
  // class: lanes per row 2^z so that a lane holds <= U_l entries (z = 5 at most: beyond, a lane holds
  // more, and beyond 8 per lane the slice takes several segments)
  auto zof = [&](unsigned len, unsigned U) {
    unsigned z = 0;
    while (z < 5u && ((len + (1u << z) - 1u) >> z) > U) ++z;
    return z;
  };
  std::vector<unsigned char> cls(n), bkt(n);
  for (unsigned i = 0; i < n; ++i) {
    const unsigned len = rowlen(i);
    cls[i]             = static_cast<unsigned char>(len ? zof(len, ulev[lev[i]]) : 0u);
    const unsigned w   = (len + (1u << cls[i]) - 1u) >> cls[i];
    bkt[i] = static_cast<unsigned char>(len == 0 ? 0u : w <= 1 ? 1u : w <= 2 ? 2u : w <= 4 ? 3u : w <= 6 ? 4u : w <= 8 ? 5u : 6u);
  }
  // slots: level-major, sweep order inside a level set (rows of S are in sweep order)
  std::vector<unsigned> slot(n);
  {
    std::vector<unsigned> cnt(depth + 1u, 0u);
    for (unsigned i = 0; i < n; ++i) ++cnt[lev[i] + 1u];
    for (unsigned l = 0; l < depth; ++l) cnt[l + 1] += cnt[l];
    for (unsigned i = 0; i < n; ++i) slot[i] = cnt[lev[i]]++;
  }
  for (unsigned i = 0; i < n; ++i) {
    const unsigned code = S.gid[i] & kCodeSlotMask;
    if (code < m) H.slot_of[code] = slot[i];  // the solution itself (codes >= m: auxiliary unknowns)
  }
  // order: level, (empty rows first), class desc, bucket desc, sweep order
  std::vector<unsigned> ord(n);
  std::iota(ord.begin(), ord.end(), 0u);
  std::stable_sort(ord.begin(), ord.end(), [&](unsigned a, unsigned b) {
    if (lev[a] != lev[b]) return lev[a] < lev[b];
    const bool ea = rowlen(a) == 0, eb = rowlen(b) == 0;
    if (ea != eb) return ea;
    if (cls[a] != cls[b]) return cls[a] > cls[b];
    if (bkt[a] != bkt[b]) return bkt[a] > bkt[b];
    return a < b;
  });
  // ---- slices in level order; slice q (global count) goes to warp q % nwarps
  struct Seg {
    unsigned warp, off;  // offset in words inside the warp's private stream
  };
  std::vector<std::vector<unsigned>> ws(nwarps);  // private streams
  std::vector<std::vector<unsigned>> seg_off(nwarps);
  std::vector<unsigned>              sentinel_of_level(depth, kWsNone);
  // Warp assignment.  A warp works through its segments one after the other and a segment costs about
  // one L2 round trip whatever its width, so the sweep lasts as long as the warp with the MOST
  // segments (measured: a dependency-free second pass takes as long as the first).  Hence plain
  // round-robin with counters that never restart: every warp gets the same number of segments and
  // the slices of one level set land on distinct warps.  Thin level sets (fewer slices than a warp
  // GROUP has warps) alternate between the groups -- level l on group l % groups -- so that one
  // group gathers for level l + 1 while the other finishes level l; wide ones use all warps.
  // A warp is throttled by a sentinel only when it JUMPS far ahead of its previous segment.
  std::vector<int>      last_level(nwarps, -1000000);
  unsigned              nslices = 0;
  unsigned long long    q_all = 0;
  std::vector<unsigned long long> q_grp(groups, 0ull);
  const unsigned        jump_after = static_cast<unsigned>(std::max<int>(static_cast<int>(window), ws_env("HIFIR_B200_WS_JUMP", 8)));
  auto slice_at = [&](unsigned p, bool &copy) {  // rows of the slice that starts at ord[p]
    const unsigned i0 = ord[p], l = lev[i0];
    unsigned       cnt = 1;
    copy               = rowlen(i0) == 0;
    if (copy) {
      while (cnt < 32u * kWsU && p + cnt < n && lev[ord[p + cnt]] == l && rowlen(ord[p + cnt]) == 0) ++cnt;
    } else {
      const unsigned z = cls[i0], cap = 32u >> z;
      while (cnt < cap && p + cnt < n && lev[ord[p + cnt]] == l && rowlen(ord[p + cnt]) != 0 && cls[ord[p + cnt]] == z &&
             bkt[ord[p + cnt]] == bkt[i0])
        ++cnt;
    }
    return cnt;
  };
  std::vector<unsigned> slices_of_level(depth, 0u);
  for (unsigned p = 0; p < n;) {
    bool copy;
    ++slices_of_level[lev[ord[p]]];
    p += slice_at(p, copy);
  }
  auto next_warp = [&](unsigned l) {
    if (groups > 1u && slices_of_level[l] <= gwarps) {
      const unsigned g = l % groups;
      return g * gwarps + static_cast<unsigned>(q_grp[g]++ % gwarps);
    }
    return static_cast<unsigned>(q_all++ % nwarps);
  };
  std::vector<unsigned>              ent;
  auto rhs_code = [&](unsigned i) {
    const unsigned code = S.gid[i];
    unsigned       r    = code & kCodeSlotMask;
    if (r >= m) r -= m;
    if (rhs_index) r = rhs_index[r];
    return r | (code & kCodeZeroRhs);
  };
  auto push_seg = [&](unsigned warp, unsigned width, unsigned z, unsigned flags, unsigned level) -> unsigned * {
    std::vector<unsigned> &st = ws[warp];
    const unsigned         o  = static_cast<unsigned>(st.size());
    seg_off[warp].push_back(o);
    st.resize(o + seg_words(width, (flags & kSegCopy) != 0, f32), 0u);
    unsigned *hd = st.data() + o;
    hd[0]        = width | (z << 8) | (flags << 16);
    hd[1]        = 0;  // size of the segment `stages` ahead: filled by the kernel-side ring depth at finalize
    const bool jump = static_cast<int>(level) - last_level[warp] > static_cast<int>(jump_after);
    hd[2]        = (jump && level >= window) ? sentinel_of_level[level - window] : kWsNone;
    hd[3]        = level;
    last_level[warp] = static_cast<int>(level);
    ++H.nsegs;
    return hd;
  };
  for (unsigned p = 0; p < n;) {
    const unsigned i0 = ord[p], l = lev[i0];
    bool           is_copy;
    const unsigned cnt = slice_at(p, is_copy);
    if (is_copy) {  // COPY segment: up to 8 rows per lane
      const unsigned width = (cnt + 31u) / 32u;
      unsigned *     hd    = push_seg(next_warp(l), width, 0u, kSegFirst | kSegLast | kSegCopy, l);
      unsigned *     codes = hd + kWsHdrWords, *slots = codes + width * 32u;
      for (unsigned r = 0; r < width * 32u; ++r) {
        // row r of the segment: lane r % 32, position r / 32 -> stored at [pos * 32 + lane] = [r]
        codes[r] = r < cnt ? rhs_code(ord[p + r]) : kWsNone;
        slots[r] = r < cnt ? slot[ord[p + r]] : kWsNone;
      }
      sentinel_of_level[l] = slot[ord[p + cnt - 1u]];
      ++nslices;
      p += cnt;
      H.copy_rows += cnt;
      continue;
    }
    const unsigned z = cls[i0], lpr = 1u << z;
    unsigned       width = 0;
    for (unsigned r = 0; r < cnt; ++r) width = std::max(width, (rowlen(ord[p + r]) + lpr - 1u) >> z);
    const unsigned nseg = (width + kWsU - 1u) / kWsU, warp = next_warp(l);
    for (unsigned sg = 0; sg < nseg; ++sg) {
      const unsigned w0 = sg * kWsU, w = std::min(kWsU, width - w0);
      unsigned *     hd = push_seg(warp, w, z, (sg == 0 ? kSegFirst : 0u) | (sg + 1 == nseg ? kSegLast : 0u), l);
      unsigned *     codes = hd + kWsHdrWords, *slots = codes + 32u, *cols = slots + 32u;
      for (unsigned j = 0; j < 32u; ++j) {
        const unsigned r = j >> z;
        codes[j]         = r < cnt ? rhs_code(ord[p + r]) : kWsNone;
        slots[j]         = r < cnt ? slot[ord[p + r]] : kWsNone;
      }
      for (unsigned k = 0; k < w * 32u; ++k) cols[k] = kWsNone;
      unsigned char *vals = reinterpret_cast<unsigned char *>(cols + w * 32u);
      for (unsigned r = 0; r < cnt; ++r) {
        const unsigned i = ord[p + r], b = S.ptr[i], e = S.ptr[i + 1];
        // entries in slot order = producer level, then sweep order: the ones that become ready last come last
        ent.resize(e - b);
        std::iota(ent.begin(), ent.end(), b);
        std::stable_sort(ent.begin(), ent.end(), [&](unsigned x, unsigned y) { return slot[S.col[x]] < slot[S.col[y]]; });
        for (unsigned qq = 0; qq < e - b; ++qq) {  // entry qq of the row -> lane r*lpr + qq % lpr, position qq / lpr
          const unsigned pos = qq >> z;
          if (pos < w0 || pos >= w0 + w) continue;
          const unsigned at = (pos - w0) * 32u + r * lpr + (qq & (lpr - 1u));
          cols[at]          = slot[S.col[ent[qq]]];
          if (f32) {
            const float v = static_cast<float>(S.val[ent[qq]]);
            std::memcpy(vals + static_cast<std::size_t>(at) * 4u, &v, 4);
          } else {
            std::memcpy(vals + static_cast<std::size_t>(at) * 8u, &S.val[ent[qq]], 8);
          }
        }
        if (sg == 0) H.padded += static_cast<std::size_t>(width) * lpr - (e - b);
      }
    }
    sentinel_of_level[l] = slot[ord[p + cnt - 1u]];
    ++nslices;
    p += cnt;
  }
  H.entries = S.col.size();
  H.depth   = depth;
  H.slices  = nslices;
  // ---- concatenate the private streams; descriptor = {offset (words / 4), segments, 0, 0, first sizes}
  std::size_t total = 0;
  for (unsigned w = 0; w < nwarps; ++w) total += ws[w].size();
  if (total / 4u > 0xffffffffull) throw std::length_error("warp streams too large");
  H.stream.reserve(total);
  H.max_segs = 0;
  unsigned seg_base = 0;
  for (unsigned w = 0; w < nwarps; ++w) {
    unsigned *d = H.wdesc.data() + static_cast<std::size_t>(w) * 8u;
    d[0]        = static_cast<unsigned>(H.stream.size() / 4u);
    d[1]        = static_cast<unsigned>(seg_off[w].size());
    d[2]        = seg_base;  // first segment of the warp in the global numbering (trace records)
    seg_base += d[1];
    H.max_segs  = std::max<std::size_t>(H.max_segs, seg_off[w].size());
    H.stream.insert(H.stream.end(), ws[w].begin(), ws[w].end());
  }
  // segment sizes for the ring: wdesc[4..7] = sizes (in 16-byte units) of the first 4 segments, header
  // word 1 of segment k = size of segment k + stages (set by finalize_ring)
  H.seg_off = std::move(seg_off);
  if (ws_env("HIFIR_B200_WS_STATS", 0)) {  // developer: segments by entries per lane
    std::size_t hist[kWsU + 1] = {0}, copies = 0;
    for (unsigned w = 0; w < nwarps; ++w)
      for (unsigned off : H.seg_off[w]) {
        const unsigned hx = ws[w][off];
        if ((hx >> 16) & kSegCopy)
          ++copies;
        else
          ++hist[std::min(kWsU, hx & 0xffu)];
      }
    std::fprintf(stderr, "[ws stats] segments %zu copy %zu by width:", H.nsegs, copies);
    for (unsigned u = 1; u <= kWsU; ++u) std::fprintf(stderr, " %u:%zu", u, hist[u]);
    std::fprintf(stderr, "\n");
  }
}

// header word 1 of segment k = size (16-byte units) of segment k + stages of the same warp; the
// descriptor carries the sizes of the first `stages` segments
void ws_finalize_ring(WsHost &H, unsigned stages) {
  if (stages > 4u) throw std::logic_error("at most 4 ring stages");
  for (unsigned w = 0; w < H.nwarps; ++w) {
    unsigned *                   d   = H.wdesc.data() + static_cast<std::size_t>(w) * 8u;
    const std::vector<unsigned> &so  = H.seg_off[w];
    const std::size_t            base = static_cast<std::size_t>(d[0]) * 4u, ns = so.size();
    const std::size_t            end  = w + 1 < H.nwarps ? static_cast<std::size_t>(H.wdesc[(w + 1) * 8u]) * 4u : H.stream.size();
    auto size16 = [&](std::size_t k) {
      const std::size_t e = k + 1 < ns ? base + so[k + 1] : end;
      return static_cast<unsigned>((e - (base + so[k])) / 4u);
    };
    for (unsigned s = 0; s < 4u; ++s) d[4 + s] = s < ns ? size16(s) : 0u;
    for (std::size_t k = 0; k < ns; ++k) H.stream[base + so[k] + 1u] = k + stages < ns ? size16(k + stages) : 0u;
  }
}

// Fused L-then-U plan: warp w's stream = its L segments followed by its U segments (flagged kSegUpper,
// levels continued after the L levels).  One launch serves the whole  U^{-1} D^{-1} L^{-1}  solve: the
// ring keeps running across the seam, and the first U rows simply poll the last L rows' tags.
void ws_concat_ldu(const WsHost &L, const WsHost &U, WsHost &H) {
  if (L.nwarps != U.nwarps) throw std::logic_error("ws_concat_ldu: plans of different width");
  H          = WsHost();
  H.nwarps   = L.nwarps;
  H.nslots   = std::max(L.nslots, U.nslots);
  H.depth    = L.depth + U.depth;
  H.slices   = L.slices + U.slices;
  H.entries  = L.entries + U.entries;
  H.padded   = L.padded + U.padded;
  H.nsegs    = L.nsegs + U.nsegs;
  H.slot_of  = U.slot_of;  // the final solution is the U sweep's
  H.wdesc.assign(static_cast<std::size_t>(H.nwarps) * 8u, 0u);
  H.seg_off.assign(H.nwarps, {});
  H.stream.reserve(L.stream.size() + U.stream.size());
  unsigned seg_base = 0;
  auto     part = [](const WsHost &P, unsigned w, const unsigned *&b, const unsigned *&e) {
    b = P.stream.data() + static_cast<std::size_t>(P.wdesc[static_cast<std::size_t>(w) * 8u]) * 4u;
    e = w + 1 < P.nwarps ? P.stream.data() + static_cast<std::size_t>(P.wdesc[static_cast<std::size_t>(w + 1) * 8u]) * 4u
                         : P.stream.data() + P.stream.size();
  };
  for (unsigned w = 0; w < H.nwarps; ++w) {
    unsigned *d = H.wdesc.data() + static_cast<std::size_t>(w) * 8u;
    d[0]        = static_cast<unsigned>(H.stream.size() / 4u);
    const unsigned *b, *e;
    part(L, w, b, e);
    const std::size_t lwords = static_cast<std::size_t>(e - b);
    H.stream.insert(H.stream.end(), b, e);
    H.seg_off[w] = L.seg_off[w];
    part(U, w, b, e);
    const std::size_t o0 = H.stream.size();
    H.stream.insert(H.stream.end(), b, e);
    for (unsigned so : U.seg_off[w]) {
      H.seg_off[w].push_back(static_cast<unsigned>(lwords + so));
      unsigned *hd = H.stream.data() + o0 + so;
      hd[0] |= kSegUpper << 16;
      hd[3] += L.depth;
    }
    d[1] = static_cast<unsigned>(H.seg_off[w].size());
    d[2] = seg_base;
    seg_base += d[1];
    H.max_segs = std::max<std::size_t>(H.max_segs, H.seg_off[w].size());
  }
}

// The warps' streams of a packed plan in an order the device can run them: every warp in stream order, a
// segment as soon as its sentinel, every slot it gathers and -- U part of a fused plan -- the L results it
// reads as right-hand sides are published.  What a segment computes does not depend on the order in which
// ready segments of different warps run, so this walk needs no creation order: it serves a plan copied
// back from the device as well.  run(warp, header) is called for every segment that runs; pos (out):
// segments run per warp.  Returns the number of segments that can never run (0: deadlock free).
template <class F>
std::size_t ws_walk_dataflow(const WsHost &H, bool fused, std::vector<std::size_t> &pos, F &&run) {
  std::vector<char> ready[2] = {std::vector<char>(H.nslots, 0), std::vector<char>(fused ? H.nslots : 0u, 0)};
  pos.assign(H.nwarps, 0);
  std::size_t left = 0;
  for (unsigned w = 0; w < H.nwarps; ++w) left += H.seg_off[w].size();
  for (bool progress = true; progress && left;) {
    progress = false;
    for (unsigned w = 0; w < H.nwarps; ++w) {
      const std::size_t base = static_cast<std::size_t>(H.wdesc[static_cast<std::size_t>(w) * 8u]) * 4u;
      while (pos[w] < H.seg_off[w].size()) {
        const unsigned *hd    = H.stream.data() + base + H.seg_off[w][pos[w]];
        const unsigned  width = hd[0] & 0xffu, flags = hd[0] >> 16;
        const bool      copy  = (flags & kSegCopy) != 0u, u2 = fused && (flags & kSegUpper) != 0u;
        std::vector<char> &rd    = ready[u2 ? 1 : 0];
        const unsigned     nrow  = copy ? width * 32u : 32u;
        const unsigned *   codes = hd + kWsHdrWords, *slots = codes + nrow;
        bool               ok    = hd[2] == kWsNone || rd[hd[2]];
        if (ok && !copy) {
          const unsigned *cols = hd + kWsHdrWords + 64u;
          for (unsigned k = 0; k < width * 32u && ok; ++k)
            if (cols[k] != kWsNone && !rd[cols[k]]) ok = false;
        }
        for (unsigned r = 0; u2 && r < nrow && ok; ++r)
          if (slots[r] != kWsNone && !(codes[r] & kCodeZeroRhs) && !ready[0][codes[r] & kCodeSlotMask]) ok = false;
        if (!ok) break;
        run(w, hd);
        if (copy || (flags & kSegLast))
          for (unsigned r = 0; r < nrow; ++r)
            if (slots[r] != kWsNone) rd[slots[r]] = 1;
        ++pos[w];
        --left;
        progress = true;
      }
    }
  }
  return left;
}

// CPU emulation of the warp-stream sweep on the packed data, in the device's arithmetic order: per-lane fma
// over the entry positions, the shfl_xor butterfly of the device, one accumulator per lane of every warp
// (a slice of several segments carries it from one segment to the next).  x has H.nslots entries.
// parity < 0: plain values.  parity 0 / 1: every published value goes through tag_set (its last mantissa
// bit replaced by the parity) before any consumer reads it, as on the device, and the right-hand side of an
// upper sweep -- on the device the L sweep's tagged result -- is tagged as well.  x2 (fused plan): the U
// segments publish to x2 and read their right-hand side from the L segments' results in x.
void ws_host_emulate_packed(const WsHost &H, bool upper, bool f32, const double *rhs, const double *diag, double *x,
                            int parity, double *x2) {
  const bool          fused = x2 != nullptr;
  std::vector<double> accs(static_cast<std::size_t>(H.nwarps) * 32u, 0.0);
  std::vector<std::size_t> pos;
  auto pub = [&](double v) { return parity < 0 ? v : tag_set_host(v, static_cast<unsigned>(parity)); };
  const std::size_t stuck = ws_walk_dataflow(H, fused, pos, [&](unsigned w, const unsigned *hd) {
    const unsigned width = hd[0] & 0xffu, z = (hd[0] >> 8) & 0xffu, flags = hd[0] >> 16;
    const bool     up    = fused ? (flags & kSegUpper) != 0u : upper;
    double *       xw    = fused && up ? x2 : x;
    const double * rh    = fused && up ? x : rhs;  // U part of a fused plan: the L segments' results
    double *       acc   = accs.data() + static_cast<std::size_t>(w) * 32u;
    auto rhs_of = [&](unsigned code) {
      if (code & kCodeZeroRhs) return 0.0;
      const unsigned r = code & kCodeSlotMask;
      return up ? pub(rh[r]) / diag[r] : rh[r];
    };
    if (flags & kSegCopy) {
      const unsigned *codes = hd + kWsHdrWords, *slots = codes + width * 32u;
      for (unsigned r = 0; r < width * 32u; ++r)
        if (slots[r] != kWsNone) xw[slots[r]] = pub(rhs_of(codes[r]));
      return;
    }
    const unsigned *     codes = hd + kWsHdrWords, *slots = codes + 32u, *cols = slots + 32u;
    const unsigned char *vals  = reinterpret_cast<const unsigned char *>(cols + width * 32u);
    const unsigned       lpr   = 1u << z;
    for (unsigned j = 0; j < 32u; ++j) {
      if (flags & kSegFirst) acc[j] = ((j & (lpr - 1u)) == 0u && slots[j] != kWsNone) ? rhs_of(codes[j]) : 0.0;
      for (unsigned u = 0; u < width; ++u) {
        const unsigned c = cols[u * 32u + j];
        if (c == kWsNone) continue;
        double v;
        if (f32) {
          float f;
          std::memcpy(&f, vals + static_cast<std::size_t>(u * 32u + j) * 4u, 4);
          v = f;
        } else {
          std::memcpy(&v, vals + static_cast<std::size_t>(u * 32u + j) * 8u, 8);
        }
        acc[j] = std::fma(-v, xw[c], acc[j]);
      }
    }
    if (flags & kSegLast) {
      for (unsigned o = lpr >> 1; o > 0; o >>= 1) {  // the butterfly of the device (shfl_xor)
        double nw[32];
        for (unsigned j = 0; j < 32u; ++j) nw[j] = acc[j] + acc[j ^ o];
        std::memcpy(acc, nw, sizeof(nw));
      }
      for (unsigned j = 0; j < 32u; j += lpr)
        if (slots[j] != kWsNone) xw[slots[j]] = pub(acc[j]);
    }
  });
  if (stuck) throw std::logic_error("warp-stream emulation: " + std::to_string(stuck) + " segments can never run");
}

// Dataflow check of a packed plan (host only): returns the number of segments that can never run (0 = the
// static schedule is deadlock free).
std::size_t ws_check_schedule(const WsHost &H, bool f32, std::string *why) {
  std::vector<std::size_t> pos;
  (void)f32;
  const std::size_t left = ws_walk_dataflow(H, false, pos, [](unsigned, const unsigned *) {});
  if (left && why) {
    for (unsigned w = 0; w < H.nwarps && why->size() < 400; ++w)
      if (pos[w] < H.seg_off[w].size()) {
        const std::size_t base = static_cast<std::size_t>(H.wdesc[static_cast<std::size_t>(w) * 8u]) * 4u;
        const unsigned *  hd   = H.stream.data() + base + H.seg_off[w][pos[w]];
        *why += " warp " + std::to_string(w) + " seg " + std::to_string(pos[w]) + " level " + std::to_string(hd[3]) +
                " sentinel " + std::to_string(hd[2]) + ";";
      }
  }
  return left;
}

// Developer tool (host only): the segment dependency graph of a packed plan in the trace numbering
// (warp by warp).  dep_ptr[nsegs + 1], dep_idx = distinct producer segments of every segment.
void ws_segment_graph(const WsHost &H, std::vector<unsigned> &dep_ptr, std::vector<unsigned> &dep_idx) {
  std::vector<unsigned> seg_of_slot(H.nslots, kWsNone), base(H.nwarps + 1u, 0u);
  for (unsigned w = 0; w < H.nwarps; ++w) base[w + 1] = base[w] + static_cast<unsigned>(H.seg_off[w].size());
  auto header = [&](unsigned w, std::size_t k) {
    return H.stream.data() + static_cast<std::size_t>(H.wdesc[static_cast<std::size_t>(w) * 8u]) * 4u + H.seg_off[w][k];
  };
  for (unsigned w = 0; w < H.nwarps; ++w)
    for (std::size_t k = 0; k < H.seg_off[w].size(); ++k) {
      const unsigned *hd = header(w, k);
      const unsigned  width = hd[0] & 0xffu, flags = hd[0] >> 16;
      if (flags & kSegCopy) {
        const unsigned *slots = hd + kWsHdrWords + width * 32u;
        for (unsigned r = 0; r < width * 32u; ++r)
          if (slots[r] != kWsNone) seg_of_slot[slots[r]] = base[w] + static_cast<unsigned>(k);
      } else if (flags & kSegLast) {
        const unsigned *slots = hd + kWsHdrWords + 32u;
        for (unsigned j = 0; j < 32u; ++j)
          if (slots[j] != kWsNone) seg_of_slot[slots[j]] = base[w] + static_cast<unsigned>(k);
      }
    }
  dep_ptr.assign(1, 0u);
  dep_idx.clear();
  std::vector<unsigned> tmp;
  for (unsigned w = 0; w < H.nwarps; ++w)
    for (std::size_t k = 0; k < H.seg_off[w].size(); ++k) {
      const unsigned *hd = header(w, k);
      const unsigned  width = hd[0] & 0xffu, flags = hd[0] >> 16;
      tmp.clear();
      if (!(flags & kSegCopy)) {
        const unsigned *cols = hd + kWsHdrWords + 64u;
        for (unsigned q = 0; q < width * 32u; ++q)
          if (cols[q] != kWsNone) tmp.push_back(seg_of_slot[cols[q]]);
        std::sort(tmp.begin(), tmp.end());
        tmp.erase(std::unique(tmp.begin(), tmp.end()), tmp.end());
      }
      dep_idx.insert(dep_idx.end(), tmp.begin(), tmp.end());
      dep_ptr.push_back(static_cast<unsigned>(dep_idx.size()));
    }
}

// ---- device ----------------------------------------------------------------------------
namespace {
__device__ __forceinline__ unsigned ws_smem_addr(const void *p) { return static_cast<unsigned>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void ws_mbar_init(unsigned bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void ws_mbar_expect_tx(unsigned bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// The factor stream is touched once per sweep: EVICT-FIRST in L2, so that it does not push the
// solution buffers and right-hand sides (gathered at random, re-used ~9x) out to HBM -- with the
// default policy the trace showed first-try gathers of 0.7 us and right-hand side loads of ~1.2 us
// (HBM latency) on level sets whose producers had long finished.
__device__ __forceinline__ unsigned long long ws_policy_evict_first() {
  unsigned long long pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void ws_tma_g2s(unsigned dst, const void *src, unsigned bytes, unsigned bar,
                                           unsigned long long policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(dst),
      "l"(src), "r"(bytes), "r"(bar), "l"(policy)
      : "memory");
}
__device__ __forceinline__ bool ws_mbar_try_wait(unsigned bar, unsigned phase) {
  unsigned ok;
  asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(ok)
               : "r"(bar), "r"(phase)
               : "memory");
  return ok != 0;
}
// first-try gather through L1 (ld.global.ca): lanes of different gather instructions and warps of the
// SM that hit the same 128-byte line share one L2 request; a stale line only means "not ready" (the tag
// travels with the value) and the re-poll goes to L2
__device__ __forceinline__ unsigned long long ws_ld_l1(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.global.ca.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ int ws_ld_poll_i32(const int *p) {
  int v;
  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void ws_publish(unsigned long long *p, unsigned long long v, int use_store) {
  if (use_store) {
    st_publish(p, v);
  } else {
    // through the L2 atomic unit: visible to pollers ~0.2 us earlier than a plain store (round 1 A/B)
    unsigned long long old;
    asm volatile("atom.relaxed.gpu.global.exch.b64 %0, [%1], %2;" : "=l"(old) : "l"(p), "l"(v) : "memory");
  }
}
}  // namespace

struct WsParams {
  const unsigned *          wdesc;
  const unsigned *          stream;
  const double *            rhs_plain;
  const unsigned long long *rhs_tagged;
  const double *            diag;
  unsigned long long *      x;
  unsigned long long *      x2;    // fused L-then-U sweep: solution of the U sweep (x: of the L sweep)
  int *                     sync;  // [0] frontier hint (highest level some warp finished a slice of)
  int *                     error_flag;
  unsigned                  parity, window, adm_sleep;
  int                       publish_st;
  int                       l1_first;    // first-try gathers through L1
  unsigned                  spin_limit;  // poll rounds after which a wait gives up (and every other wait with it)
  unsigned                  poll_sleep;  // multi-rhs: nanoseconds between two poll rounds of a batch (0: none)
  unsigned long long *      trace;  // kTrace: 4 words per segment (decoded, admitted, gathered | rounds, published | level)
};

// One persistent CTA per SM, kWarps warps; warp (blockIdx.x + gridDim.x * warp) owns stream
// wdesc[..].  kStages ring stages of kStageBytes each per warp.
// first failing wait: remember where (error_flag[1..]: claimed, global warp, segment, level, kind, detail, upper)
__device__ __noinline__ void ws_fail(const WsParams &P, unsigned gw, unsigned k, unsigned level, int kind, unsigned detail) {
  if (atomicCAS(P.error_flag + 1, 0, 1) == 0) {
    P.error_flag[2] = static_cast<int>(gw);
    P.error_flag[3] = static_cast<int>(k);
    P.error_flag[4] = static_cast<int>(level);
    P.error_flag[5] = kind;
    P.error_flag[6] = static_cast<int>(detail);
    P.error_flag[7] = static_cast<int>(P.parity);
    __threadfence();
  }
  atomicExch(P.error_flag, kind);
}
__device__ __forceinline__ bool ws_aborted(const WsParams &P) { return ws_ld_poll_i32(P.error_flag) != 0; }

__device__ __forceinline__ unsigned long long ws_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// MODE 0: L sweep, 1: U sweep, 2: fused L-then-U sweep (a segment's header says which factor it belongs to:
// L segments gather from / publish to x, U segments x2, and read their right-hand side from x)
template <int MODE, class VT, int kWarps, int kStages, bool kTrace, bool kPipe>
__global__ void __launch_bounds__(kWarps * 32, 1) wsweep_kernel(const WsParams P) {
  constexpr unsigned kStageBytes = (kWsHdrWords + 64u + kWsU * 32u * (sizeof(VT) == 4 ? 2u : 3u)) * 4u;
  extern __shared__ __align__(128) unsigned char smem[];
  const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  const unsigned gw   = blockIdx.x + gridDim.x * warp;
  const uint4    d0   = reinterpret_cast<const uint4 *>(P.wdesc)[2 * gw];
  const uint4    d1   = reinterpret_cast<const uint4 *>(P.wdesc)[2 * gw + 1];
  const unsigned nseg = d0.y;
  if (!nseg) return;  // warps never meet at a CTA barrier
  unsigned char *ring = smem + static_cast<std::size_t>(kWarps) * kStages * 8u + static_cast<std::size_t>(warp) * kStages * kStageBytes;
  const unsigned bar0 = ws_smem_addr(smem) + warp * kStages * 8u;
  const unsigned char *src = reinterpret_cast<const unsigned char *>(P.stream) + static_cast<std::size_t>(d0.x) * 16u;
  const unsigned long long policy = ws_policy_evict_first();
  if (lane == 0) {
    for (int s = 0; s < kStages; ++s) ws_mbar_init(bar0 + s * 8u, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const unsigned sz[4] = {d1.x, d1.y, d1.z, d1.w};
    for (int s = 0; s < kStages; ++s)
      if (sz[s]) {
        ws_mbar_expect_tx(bar0 + s * 8u, sz[s] * 16u);
        ws_tma_g2s(ws_smem_addr(ring + s * kStageBytes), src, sz[s] * 16u, bar0 + s * 8u, policy);
        src += static_cast<std::size_t>(sz[s]) * 16u;
      }
  }
  __syncwarp();
  double         acc      = 0.0;
  unsigned       my_front = 0;
  const unsigned parity   = P.parity;
  // The ring stage of a segment is refilled (an ASYNC-proxy write by the TMA unit) at the END of the
  // segment, in program order after instructions that consume every register the segment's
  // shared-memory reads wrote: a warp issues in order and an instruction can not issue before its
  // source registers have arrived, so by then every read of the stage has RETURNED.  (Refilling
  // right after the reads were ISSUED is a race: under load a shared-memory read sits in the SM's
  // load/store queue behind thousands of cycles of scattered gathers -- longer than a bulk copy from
  // L2 takes to land.  Measured: stale stages -> wrong indices -> illegal addresses / rows that
  // never become ready.)
  unsigned           cc[kWsU];          // slot indices / gathered words of the current segment
  unsigned long long g[kWsU];
  // a position without entry keeps what an earlier segment gathered there -- a word that carries the tag
  // (initially: "zero carrying the tag"): the combined tag test below needs no per-position mask
#pragma unroll
  for (unsigned u = 0; u < kWsU; ++u) g[u] = static_cast<unsigned long long>(P.parity);
  bool               have_cur = false;  // kPipe: they were requested during the previous segment
  auto refill = [&](unsigned stage, unsigned size16) {
    __syncwarp();
    if (lane == 0 && size16) {
      ws_mbar_expect_tx(bar0 + stage * 8u, size16 * 16u);
      ws_tma_g2s(ws_smem_addr(ring + stage * kStageBytes), src, size16 * 16u, bar0 + stage * 8u, policy);
      src += static_cast<std::size_t>(size16) * 16u;
    }
  };
  for (unsigned k = 0; k < nseg; ++k) {
    const unsigned stage = k % kStages, phase = (k / kStages) & 1u;
    {
      unsigned spins = 0;
      bool     ok    = true;
      while (!ws_mbar_try_wait(bar0 + stage * 8u, phase)) {
        if (++spins > P.spin_limit || ((spins & 1023u) == 1023u && ws_aborted(P))) {
          ok = false;
          break;
        }
      }
      if (!ok) {  // the stage never arrived (or another warp gave up): stop, never decode garbage
        if (lane == 0 && !ws_aborted(P)) ws_fail(P, gw, k, 0u, 2, stage);
        return;
      }
    }
    const unsigned *sg    = reinterpret_cast<const unsigned *>(ring + stage * kStageBytes);
    const uint4     hd    = *reinterpret_cast<const uint4 *>(sg);
    const unsigned  width = hd.x & 0xffu, z = (hd.x >> 8) & 0xffu, flags = hd.x >> 16;
    const bool      UPPER = MODE == 2 ? (flags & kSegUpper) != 0u : MODE == 1;
    unsigned long long *const       xw  = (MODE == 2 && UPPER) ? P.x2 : P.x;           // this factor's solution
    const unsigned long long *const rht = MODE == 2 ? P.x : P.rhs_tagged;              // U: the L sweep's result
    unsigned long long *tr = kTrace ? P.trace + 4ull * (d0.z + k) : nullptr;
    unsigned long long  t_dec = 0;
    if (kTrace) t_dec = ws_timer_ns();
    if (flags & kSegCopy) {
      // rows without entries: x = rhs, 8 per lane, all loads in flight together
      unsigned code[kWsU], slot[kWsU];
      double   v[kWsU];
#pragma unroll
      for (unsigned u = 0; u < kWsU; ++u) {
        code[u] = slot[u] = kWsNone;
        if (u < width) {
          code[u] = sg[kWsHdrWords + u * 32u + lane];
          slot[u] = sg[kWsHdrWords + (width + u) * 32u + lane];
        }
      }
#pragma unroll
      for (unsigned u = 0; u < kWsU; ++u) {
        v[u] = 0.0;
        if (slot[u] != kWsNone && !(code[u] & kCodeZeroRhs)) {
          const unsigned r = code[u] & kCodeSlotMask;
          if (UPPER) {
            unsigned long long t = ld_poll(rht + r);
            for (unsigned spins = 0; !tag_ready(t, parity); t = ld_poll(rht + r))
              if (++spins > P.spin_limit || ((spins & 255u) == 255u && ws_aborted(P))) {
                if (!ws_aborted(P)) ws_fail(P, gw, k, hd.w, 3, r);
                break;
              }
            v[u] = tag_value(t) / P.diag[r];
          } else {
            v[u] = P.rhs_plain[r];
          }
        }
      }
#pragma unroll
      for (unsigned u = 0; u < kWsU; ++u)
        if (slot[u] != kWsNone) st_publish(xw + slot[u], tag_set(v[u], parity));  // consumes code and slot
      refill(stage, hd.y);
      have_cur = false;
      if (lane == 0 && hd.w > my_front + 3u) {
        my_front = hd.w;
        atomicMax(P.sync, static_cast<int>(hd.w));
      }
      if (kTrace && lane == 0) tr[0] = t_dec, tr[1] = tr[2] = 0, tr[3] = ((ws_timer_ns() - t_dec) << 16) | hd.w | 0x8000u;
      continue;
    }
    // ---- a slice segment: slot indices first, the gathers are the long pole.  With kPipe the
    // first-try gathers of this segment were issued while the PREVIOUS segment was being finished.
    unsigned long long t_adm = 0, t_gat = 0;
    if (!have_cur) {
#pragma unroll
      for (unsigned u = 0; u < kWsU; ++u) {
        cc[u] = kWsNone;
        if (u < width) cc[u] = sg[kWsHdrWords + 64u + u * 32u + lane];
      }
      // ---- admission (only a warp that jumps ahead carries a sentinel): the sentinel row of level
      // (this - window) is published
      if (hd.z != kWsNone) {
        if (lane == 0) {
          unsigned       spins = 0;
          const unsigned need  = hd.w - P.window;
          while (!tag_ready(ld_poll(xw + hd.z), parity)) {
            // far from the frontier: sleep in proportion to the distance; close to it: spin on the sentinel
            const unsigned f = static_cast<unsigned>(ws_ld_poll_i32(P.sync));
            if (need > f + 4u) __nanosleep(min((need - f) * P.adm_sleep, 20000u));
            if (++spins > P.spin_limit || ((spins & 63u) == 63u && ws_aborted(P))) {
              if (!ws_aborted(P)) ws_fail(P, gw, k, hd.w, 4, hd.z);
              break;
            }
          }
        }
        __syncwarp();
      }
      if (kTrace) t_adm = ws_timer_ns();
      // ---- gather all entries optimistically (re-polled below if not ready)
      if (P.l1_first) {
#pragma unroll
        for (unsigned u = 0; u < kWsU; ++u)
          if (cc[u] != kWsNone) g[u] = ws_ld_l1(xw + cc[u]);
      } else {
#pragma unroll
        for (unsigned u = 0; u < kWsU; ++u)
          if (cc[u] != kWsNone) g[u] = ld_poll(xw + cc[u]);
      }
    } else if (kTrace) {
      t_adm = ws_timer_ns();
    }
    // ---- software pipeline: the next segment's slot indices are in its stage already (the ring runs
    // ahead); its first-try gathers go out NOW, so that they travel while this segment is finished.
    // (A dependency-free pass of the unpipelined kernel took as long as the real sweep: a warp had
    // gathers in flight only ~1/3 of the time.)  A segment with a sentinel is not pre-gathered.
    bool               have_nxt = false;
    unsigned           ccn[kWsU];
    unsigned long long gn[kWsU];
    if (kPipe) {
#pragma unroll
      for (unsigned u = 0; u < kWsU; ++u) gn[u] = static_cast<unsigned long long>(parity);
    }
    if (kPipe && k + 1u < nseg) {
      const unsigned st1 = (k + 1u) % kStages, ph1 = ((k + 1u) / kStages) & 1u;
      if (__all_sync(0xffffffffu, ws_mbar_try_wait(bar0 + st1 * 8u, ph1))) {
        const unsigned *sg1 = reinterpret_cast<const unsigned *>(ring + st1 * kStageBytes);
        const unsigned  hx1 = sg1[0], hz1 = sg1[2], w1 = hx1 & 0xffu;
        const unsigned long long *const xn = (MODE == 2 && ((hx1 >> 16) & kSegUpper)) ? P.x2 : P.x;
        if (!((hx1 >> 16) & kSegCopy) && hz1 == kWsNone) {
#pragma unroll
          for (unsigned u = 0; u < kWsU; ++u) {
            ccn[u] = kWsNone;
            if (u < w1) ccn[u] = sg1[kWsHdrWords + 64u + u * 32u + lane];
          }
#pragma unroll
          for (unsigned u = 0; u < kWsU; ++u)
            if (ccn[u] != kWsNone) gn[u] = ld_poll(xn + ccn[u]);
          have_nxt = true;
        }
      }
    }
    const unsigned code = sg[kWsHdrWords + lane];
    const unsigned slot = sg[kWsHdrWords + 32u + lane];
    const unsigned lpr  = 1u << z;
    const bool     own  = slot != kWsNone && (lane & (lpr - 1u)) == 0u;
    double             rhs_v  = 0.0, dg = 1.0;
    unsigned long long rhs_t  = 0;
    const bool         want_r = (flags & kSegFirst) && own && !(code & kCodeZeroRhs);
    if (want_r) {
      const unsigned r = code & kCodeSlotMask;
      if (UPPER) {
        rhs_t = ld_poll(rht + r);
        dg    = P.diag[r];
      } else {
        rhs_v = P.rhs_plain[r];
      }
    }
    // fast path: one combined test of all tags (the common case: everything was ready)
    unsigned pend = 0, nrounds = 0;
    {
      unsigned bad = 0;
#pragma unroll
      for (unsigned u = 0; u < kWsU; ++u) bad |= static_cast<unsigned>(g[u]) ^ parity;
      if (UPPER && want_r) bad |= static_cast<unsigned>(rhs_t) ^ parity;
      if (bad & 1u) {
#pragma unroll
        for (unsigned u = 0; u < kWsU; ++u)
          if (cc[u] != kWsNone && !tag_ready(g[u], parity)) pend |= 1u << u;
        if (UPPER && want_r && !tag_ready(rhs_t, parity)) pend |= 1u << kWsU;
      }
    }
    if (kTrace) {
      const unsigned any = __ballot_sync(0xffffffffu, pend != 0u);  // depends on every first-try gather
      t_gat              = ws_timer_ns() + (any == 0xdeadbeefu ? 1u : 0u);
    }
    for (unsigned rounds = 0; __any_sync(0xffffffffu, pend != 0u);) {
      if (kTrace) ++nrounds;
      if (P.poll_sleep) __nanosleep(P.poll_sleep);  // developer knob: issue slots for the other warps instead of polls
#pragma unroll
      for (unsigned u = 0; u < kWsU; ++u)
        if (pend & (1u << u)) g[u] = ld_poll(xw + cc[u]);
      if (UPPER && (pend & (1u << kWsU))) rhs_t = ld_poll(rht + (code & kCodeSlotMask));
      // still pending: the low bit differs from the tag.  Computed for every position without a branch (a
      // position that was not re-read is ready or holds no entry: its pend bit is clear already) -- this loop
      // ran ~1.5 times per segment at 110 instructions per round (32 % of the kernel's instructions)
      unsigned still = 0;
#pragma unroll
      for (unsigned u = 0; u < kWsU; ++u) still |= ((static_cast<unsigned>(g[u]) ^ parity) & 1u) << u;
      if (UPPER) still |= ((static_cast<unsigned>(rhs_t) ^ parity) & 1u) << kWsU;
      pend &= still;
      if (++rounds > P.spin_limit || ((rounds & 255u) == 255u && ws_aborted(P))) {
        // hang guard: a dependency never became ready (or another warp gave up) -- remember where, go on
        if (pend && !ws_aborted(P)) {
          unsigned which = kWsNone;
#pragma unroll
          for (unsigned u = 0; u < kWsU; ++u)
            if (pend & (1u << u)) which = cc[u];
          ws_fail(P, gw, k, hd.w, 1, which);
        }
        break;
      }
    }
    if (flags & kSegFirst) {
      acc = 0.0;
      // b_i (L sweep) or (L^{-1} b)_i / d_i with a true division (prec_solve.hpp:219, :256-259)
      if (want_r) acc = UPPER ? tag_value(rhs_t) / dg : rhs_v;
    }
    // the factor values are read from the stage only now (no registers held across the gather wait);
    // every value that is read is consumed by its multiply-add (same predicate): all reads of the stage
    // have returned before it is refilled
    const VT *sv = reinterpret_cast<const VT *>(sg + kWsHdrWords + 64u + width * 32u);
#pragma unroll
    for (unsigned u = 0; u < kWsU; ++u)
      if (cc[u] != kWsNone) acc = fma(-static_cast<double>(sv[u * 32u + lane]), tag_value(g[u]), acc);
    if (flags & kSegLast) {
      for (unsigned o = lpr >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (own) ws_publish(xw + slot, tag_set(acc, parity), P.publish_st);
    }
    {
      // the refill must depend on acc (see above) WITHOUT changing its size: choose between the header
      // word and a second, volatile read of the same word -- equal values the compiler can not prove equal
      const unsigned y2 = *reinterpret_cast<const volatile unsigned *>(sg + 1);
      refill(stage, acc == 1.2345e300 ? y2 : hd.y);
    }
    have_cur = have_nxt;
    if (have_nxt) {
#pragma unroll
      for (unsigned u = 0; u < kWsU; ++u) cc[u] = ccn[u], g[u] = gn[u];
    }
    if (lane == 0 && hd.w > my_front + 3u) {  // frontier hint for the sleeping jumpers, every 4th level
      my_front = hd.w;
      atomicMax(P.sync, static_cast<int>(hd.w));
    }
    if (kTrace && lane == 0) {
      tr[0] = t_dec;
      tr[1] = t_adm - t_dec;
      tr[2] = ((t_gat - t_dec) << 8) | min(nrounds, 255u);
      tr[3] = ((ws_timer_ns() - t_dec) << 16) | hd.w;
    }
  }
}

// ---- multi-rhs: the same warp streams, lanes ACROSS the columns -------------------------------
// Row-interleaved blocks X[slot * NC + c] (the Array<std::array<T,Nrhs>> layout of
// hif::HIF::solve_mrhs, builder.hpp:433-445; per-column arithmetic = CCS::solve_as_strict_lower /
// _upper_mrhs, CompressedStorage.hpp:2286-2301, 2376-2393).  NC = 2 G columns, G in {4, 8, 16, 32}.
//
// The single-rhs kernel gives every lane its own entries: 32 scattered 8-byte gathers per instruction,
// one L1 wavefront each -- that is its throughput bound.  With NC columns the unit of dependency is a
// ROW of NC values: G consecutive lanes own the columns (two each, one 16-byte load), so one gather
// instruction moves 32 / G whole rows of 16 G bytes -- full 128-byte lines, 4 wavefronts for 512 bytes
// instead of 32 for 256.  Consequently:
//   * lane group grp = lane / G works on one row of the segment at a time (a row's entry slots are
//     walked serially: the sum over the entries needs no shuffle), 32 / G rows side by side, two rows
//     per group in flight (RIF) with B entries each;
//   * a segment with fewer rows than groups (long rows: 2^z lanes per row in the single-rhs layout)
//     splits each row's entry slots over K groups and adds the K partial sums with shuffles;
//   * the packed streams, the tags, the sentinel admission and the ring refill are those of
//     wsweep_kernel MODE 2 (fused L-then-U plan): one launch per LDU solve for all NC columns, the
//     factor is read from HBM once per NC columns.
__device__ __forceinline__ void ws_ld_poll2(const unsigned long long *p, unsigned long long &a, unsigned long long &b) {
  asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ void ws_st_publish2(unsigned long long *p, unsigned long long a, unsigned long long b) {
  asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(a), "l"(b) : "memory");
}
// the same through the L2 atomic unit (16-byte exchange): developer experiment, HIFIR_B200_MRHS_PUBLISH_ATOM=1
__device__ __forceinline__ void ws_atom_publish2(unsigned long long *p, unsigned long long a, unsigned long long b) {
  asm volatile(
      "{\n\t.reg .b128 v, o;\n\tmov.b128 v, {%1, %2};\n\tatom.relaxed.gpu.global.exch.b128 o, [%0], v;\n\t}" ::"l"(p),
      "l"(a), "l"(b)
      : "memory");
}
__device__ __forceinline__ bool ws_ready2(unsigned long long a, unsigned long long b, unsigned parity) {
  return !(((static_cast<unsigned>(a) ^ parity) | (static_cast<unsigned>(b) ^ parity)) & 1u);
}

template <class VT, int G, unsigned B>
__global__ void __launch_bounds__(24 * 32, 1) wsweep_cols_kernel(const WsParams P) {
  constexpr int      kWarps = 24, kStages = 2;
  constexpr unsigned NC = 2u * G, EPI = 32u / G;  // columns; rows (or row parts) per gather instruction
  // B = 4 or 8 entries of a row in flight per lane (a second ROW in flight spills the gathered words --
  // 85 registers per thread at 24 warps -- and measured slower)
  constexpr unsigned kStageBytes = (kWsHdrWords + 64u + kWsU * 32u * (sizeof(VT) == 4 ? 2u : 3u)) * 4u;
  extern __shared__ __align__(128) unsigned char smem[];
  const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  const unsigned gw   = blockIdx.x + gridDim.x * warp;
  const uint4    d0   = reinterpret_cast<const uint4 *>(P.wdesc)[2 * gw];
  const uint4    d1   = reinterpret_cast<const uint4 *>(P.wdesc)[2 * gw + 1];
  const unsigned nseg = d0.y;
  if (!nseg) return;
  unsigned char *ring = smem + static_cast<std::size_t>(kWarps) * kStages * 8u + static_cast<std::size_t>(warp) * kStages * kStageBytes;
  const unsigned bar0 = ws_smem_addr(smem) + warp * kStages * 8u;
  const unsigned char *src = reinterpret_cast<const unsigned char *>(P.stream) + static_cast<std::size_t>(d0.x) * 16u;
  const unsigned long long policy = ws_policy_evict_first();
  if (lane == 0) {
    for (int s = 0; s < kStages; ++s) ws_mbar_init(bar0 + s * 8u, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    const unsigned sz[4] = {d1.x, d1.y, d1.z, d1.w};
    for (int s = 0; s < kStages; ++s)
      if (sz[s]) {
        ws_mbar_expect_tx(bar0 + s * 8u, sz[s] * 16u);
        ws_tma_g2s(ws_smem_addr(ring + s * kStageBytes), src, sz[s] * 16u, bar0 + s * 8u, policy);
        src += static_cast<std::size_t>(sz[s]) * 16u;
      }
  }
  __syncwarp();
  const unsigned parity = P.parity;
  const unsigned grp = lane / G, cp = (lane % G) * 2u;  // lane group; first of this lane's two columns
  unsigned       my_front = 0;
  // right-hand side of a row: b (L segments) or the L sweep's tagged result divided by d (U segments)
  auto rhs_issue = [&](bool upper, unsigned r, unsigned long long &t0, unsigned long long &t1, double &dg) {
    if (upper) {
      ws_ld_poll2(P.x + static_cast<std::size_t>(r) * NC + cp, t0, t1);
      dg = P.diag[r];
    } else {
      const double2 v = *reinterpret_cast<const double2 *>(P.rhs_plain + static_cast<std::size_t>(r) * NC + cp);
      t0 = static_cast<unsigned long long>(__double_as_longlong(v.x));
      t1 = static_cast<unsigned long long>(__double_as_longlong(v.y));
    }
  };
  auto rhs_finish = [&](bool upper, unsigned r, unsigned long long t0, unsigned long long t1, double dg, double &a0,
                        double &a1, unsigned k, unsigned level) {
    if (upper) {
      for (unsigned spins = 0; !ws_ready2(t0, t1, parity); ws_ld_poll2(P.x + static_cast<std::size_t>(r) * NC + cp, t0, t1))
        if (++spins > P.spin_limit || ((spins & 255u) == 255u && ws_aborted(P))) {
          if (!ws_aborted(P)) ws_fail(P, gw, k, level, 3, r);
          break;
        }
      a0 = tag_value(t0) / dg;  // true division (prec_solve.hpp:219)
      a1 = tag_value(t1) / dg;
    } else {
      a0 = __longlong_as_double(static_cast<long long>(t0));
      a1 = __longlong_as_double(static_cast<long long>(t1));
    }
  };
  for (unsigned k = 0; k < nseg; ++k) {
    const unsigned stage = k % kStages, phase = (k / kStages) & 1u;
    {
      unsigned spins = 0;
      bool     ok    = true;
      while (!ws_mbar_try_wait(bar0 + stage * 8u, phase)) {
        if (++spins > P.spin_limit || ((spins & 1023u) == 1023u && ws_aborted(P))) {
          ok = false;
          break;
        }
      }
      if (!ok) {
        if (lane == 0 && !ws_aborted(P)) ws_fail(P, gw, k, 0u, 2, stage);
        return;
      }
    }
    const unsigned *sg    = reinterpret_cast<const unsigned *>(ring + stage * kStageBytes);
    const uint4     hd    = *reinterpret_cast<const uint4 *>(sg);
    const unsigned  width = hd.x & 0xffu, z = (hd.x >> 8) & 0xffu, flags = hd.x >> 16;
    const bool      upper = (flags & kSegUpper) != 0u;
    unsigned long long *const xw = upper ? P.x2 : P.x;  // this factor's solution
    unsigned keep = 0;  // digest of everything read from the stage: the refill below depends on it
    if (flags & kSegCopy) {
      // rows without entries: x = rhs; width * 32 rows, four per lane group in flight
      const unsigned nrows = width * 32u;
      for (unsigned r0 = 0; r0 < nrows; r0 += EPI * 4u) {
        unsigned           code[4], slot[4];
        unsigned long long t0[4], t1[4];
        double             dg[4];
#pragma unroll
        for (unsigned j = 0; j < 4; ++j) {
          const unsigned row = r0 + j * EPI + grp;
          code[j]            = sg[kWsHdrWords + row];
          slot[j]            = sg[kWsHdrWords + nrows + row];
          keep ^= code[j] + slot[j];
          t0[j] = t1[j] = 0ull;
          dg[j]         = 1.0;
          if (slot[j] != kWsNone && !(code[j] & kCodeZeroRhs)) rhs_issue(upper, code[j] & kCodeSlotMask, t0[j], t1[j], dg[j]);
        }
#pragma unroll
        for (unsigned j = 0; j < 4; ++j)
          if (slot[j] != kWsNone) {
            double a0 = 0.0, a1 = 0.0;
            if (!(code[j] & kCodeZeroRhs)) rhs_finish(upper, code[j] & kCodeSlotMask, t0[j], t1[j], dg[j], a0, a1, k, hd.w);
            ws_st_publish2(xw + static_cast<std::size_t>(slot[j]) * NC + cp, tag_set(a0, parity), tag_set(a1, parity));
          }
      }
    } else {
      const unsigned lpr = 1u << z, R = 32u >> z;    // lanes per row of the single-rhs layout; rows
      const unsigned Rg  = R < EPI ? R : EPI;        // rows the lane groups work on side by side
      const unsigned K   = EPI / Rg;                 // lane groups that share one row
      const unsigned sub = grp % Rg, part = grp / Rg;
      if (hd.z != kWsNone) {  // admission of a warp that jumps ahead (throttle only)
        if (lane == 0) {
          unsigned       spins = 0;
          const unsigned need  = hd.w - P.window;
          while (!tag_ready(ld_poll(xw + static_cast<std::size_t>(hd.z) * NC), parity)) {
            const unsigned f = static_cast<unsigned>(ws_ld_poll_i32(P.sync));
            if (need > f + 4u) __nanosleep(min((need - f) * P.adm_sleep, 20000u));
            if (++spins > P.spin_limit || ((spins & 63u) == 63u && ws_aborted(P))) {
              if (!ws_aborted(P)) ws_fail(P, gw, k, hd.w, 4, hd.z);
              break;
            }
          }
        }
        __syncwarp();
      }
      const unsigned *sc    = sg + kWsHdrWords + 64u;
      const VT *      sv    = reinterpret_cast<const VT *>(sc + width * 32u);
      const bool      first = (flags & kSegFirst) != 0u, last = (flags & kSegLast) != 0u;
      // The entry slots of a row are walked in batches of B, addressed by a running pointer and compile-time
      // offsets (word of entry u of lane l of the row: u * 32 + first lane + l).  Layouts:
      //   CLS 0..2  2^CLS < B lanes per row: a batch wraps over the lanes, (u, l) = (0,0) .. (0,2^z-1) (1,0) ...;
      //             the row may end inside a batch (rem)
      //   CLS 3     B or more lanes per row, one lane group per row: consecutive lanes, then the next u
      //   CLS 4     K lane groups share the row: every K-th lane (the partial sums are added below)
      auto run = [&](auto cls_tag) {
        constexpr unsigned CLS = decltype(cls_tag)::value;
        for (unsigned r0 = 0; r0 < R; r0 += Rg) {
          const unsigned ol   = (r0 + sub) << z;  // the row's first lane in the single-rhs layout
          const unsigned code = sg[kWsHdrWords + ol], slot = sg[kWsHdrWords + 32u + ol];
          keep ^= code + slot;
          const bool live = slot != kWsNone, head = live && part == 0u;
          const bool want = head && first && !(code & kCodeZeroRhs);
          double     a0 = 0.0, a1 = 0.0, dg = 1.0;
          unsigned long long t0 = 0ull, t1 = 0ull;
          if (want)
            rhs_issue(upper, code & kCodeSlotMask, t0, t1, dg);
          else if (head && !first)
            // continuation of a slice of several segments (rows beyond 256 entries): the partial sums
            // were parked in the row's own slot under the OTHER tag (nobody consumes them)
            ws_ld_poll2(xw + static_cast<std::size_t>(slot) * NC + cp, t0, t1);
          // gathered rows; a slot without entry keeps an older (finite) row and meets the value 0.0
          unsigned long long g0[B], g1[B];
#pragma unroll
          for (unsigned j = 0; j < B; ++j) g0[j] = g1[j] = 0ull;
          bool firstb = true;
          auto batch  = [&](const unsigned *pc, const VT *pv, unsigned rem) {  // rem: slots left (CLS 0..2)
            unsigned col[B];
#pragma unroll
            for (unsigned j = 0; j < B; ++j) {
              const unsigned off = CLS <= 2u ? (j >> CLS) * 32u + (j & ((1u << CLS) - 1u)) : CLS == 3u ? j : j * K;
              col[j]             = kWsNone;
              if ((CLS >= 3u || j < rem) && live) col[j] = pc[off];
              if (col[j] != kWsNone) ws_ld_poll2(xw + static_cast<std::size_t>(col[j]) * NC + cp, g0[j], g1[j]);
            }
            unsigned bad = 0;
#pragma unroll
            for (unsigned j = 0; j < B; ++j)
              bad |= col[j] != kWsNone ? (static_cast<unsigned>(g0[j]) ^ parity) | (static_cast<unsigned>(g1[j]) ^ parity) : 0u;
            if (__any_sync(0xffffffffu, (bad & 1u) != 0u)) {
              // Some row was not published yet (right behind the frontier this is the common case: ~3 poll
              // rounds per batch were measured).  Every lane polls its own piece: letting only the first lane
              // of a group poll (1 sector instead of the row) costs one more round trip at the end and
              // measured 14 % slower -- the chain of dependent round trips is what bounds the sweep.
              unsigned pend = 0;
#pragma unroll
              for (unsigned j = 0; j < B; ++j)
                if (col[j] != kWsNone && !ws_ready2(g0[j], g1[j], parity)) pend |= 1u << j;
              for (unsigned rounds = 0; __any_sync(0xffffffffu, pend != 0u);) {
                if (P.poll_sleep) __nanosleep(P.poll_sleep);
#pragma unroll
                for (unsigned j = 0; j < B; ++j)
                  if (pend & (1u << j)) {
                    ws_ld_poll2(xw + static_cast<std::size_t>(col[j]) * NC + cp, g0[j], g1[j]);
                    if (ws_ready2(g0[j], g1[j], parity)) pend &= ~(1u << j);
                  }
                if (++rounds > P.spin_limit || ((rounds & 255u) == 255u && ws_aborted(P))) {
                  if (pend && !ws_aborted(P)) ws_fail(P, gw, k, hd.w, 1, slot);
                  break;
                }
              }
            }
            if (firstb) {  // the right-hand side (parked sum) travelled with the first batch of gathers
              firstb = false;
              if (want) {
                rhs_finish(upper, code & kCodeSlotMask, t0, t1, dg, a0, a1, k, hd.w);
              } else if (head && !first) {
                a0 = tag_value(t0);
                a1 = tag_value(t1);
              }
            }
#pragma unroll
            for (unsigned j = 0; j < B; ++j) {
              const unsigned off = CLS <= 2u ? (j >> CLS) * 32u + (j & ((1u << CLS) - 1u)) : CLS == 3u ? j : j * K;
              double         v   = 0.0;  // (beyond the row's slots the stage holds other data: never read)
              if (CLS >= 3u || j < rem) v = static_cast<double>(pv[off]);
              a0 = fma(-v, tag_value(g0[j]), a0);
              a1 = fma(-v, tag_value(g1[j]), a1);
            }
          };
          if (CLS <= 2u) {
            const unsigned  T  = width << CLS, adv = (B >> CLS) * 32u;
            const unsigned *pc = sc + ol;
            const VT *      pv = sv + ol;
            for (unsigned t = 0; t < T; t += B, pc += adv, pv += adv) batch(pc, pv, T - t);
          } else {
            const unsigned step = CLS == 3u ? B : B * K, nb = lpr / step;  // batches per entry index u
            for (unsigned u = 0; u < width; ++u) {
              const unsigned *pc = sc + u * 32u + ol + part;
              const VT *      pv = sv + u * 32u + ol + part;
              for (unsigned b = 0; b < nb; ++b, pc += step, pv += step) batch(pc, pv, B);
            }
          }
          if (CLS == 4u) {  // the lane groups that shared a row add their partial sums
            for (unsigned o = Rg * G; o < 32u; o <<= 1) {
              a0 += __shfl_xor_sync(0xffffffffu, a0, o);
              a1 += __shfl_xor_sync(0xffffffffu, a1, o);
            }
          }
          if (head) {
            const unsigned tag = last ? parity : (parity ^ 1u);  // parked partial sums: the other tag
            if (P.publish_st)
              ws_st_publish2(xw + static_cast<std::size_t>(slot) * NC + cp, tag_set(a0, tag), tag_set(a1, tag));
            else
              ws_atom_publish2(xw + static_cast<std::size_t>(slot) * NC + cp, tag_set(a0, tag), tag_set(a1, tag));
          }
          keep ^= static_cast<unsigned>(__double2hiint(a0));
        }
      };
      if (lpr < B) {
        if (z == 0u)
          run(std::integral_constant<unsigned, 0u>());
        else if (z == 1u)
          run(std::integral_constant<unsigned, 1u>());
        else
          run(std::integral_constant<unsigned, 2u>());
      } else if (K == 1u) {
        run(std::integral_constant<unsigned, 3u>());
      } else {
        run(std::integral_constant<unsigned, 4u>());
      }
    }
    // refill after everything read from the stage was used: the size depends on the digest without being
    // changed by it (two reads of the same header word the compiler can not prove equal)
    const unsigned y2     = *reinterpret_cast<const volatile unsigned *>(sg + 1);
    const unsigned size16 = keep == 0x12345678u ? y2 : hd.y;
    __syncwarp();
    if (lane == 0 && size16) {
      ws_mbar_expect_tx(bar0 + stage * 8u, size16 * 16u);
      ws_tma_g2s(ws_smem_addr(ring + stage * kStageBytes), src, size16 * 16u, bar0 + stage * 8u, policy);
      src += static_cast<std::size_t>(size16) * 16u;
    }
    if (lane == 0 && hd.w > my_front + 3u) {
      my_front = hd.w;
      atomicMax(P.sync, static_cast<int>(hd.w));
    }
  }
}

// ---- plan construction / launch -------------------------------------------------------------
namespace {
struct WsConfig {
  unsigned warps, stages;
};
WsConfig ws_config() {
  WsConfig c;
  // measured at Poisson 128^3 (ms per apply): 16 x 4 1.10, 24 x 2 1.05, 32 x 2 1.24
  c.warps  = static_cast<unsigned>(ws_env("HIFIR_B200_WS_WARPS", 24));
  c.stages = static_cast<unsigned>(ws_env("HIFIR_B200_WS_STAGES", 2));
  const bool ok = (c.warps == 16u && c.stages >= 2u && c.stages <= 4u) || (c.warps == 24u && c.stages == 2u) ||
                  (c.warps == 32u && c.stages == 2u) || (c.warps == 20u && c.stages == 3u) || (c.warps == 28u && c.stages == 2u);
  if (!ok) c.warps = 24u, c.stages = 2u;
  return c;
}
}  // namespace

void build_ws_plan(const HostCsr &S, bool upper, SweepPlan &plan, std::size_t *tally, unsigned nsm,
                   const unsigned *rhs_index, unsigned warps, unsigned stages) {
  WsConfig cfg = ws_config();
  if (warps) cfg.warps = warps, cfg.stages = stages;
  plan.ws        = true;
  plan.stream    = false;
  plan.upper     = upper;
  plan.nr        = 1;
  plan.m         = static_cast<unsigned>(S.orig_rows);
  plan.nblocks   = 0;
  plan.ws_grid   = nsm;
  plan.ws_warps  = cfg.warps;
  plan.ws_stages = cfg.stages;
  plan.ws_window = static_cast<unsigned>(std::max(1, ws_env("HIFIR_B200_WS_WINDOW", 2)));
  if (!S.nrows) return;
  WsHost H;
  // the multi-rhs kernel (explicit configuration) amortizes a segment over all columns: full segments
  // of 8 entries per lane, no spreading of thin level sets over many lanes (fewer reductions / publishes)
  pack_warp_streams(S, H, nsm * cfg.warps, plan.ws_window, plan.f32, rhs_index, warps ? 8u : 0u);
  ws_finalize_ring(H, cfg.stages);
  plan.nblocks    = H.slices;
  plan.slab_bytes = H.stream.size() * 4u;
  plan.st_depth   = H.depth;
  plan.st_padded  = H.padded;
  plan.ws_nslots  = H.nslots;
  plan.ws_nsegs   = static_cast<unsigned>(H.nsegs);
  plan.slot_of    = std::move(H.slot_of);
  plan.ws_wdesc.upload(H.wdesc, tally);
  plan.ws_stream.upload(H.stream, tally);
}

// fused plan of one level: L and U merged factors -> one stream per warp (ws_concat_ldu)
void build_ws_ldu_plan(const HostCsr &SL, const HostCsr &SU, SweepPlan &plan, SweepPlan &L, SweepPlan &U, std::size_t *tally,
                       unsigned nsm) {
  const WsConfig cfg = ws_config();
  const unsigned window = static_cast<unsigned>(std::max(1, ws_env("HIFIR_B200_WS_WINDOW", 2)));
  WsHost HL, HU, H;
  pack_warp_streams(SL, HL, nsm * cfg.warps, window, plan.f32, nullptr, 0u);
  pack_warp_streams(SU, HU, nsm * cfg.warps, window, plan.f32, HL.slot_of.empty() ? nullptr : HL.slot_of.data(), 0u);
  ws_concat_ldu(HL, HU, H);
  ws_finalize_ring(H, cfg.stages);
  plan.ws = true, plan.stream = false, plan.upper = false, plan.fused = true, plan.nr = 1;
  plan.m         = static_cast<unsigned>(SL.orig_rows);
  plan.ws_grid   = nsm, plan.ws_warps = cfg.warps, plan.ws_stages = cfg.stages, plan.ws_window = window;
  plan.nblocks   = H.slices;
  plan.slab_bytes = H.stream.size() * 4u;
  plan.st_depth  = H.depth;
  plan.st_padded = H.padded;
  plan.ws_nslots = H.nslots;
  plan.ws_nsegs  = static_cast<unsigned>(H.nsegs);
  plan.ws_wdesc.upload(H.wdesc, tally);
  plan.ws_stream.upload(H.stream, tally);
  // the unfused descriptions (slot maps, statistics) without their device streams
  L.ws = U.ws = true, L.upper = false, U.upper = true;
  L.m = U.m = plan.m;
  L.slot_of = HL.slot_of, U.slot_of = HU.slot_of;
  L.st_depth = HL.depth, U.st_depth = HU.depth;
  L.st_padded = HL.padded, U.st_padded = HU.padded;
  L.slab_bytes = HL.stream.size() * 4u, U.slab_bytes = HU.stream.size() * 4u;
  L.ws_nslots = HL.nslots, U.ws_nslots = HU.nslots;
  L.nblocks = U.nblocks = 0;  // not launchable on their own
}

void ws_debug_graph(const HostCsr &S, unsigned nsm, std::vector<unsigned> &dep_ptr, std::vector<unsigned> &dep_idx) {
  const WsConfig cfg = ws_config();
  WsHost         H;
  pack_warp_streams(S, H, nsm * cfg.warps, static_cast<unsigned>(std::max(1, ws_env("HIFIR_B200_WS_WINDOW", 2))), false,
                    nullptr, 0u);
  ws_segment_graph(H, dep_ptr, dep_idx);
}

void ws_host_emulate(const HostCsr &S, bool upper, const double *rhs, const double *diag, double *x_by_row,
                     std::size_t stats[4], bool f32, int parity) {
  const WsConfig cfg = ws_config();
  WsHost         H;
  pack_warp_streams(S, H, 148u * cfg.warps, static_cast<unsigned>(std::max(1, ws_env("HIFIR_B200_WS_WINDOW", 2))), f32,
                    nullptr, 0u);
  ws_finalize_ring(H, cfg.stages);
  {
    std::string       why;
    const std::size_t stuck = ws_check_schedule(H, f32, &why);
    if (stuck) throw std::logic_error("warp-stream schedule can not complete: " + std::to_string(stuck) + " segments stuck;" + why);
  }
  std::vector<double> x(H.nslots, 0.0);
  ws_host_emulate_packed(H, upper, f32, rhs, diag, x.data(), parity);
  for (std::size_t r = 0; r < S.orig_rows; ++r) x_by_row[r] = x[H.slot_of[r]];
  stats[0] = H.slices;
  stats[1] = H.padded;
  stats[2] = H.stream.size() * 4u;
  stats[3] = H.depth;
}

// The emulation of a plan as the device holds it: wdesc and the segment stream copied back, every warp's
// segment offsets recovered from the segment headers (a warp's segments are contiguous).  x (and x2 for a
// fused plan): ws_nslots entries.
void ws_emulate_device_plan(const SweepPlan &plan, const double *rhs, const double *diag, double *x, double *x2,
                            unsigned parity) {
  WsHost H;
  H.nwarps = plan.ws_grid * plan.ws_warps;
  H.nslots = plan.ws_nslots;
  H.wdesc.resize(plan.ws_wdesc.n);
  H.stream.resize(plan.ws_stream.n);
  if (H.wdesc.size() != static_cast<std::size_t>(H.nwarps) * 8u) throw std::logic_error("warp-stream plan: descriptor size");
  HIF_CUDA(cudaMemcpy(H.wdesc.data(), plan.ws_wdesc.p, H.wdesc.size() * 4u, cudaMemcpyDeviceToHost));
  HIF_CUDA(cudaMemcpy(H.stream.data(), plan.ws_stream.p, H.stream.size() * 4u, cudaMemcpyDeviceToHost));
  H.seg_off.assign(H.nwarps, {});
  for (unsigned w = 0; w < H.nwarps; ++w) {
    const std::size_t base = static_cast<std::size_t>(H.wdesc[static_cast<std::size_t>(w) * 8u]) * 4u;
    std::size_t       off  = 0;
    for (unsigned k = 0; k < H.wdesc[static_cast<std::size_t>(w) * 8u + 1u]; ++k) {
      if (base + off + kWsHdrWords > H.stream.size()) throw std::logic_error("warp-stream plan: segment beyond the stream");
      const unsigned hx = H.stream[base + off];
      H.seg_off[w].push_back(static_cast<unsigned>(off));
      off += seg_words(hx & 0xffu, ((hx >> 16) & kSegCopy) != 0u, plan.f32);
    }
  }
  ws_host_emulate_packed(H, plan.upper, plan.f32, rhs, diag, x, static_cast<int>(parity), plan.fused ? x2 : nullptr);
}

namespace {
template <int UPPER, class VT, int kWarps, int kStages>
void launch_ws_K(Handle *h, const SweepPlan &plan, const WsParams &P) {
  constexpr unsigned kStageBytes = (kWsHdrWords + 64u + kWsU * 32u * (sizeof(VT) == 4 ? 2u : 3u)) * 4u;
  constexpr unsigned smem        = kWarps * kStages * (8u + kStageBytes);
  const bool         pipe        = ws_env("HIFIR_B200_WS_PIPE", 0) != 0;
  auto               kern        = pipe ? wsweep_kernel<UPPER, VT, kWarps, kStages, false, true> : wsweep_kernel<UPPER, VT, kWarps, kStages, false, false>;
  // per device, once (cudaFuncSetAttribute is per device)
  static bool configured[64][2] = {{false}};
  if (h->device < 64 && !configured[h->device][pipe ? 1 : 0]) {
    HIF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    configured[h->device][pipe ? 1 : 0] = true;
  }
  if (P.trace) {
    if (kWarps != 24 || kStages != 2 || sizeof(VT) != 8) throw std::logic_error("tracing needs the 24 x 2 double configuration");
    auto tk = wsweep_kernel<UPPER, double, 24, 2, true, false>;
    HIF_CUDA(cudaFuncSetAttribute(tk, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    tk<<<plan.ws_grid, kWarps * 32, smem, h->stream>>>(P);
    return;
  }
  kern<<<plan.ws_grid, kWarps * 32, smem, h->stream>>>(P);
}
template <int UPPER, class VT>
void launch_ws_V(Handle *h, const SweepPlan &plan, const WsParams &P) {
  const unsigned w = plan.ws_warps, s = plan.ws_stages;
  if (w == 16 && s == 4)
    launch_ws_K<UPPER, VT, 16, 4>(h, plan, P);
  else if (w == 16 && s == 3)
    launch_ws_K<UPPER, VT, 16, 3>(h, plan, P);
  else if (w == 16 && s == 2)
    launch_ws_K<UPPER, VT, 16, 2>(h, plan, P);
  else if (w == 24 && s == 2)
    launch_ws_K<UPPER, VT, 24, 2>(h, plan, P);
  else if (w == 20 && s == 3)
    launch_ws_K<UPPER, VT, 20, 3>(h, plan, P);
  else if (w == 28 && s == 2)
    launch_ws_K<UPPER, VT, 28, 2>(h, plan, P);
  else if (w == 32 && s == 2)
    launch_ws_K<UPPER, VT, 32, 2>(h, plan, P);
  else
    throw std::logic_error("unsupported warp-stream configuration (warps x stages)");
}
}  // namespace

namespace {
template <class VT, int G>
void launch_ws_cols_G(Handle *h, const SweepPlan &plan, const WsParams &P) {
  constexpr unsigned kStageBytes = (kWsHdrWords + 64u + kWsU * 32u * (sizeof(VT) == 4 ? 2u : 3u)) * 4u;
  constexpr unsigned smem        = 24u * 2u * (8u + kStageBytes);
  static const int   bt          = ws_env("HIFIR_B200_MRHS_BATCH", 4);  // entries of a row in flight per lane
  auto               kern        = bt >= 8 ? wsweep_cols_kernel<VT, G, 8u> : bt >= 4 ? wsweep_cols_kernel<VT, G, 4u> : wsweep_cols_kernel<VT, G, 2u>;
  static bool        configured[64] = {false};
  if (h->device >= 64 || !configured[h->device]) {
    HIF_CUDA(cudaFuncSetAttribute(wsweep_cols_kernel<VT, G, 8u>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    HIF_CUDA(cudaFuncSetAttribute(wsweep_cols_kernel<VT, G, 4u>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    HIF_CUDA(cudaFuncSetAttribute(wsweep_cols_kernel<VT, G, 2u>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    if (h->device < 64) configured[h->device] = true;
  }
  kern<<<plan.ws_grid, 24 * 32, smem, h->stream>>>(P);
}
template <class VT>
void launch_ws_cols_V(Handle *h, const SweepPlan &plan, const WsParams &P, unsigned nc) {
  if (nc == 8u)
    launch_ws_cols_G<VT, 4>(h, plan, P);
  else if (nc == 16u)
    launch_ws_cols_G<VT, 8>(h, plan, P);
  else if (nc == 32u)
    launch_ws_cols_G<VT, 16>(h, plan, P);
  else if (nc == 64u)
    launch_ws_cols_G<VT, 32>(h, plan, P);
  else
    throw std::logic_error("multi-rhs sweep: 8, 16, 32 or 64 columns per pass");
}
}  // namespace

// multi-rhs LDU solve on the fused warp-stream plan of a level: nc in {8, 16, 32, 64} columns, row-interleaved
void launch_ws_sweep_cols(Handle *h, const SweepPlan &plan, const double *rhs_plain, const double *diag, unsigned long long *xL,
                          unsigned long long *xU, unsigned parity, int *sync, unsigned nc) {
  if (!plan.nblocks) return;
  if (!plan.fused || plan.ws_warps != 24u || plan.ws_stages != 2u)
    throw std::logic_error("multi-rhs sweep needs the fused 24 x 2 warp-stream plan");
  WsParams P;
  P.trace      = nullptr;
  P.wdesc      = plan.ws_wdesc.p;
  P.stream     = plan.ws_stream.p;
  P.rhs_plain  = rhs_plain;
  P.rhs_tagged = nullptr;
  P.diag       = diag;
  P.x          = xL;
  P.x2         = xU;
  P.sync       = sync;
  P.error_flag = h->error_flag.p;
  P.parity     = parity;
  P.window     = plan.ws_window;
  P.adm_sleep  = static_cast<unsigned>(std::max(0, ws_env("HIFIR_B200_WS_SLEEP", 200)));
  P.publish_st = ws_env("HIFIR_B200_MRHS_PUBLISH_ATOM", 0) ? 0 : 1;
  P.l1_first   = 0;
  P.spin_limit = static_cast<unsigned>(std::max(1000, ws_env("HIFIR_B200_WS_SPIN_LIMIT", 1 << 21)));
  P.poll_sleep = static_cast<unsigned>(std::max(0, ws_env("HIFIR_B200_MRHS_POLL_SLEEP", 0)));
  // developer experiment (HIFIR_B200_WS_REPEAT): launch the sweep again -- every slot carries the tag already,
  // the second pass never waits: its duration is the pure throughput bound of the kernel on this factor
  static const int repeat = ws_env("HIFIR_B200_WS_REPEAT", 0);
  for (int r = 0; r <= repeat; ++r) {
    if (plan.f32)
      launch_ws_cols_V<float>(h, plan, P, nc);
    else
      launch_ws_cols_V<double>(h, plan, P, nc);
    HIF_KERNEL_CHECK();
  }
  ++h->launch_count;
}

void launch_ws_sweep(Handle *h, const SweepPlan &plan, const double *rhs_plain, const unsigned long long *rhs_tagged,
                     const double *diag, unsigned long long *x, unsigned parity, int *sync, unsigned long long *trace,
                     unsigned long long *x2) {
  if (!plan.nblocks) return;
  WsParams P;
  P.trace      = trace;
  P.x2         = x2;
  P.wdesc      = plan.ws_wdesc.p;
  P.stream     = plan.ws_stream.p;
  P.rhs_plain  = rhs_plain;
  P.rhs_tagged = rhs_tagged;
  P.diag       = diag;
  P.x          = x;
  P.sync       = sync;
  P.error_flag = h->error_flag.p;
  P.parity     = parity;
  P.window     = plan.ws_window;
  P.adm_sleep  = static_cast<unsigned>(std::max(0, ws_env("HIFIR_B200_WS_SLEEP", 200)));
  P.publish_st = ws_env("HIFIR_B200_WS_PUBLISH_ST", 0);
  P.l1_first   = ws_env("HIFIR_B200_WS_L1", 0);
  P.spin_limit = static_cast<unsigned>(std::max(1000, ws_env("HIFIR_B200_WS_SPIN_LIMIT", 1 << 21)));
  P.poll_sleep = static_cast<unsigned>(std::max(0, ws_env("HIFIR_B200_WS_POLL_SLEEP", 0)));
  if (plan.fused) {
    if (!x2) throw std::logic_error("fused L-then-U sweep needs both solution buffers");
    if (plan.f32)
      launch_ws_V<2, float>(h, plan, P);
    else
      launch_ws_V<2, double>(h, plan, P);
  } else if (plan.upper) {
    if (plan.f32)
      launch_ws_V<1, float>(h, plan, P);
    else
      launch_ws_V<1, double>(h, plan, P);
  } else {
    if (plan.f32)
      launch_ws_V<0, float>(h, plan, P);
    else
      launch_ws_V<0, double>(h, plan, P);
  }
  HIF_KERNEL_CHECK();
  ++h->launch_count;
  // developer experiment: launch the sweep again -- every slot already carries the current tag, so the
  // second pass never waits: its duration is the pure throughput bound of the kernel on this factor
  static const int repeat = ws_env("HIFIR_B200_WS_REPEAT", 0);
  for (int r = 0; r < repeat && !plan.fused; ++r) {
    if (plan.upper) {
      if (plan.f32) launch_ws_V<1, float>(h, plan, P); else launch_ws_V<1, double>(h, plan, P);
    } else {
      if (plan.f32) launch_ws_V<0, float>(h, plan, P); else launch_ws_V<0, double>(h, plan, P);
    }
    HIF_KERNEL_CHECK();
  }
}

}  // namespace hifgpu
