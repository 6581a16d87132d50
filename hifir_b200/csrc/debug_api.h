/* debug_api.h -- developer / test entry points of libhifir_b200.so.
 *
 * NOT part of the drop-in boundary (include/hifir_b200.h): these hooks exist so that the host-side
 * attach-time logic (algebraic level merging, packing into warp streams) can be checked bit for bit
 * by the CPU test suite without a GPU, and so that layout experiments can be scored on the host. */
#ifndef HIFIR_B200_DEBUG_API_H_
#define HIFIR_B200_DEBUG_API_H_

#include "../../include/hifir_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Host only: merges and packs the strictly triangular CCS block T exactly as attach does and solves
 * with the packed data on the CPU, segment by segment in the device's arithmetic order: x = T^{-1} rhs
 * (lower, diag ignored) or x = T^{-1} (rhs ./ diag) (upper).  stats = {slices, padded entries, packed
 * bytes, dependency depth of the packed factor}.  parity < 0: plain values; 0 or 1: every published
 * value (and the right-hand side of an upper sweep) carries the readiness tag of that parity in its
 * last mantissa bit before it is read, as on the device. */
LhfStatus lhfdGpuDebugSweepHost(const LhfdGpuCcs *T, int upper, const double *rhs, const double *diag,
                                double *x, size_t stats[4], int parity);

/* The same for a single-precision factor block: the packed (merged) values are rounded to float
 * exactly as lhfsGpuAttachLevels stores them; rhs / diag / x are double. */
LhfStatus lhfsGpuDebugSweepHost(const LhfsGpuCcs *T, int upper, const double *rhs, const double *diag,
                                double *x, size_t stats[4], int parity);

/* One triangular sweep of an attached handle on the device, checked against the host emulation of the
 * plan the device holds.  transposed != 0: the transposed twin (built on first use).  which: 0 = L,
 * 1 = U, 2 = the fused L-then-U plan (attach fuses unless HIFIR_B200_WS_FUSE=0: then 0 and 1).  The
 * launch is the one the apply issues for that factor, on the handle's stream, into tagged scratch
 * buffers of the hook's own (per level and factor, zeroed at allocation, own epoch counter starting at
 * parity 1): they hold the previous call's values under the other parity, as the apply's buffers do.
 * rhs (m, original row order): b of L / fused, y of U (the sweep then solves U x = y ./ d; y enters
 * tagged, as the L result does in the apply).  The packed plan is copied back from the device and
 * emulated on the host, tag for tag, in an order its dataflow allows.
 * Out: words / emul = the device's tagged result words and the emulation's, slot order (fused plan: the
 * L buffer, then the U buffer), *nwords of them (cap >= 2 m, fused 4 m); slot_of[r] = word of row r of
 * the result (fused plan: slot_of[m + r] = word of row r of the L part, slot_of has 2 m entries);
 * x[r] = the result word of row r as the consumers of the apply read it (the tag bit included); parity. */
LhfStatus lhfdGpuDebugSweepDev(LhfdGpuHdl hdl, int transposed, size_t level, int which, const double *rhs, double *x,
                               unsigned long long *words, unsigned long long *emul, size_t cap, size_t *nwords,
                               unsigned *slot_of, unsigned *parity);

/* lhfdGpuDebugSweepHost on factor (level, upper) of an arena file, with the plan stored in the file
 * when it has one. */
LhfStatus lhfGpuDebugFileSweepHost(const char *path, size_t level, int upper, const double *rhs, double *x,
                                   size_t stats[4]);

/* Host only: the attach-time merge plan of the strictly triangular CCS block T (merge.cu) under the
 * current settings.  out = {rows, entries, depth, merged rows, merged entries, merged depth (dependent
 * steps), super levels, predicted time of one sweep in us under the committed cost model}. */
LhfStatus lhfdGpuDebugMergePlan(const LhfdGpuCcs *T, int upper, double out[8]);

/* Host only: gather-locality statistics of candidate row orders / slot numberings (planlab.cu). */
LhfStatus lhfdGpuDebugPlanLab(const LhfdGpuCcs *T, int upper, const int *key, const double *opts, double *out);

/* One apply with per-segment tracing of one warp-stream sweep (level, which: 0 = down L, 1 = down U,
 * 2 = up L, 3 = up U).  out[4*s + ...] for segment s (numbered warp by warp): 0 decoded at ns
 * (globaltimer); relative to that: 1 admitted, 2 (first-try gathers returned) << 8 | re-poll rounds,
 * 3 (published) << 16 | level (bit 15: copy segment). */
LhfStatus lhfdGpuDebugTraceSweep(LhfdGpuHdl hdl, const double *d_b, double *d_x, int level, int which,
                                 unsigned long long *out, size_t max_segs, size_t *nsegs);

/* Host only: segment dependency graph of the packed warp streams of T, segments numbered as in the
 * trace (warp by warp): segment s gathers results published by dep_idx[dep_ptr[s] .. dep_ptr[s+1]). */
LhfStatus lhfdGpuDebugSegmentGraph(const LhfdGpuCcs *T, int upper, size_t max_segs, size_t max_deps, unsigned *dep_ptr,
                                   unsigned *dep_idx, size_t *nsegs);

/* The device 2-norm of the refinement / Krylov loops (max-scaled, two passes: utils/math.hpp:112-137)
 * of a device vector -- for a direct test incl. inputs whose squares overflow. */
LhfStatus lhfdGpuDebugNorm2Dev(LhfdGpuHdl hdl, const double *d_v, size_t n, double *out);

/* Bit-exact checks of the attach-time integer handling: copies the device-resident index arrays of
 * level `level` back to the host.  which: 0 p, 1 q_inv, 2 E row pointers, 3 E columns (original
 * numbering), 4 F row pointers, 5 F columns, 6 jpvt (level ignored).  out receives min(count, max)
 * 32-bit words; *count = number of words of the array. */
LhfStatus lhfdGpuDebugExportInts(LhfdGpuHdl hdl, size_t level, int which, int *out, size_t max, size_t *count);

#ifdef __cplusplus
}
#endif
#endif
