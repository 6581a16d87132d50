// sweep.cu -- plan construction and launch dispatch of the triangular sweeps.
//
// Two kernels serve CCS::solve_as_strict_lower / _upper (ds/CompressedStorage.hpp:2267-2279,
// 2356-2369) on the merged factors of merge.cu:
//   ws      (default)  statically scheduled warp streams, wsweep.cu
//   stream             round 1's ticket-scheduled level-major streaming kernel, stream.cu (kept for
//                      A/B measurements and as the multi-rhs kernel until the warp-stream one lands)
#include <cstdlib>
#include <cstring>

#include "hifgpu.h"

namespace hifgpu {

int sweep_kind() {
  const char *e = std::getenv("HIFIR_B200_SWEEP");
  if (e && std::strcmp(e, "stream") == 0) return 1;
  return 2;
}

void build_sweep_plan(const HostCsr &Tnat, bool upper, SweepPlan &plan, std::size_t *tally, unsigned nsm,
                      const unsigned *rhs_index, int kind) {
  plan.m       = static_cast<unsigned>(Tnat.nrows);
  plan.upper   = upper;
  plan.nblocks = 0;
  plan.nr      = 1;
  if (!plan.m) return;
  const MergeParams mp = MergeParams::from_env();
  HostCsr           T  = merged_sweep_form(Tnat, upper, mp, &plan.merge);  // or the stored plan of an arena file
  const MergeStats  ms = plan.merge;
  if ((kind < 0 ? sweep_kind() : kind) == 2)
    build_ws_plan(T, upper, plan, tally, nsm, rhs_index);
  else
    build_stream_plan(T, upper, plan, tally);
  plan.merge = ms;
}


// CPU emulation of a sweep on the packed data -- lets the host-side merging + packing be tested
// without a GPU (tests/test_abi.py)
void sweep_host_emulate(const HostCsr &T, bool upper, const double *rhs, const double *diag, double *x,
                        std::size_t stats[4], bool f32, int parity) {
  const MergeParams mp = MergeParams::from_env();
  MergeStats        ms;
  HostCsr           S = merged_sweep_form(T, upper, mp, &ms);
  const unsigned    m = static_cast<unsigned>(T.nrows);
  if (sweep_kind() == 2) {
    ws_host_emulate(S, upper, rhs, diag, x, stats, f32, parity);
    return;
  }
  std::vector<double> xg(2 * static_cast<std::size_t>(m), 0.0);
  stream_host_emulate(S, upper, rhs, diag, xg.data(), stats, f32, parity);
  std::copy(xg.begin(), xg.begin() + m, x);
}

void launch_sweep(Handle *h, const SweepPlan &plan, const double *rhs_plain, const unsigned long long *rhs_tagged,
                  const double *diag, unsigned long long *x, unsigned parity, int *sync, unsigned nr,
                  unsigned long long *trace) {
  if (!plan.nblocks) return;
  if (plan.ws) {
    if (nr > 1) throw std::logic_error("the warp-stream plan serves one right-hand side");
    launch_ws_sweep(h, plan, rhs_plain, rhs_tagged, diag, x, parity, sync, trace);
    return;
  }
  launch_stream_sweep(h, plan, rhs_plain, rhs_tagged, diag, x, parity, sync, nullptr, nr ? nr : plan.nr);
}

}  // namespace hifgpu
