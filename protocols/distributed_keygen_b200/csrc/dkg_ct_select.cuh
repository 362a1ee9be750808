// Constant-time window-table selection (DESIGN.md §2.11), shared by the thread-per-instance
// kernels whose tables are vector-major / lane-minor with one component per entry: the direct
// kernel (dkg_modexp.cuh) and the grouped kernel (dkg_grouped.cuh).
//
// Instead of reading entry `idx` of the window table, read EVERY entry and the Montgomery one in
// one fixed order, keep the wanted value under a mask and write it to a spare slot; the
// multiplication then reads the slot.  The sequence of addresses and the control flow are the
// same for every digit.  The accessor is a template parameter so that the host build
// (tests/host/ct_select_host.cpp) can record every address the selection reads.
#pragma once
#include "dkg_prims.cuh"   // DKG_HD

namespace dkg {

// Accessor interface (VW 32-bit words per vector, vectors 0..nvec-1 of a value):
//   void one(int v, uint32_t (&r)[VW]) const          vector v of the Montgomery one
//   void entry(int k, int v, uint32_t (&r)[VW]) const  vector v of table entry k (0..n-1)
//   void put(int v, const uint32_t (&r)[VW]) const     vector v of the spare slot
// idx < n selects entry idx; any other idx selects the one (the direct kernel's digit-0 marker
// 0xfe, or digit - 1 wrapped around for digit 0).
template <int VW, class Acc>
DKG_HD void ct_select(const Acc& a, int n, int nvec, uint32_t idx) {
  const uint32_t m1 = 0u - (uint32_t)(idx >= (uint32_t)n);
  for (int v = 0; v < nvec; ++v) {
    uint32_t acc[VW], t[VW];
    a.one(v, acc);
#pragma unroll
    for (int q = 0; q < VW; ++q) acc[q] &= m1;
    for (int k = 0; k < n; ++k) {
      const uint32_t mk = 0u - (uint32_t)((uint32_t)k == idx);
      a.entry(k, v, t);
#pragma unroll
      for (int q = 0; q < VW; ++q) acc[q] |= t[q] & mk;
    }
    a.put(v, acc);
  }
}

}  // namespace dkg
