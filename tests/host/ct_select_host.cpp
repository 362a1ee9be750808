// Host build of the kernels' constant-time table selection (csrc/dkg_ct_select.cuh) with an
// accessor that records every address it reads.  Test scaffolding only: lets
// `pytest -m "not gpu"` check that the selected value is right and that the sequence of addresses
// read is the same for every digit.
#include <cstddef>
#include <cstdint>
#include "dkg_ct_select.cuh"

namespace {
constexpr int VW = 4;

// table: n entries of nvec vectors of VW words, entry k vector v at table[(k * nvec + v) * VW]
struct RecordingTable {
  const uint32_t* table;
  const uint32_t* onev;
  uint32_t* slot;
  int nvec;
  const uint32_t** trace;   // addresses read, in order
  int* len;
  int cap;
  void record(const uint32_t* a) const {
    if (*len < cap) trace[*len] = a;
    ++*len;
  }
  void one(int v, uint32_t (&r)[VW]) const {
    for (int q = 0; q < VW; ++q) { record(onev + v * VW + q); r[q] = onev[v * VW + q]; }
  }
  void entry(int k, int v, uint32_t (&r)[VW]) const {
    const uint32_t* src = table + ((size_t)k * nvec + v) * VW;
    for (int q = 0; q < VW; ++q) { record(src + q); r[q] = src[q]; }
  }
  void put(int v, const uint32_t (&r)[VW]) const {
    for (int q = 0; q < VW; ++q) slot[v * VW + q] = r[q];
  }
};
}  // namespace

// Selects entry `idx` (or the one for an index outside the table) of an n-entry table into `out`
// (nvec * 4 words).  trace receives the addresses read; returns their number (-1 if over cap).
extern "C" int host_ct_select(const uint32_t* table, const uint32_t* one, int n, int nvec, uint32_t idx,
                              uint32_t* out, const uint32_t** trace, int cap) {
  int len = 0;
  const RecordingTable acc{table, one, out, nvec, trace, &len, cap};
  dkg::ct_select<VW>(acc, n, nvec, idx);
  return len <= cap ? len : -1;
}
