// Grouped modular exponentiation: every group has its own odd modulus and exponent and
// `per_group` bases -- the biprimality-test batch of the reference's key generation
// (DistributedPaillier.__biprime_test_v_calculation, distributed_keygen.py:1094,1097, looped over
// the surviving candidates by compute_modulus :1313-1329: up to 40 bases g per candidate N,
// exponent (N - p_i - q_i + 1)/4 or (p_i + q_i)/4).
//
// Same thread-per-instance block-Montgomery machinery as the fixed-modulus kernel, but the modulus,
// its block inverse, R mod N, R^2 mod N and the window digits are per lane: a setup kernel derives
// them on the device per group (one thread per group), the main kernel copies each lane's modulus
// into shared memory next to X.  All lanes run the same number of windows (exponents are padded
// with leading zero digits to the longest one in the batch), so the warp never diverges.
#pragma once
#include "dkg_modexp.cuh"
#include "dkg_grouped_params_fwd.h"

namespace dkg {

// One thread per group: Montgomery constants and window digits (CT: extracted without a branch on
// the exponent's bits, for the constant-time instantiation of the grouped kernel).
template <bool CT>
__global__ void __launch_bounds__(64) group_setup_kernel(const GroupedParams p) {
  const unsigned long long g = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= p.groups) return;
  // arithmetic: blocks of K limbs, Lp limbs per number, R = 2^(32 Lp); memory: slots of KP limbs
  const int KP = p.K, K = p.Ka, Lp = K * (p.Lp / KP);
  auto slot = [&](int l) { return (l / K) * KP + l % K; };
  uint32_t n[kGroupedMaxLimbs], x[kGroupedMaxLimbs], d[kGroupedMaxLimbs];
  const uint32_t* src = p.moduli + g * (unsigned long long)p.limbs;
  for (int l = 0; l < Lp; ++l) { n[l] = l < p.limbs ? src[l] : 0u; x[l] = 0; }
  uint32_t* row = p.gconsts + g * (unsigned long long)(3 * p.Lp + KP);
  for (int l = 0; l < 3 * p.Lp + KP; ++l) row[l] = 0;
  for (int l = 0; l < Lp; ++l) row[slot(l)] = n[l];

  // -N^-1 mod 2^(32K) by Hensel lifting one limb at a time (prod = n * inv mod 2^(32K))
  {
    uint32_t inv0 = n[0];
    for (int i = 0; i < 5; ++i) inv0 *= 2u - n[0] * inv0;
    uint32_t inv[32], prod[32];
    for (int i = 0; i < K; ++i) { inv[i] = 0; prod[i] = 0; }
    for (int i = 0; i < K; ++i) {
      const uint32_t target = (i == 0) ? (1u - prod[0]) : (0u - prod[i]);
      const uint32_t dg = target * inv0;
      inv[i] = dg;
      uint64_t carry = 0;
      for (int j = 0; i + j < K; ++j) {
        const uint64_t t = (uint64_t)dg * n[j] + prod[i + j] + carry;
        prod[i + j] = (uint32_t)t;
        carry = t >> 32;
      }
    }
    uint64_t carry = 1;
    for (int i = 0; i < K; ++i) {
      const uint64_t t = (uint64_t)(~inv[i]) + carry;
      row[p.Lp + i] = (uint32_t)t;
      carry = t >> 32;
    }
  }
  // x = 2^k mod n by doubling; ONER at k = 32 Lp, R2 at k = 64 Lp   (n == 1 gives 0)
  x[0] = 1;
  {
    uint32_t hi = 0;
    for (int l = 1; l < Lp; ++l) hi |= n[l];
    if (hi == 0 && n[0] == 1) x[0] = 0;
  }
  for (int k = 0; k < 64 * Lp; ++k) {
    // d = 2x - n ; keep d if it did not borrow (2x >= n), else 2x
    uint32_t carry = 0, borrow = 0;
    for (int l = 0; l < Lp; ++l) {
      const uint32_t two = (x[l] << 1) | carry;
      carry = x[l] >> 31;
      x[l] = two;
      const uint64_t t = (uint64_t)two - n[l] - borrow;
      d[l] = (uint32_t)t;
      borrow = (uint32_t)(t >> 63);
    }
    const bool take = carry != 0 || borrow == 0;
    if (take)
      for (int l = 0; l < Lp; ++l) x[l] = d[l];
    if (k == 32 * Lp - 1)
      for (int l = 0; l < Lp; ++l) row[p.Lp + KP + p.Lp + slot(l)] = x[l];  // ONER
  }
  for (int l = 0; l < Lp; ++l) row[p.Lp + KP + slot(l)] = x[l];  // R2

  // window digits, most significant first, padded with leading zeros to p.ndigits windows
  const uint32_t* e = p.exps + g * (unsigned long long)p.exp_limbs;
  uint8_t* dg = p.digits + g * (unsigned long long)p.ndigits;
  for (int t = 0; t < p.ndigits; ++t) {
    const int lowbit = p.wbits * (p.ndigits - 1 - t);
    if constexpr (CT) {
      // shifts and masks: the only conditions are on bit positions, never on the exponent's bits
      const int wi = lowbit / 32;
      const uint64_t lo = wi < p.exp_limbs ? e[wi] : 0u, hi = wi + 1 < p.exp_limbs ? e[wi + 1] : 0u;
      dg[t] = (uint8_t)(((hi << 32 | lo) >> (lowbit % 32)) & ((1u << p.wbits) - 1u));
    } else {
      unsigned v = 0;
      for (int b = 0; b < p.wbits; ++b) {
        const int bit = lowbit + b;
        if (bit < 32 * p.exp_limbs && ((e[bit / 32] >> (bit % 32)) & 1u)) v |= 1u << b;
      }
      dg[t] = (uint8_t)v;
    }
  }
}

// CT: constant-time table access (DESIGN.md §2.11), its own instantiation chosen by the host
template <int K, int M, bool CT = false>
__global__ void __launch_bounds__(DKG_MAX_THREADS, 1) modexp_grouped_kernel(const GroupedParams p) {
  constexpr int KP = kpad<K>;          // slot of one block in memory (odd K: one zero pad limb)
  using V = typename VecSel<KP>::T;
  constexpr int VW = VecSel<KP>::VW;
  constexpr int Lp = KP * M;           // limbs of a number in memory
  constexpr int LV = Lp / VW;
  constexpr int KV = KP / VW;

  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  // schedule table (sched_total_words_closed(M) words, 16-byte padded), then
  // per warp: X[LV*32] | N[LV*32] | NINV[KV*32] vectors
  static_assert(sched_offset<M>(kSchedModes) == sched_total_words_closed(M), "schedule table size out of sync");
  constexpr int SCHED_BYTES = (sched_total_words_closed(M) * 4 + 15) / 16 * 16;
  fill_schedule<M>(reinterpret_cast<uint32_t*>(smem_raw));
  __syncthreads();
  V* Xw = reinterpret_cast<V*>(smem_raw + SCHED_BYTES) + (size_t)warp * (2 * LV + KV) * 32;
  V* Nw = Xw + LV * 32;
  V* NIw = Nw + LV * 32;
  uint32_t* Xw32 = reinterpret_cast<uint32_t*>(Xw);

  const unsigned gwarp = blockIdx.x * nwarps + warp;
  uint32_t* scratch32 = p.scratch + (size_t)gwarp * p.scratch_per_warp;
  V* tab = reinterpret_cast<V*>(scratch32);
  V* Qg = reinterpret_cast<V*>(scratch32 + p.scratch_q_offset);
  V* R2l = Qg + LV * 32;    // this warp's lanes' R^2 mod N, lane layout
  V* ONEl = R2l + LV * 32;  // and R mod N

  WarpIO<K, M, true, true> io;
  io.sched_s = (uint32_t)__cvta_generic_to_shared(smem_raw);
  io.xs = (uint32_t)__cvta_generic_to_shared(Xw + lane);
  io.ss = io.xs;   // (no second operand here: the prefetch's dummy reads go to X)
  io.ns = (uint32_t)__cvta_generic_to_shared(Nw + lane);
  io.nis = (uint32_t)__cvta_generic_to_shared(NIw + lane);
  io.Qg = Qg + lane; io.Y = nullptr;

  const unsigned long long count = p.groups * (unsigned long long)p.per_group;
  const unsigned long long nwork = (count + 31ull) / 32ull;
  for (;;) {
    unsigned int wg = 0;
    if (lane == 0) wg = atomicAdd(p.counter, 1u);
    wg = __shfl_sync(0xffffffffu, wg, 0);
    if (wg >= nwork) break;
    const unsigned long long first = (unsigned long long)wg * 32ull;
    const int cnt = (int)((count - first) < 32ull ? (count - first) : 32ull);
    const unsigned long long my = first + (unsigned long long)(lane < cnt ? lane : cnt - 1);
    const unsigned long long gid = my / (unsigned long long)p.per_group;

    for (int r = 0; r < 32; ++r) {
      const uint32_t* row = p.bases + (first + (unsigned long long)r) * (unsigned long long)p.limbs;
      for (int l = lane; l < Lp; l += 32) {      // l: limb in slot layout, src: the dense limb (or a pad)
        const int src = (l / KP) * K + (l % KP);
        const bool pad = (l % KP) >= K;
        uint32_t v = pad ? 0u : ((r < cnt) ? (src < p.limbs ? row[src] : 0u) : (l == 0 ? 1u : 0u));
        Xw32[((l / VW) * 32 + r) * VW + (l % VW)] = v;
      }
    }
    // this lane's constants
    {
      const uint32_t* row = p.gconsts + gid * (unsigned long long)(3 * Lp + KP);
      const V* nsrc = reinterpret_cast<const V*>(row);            // rows are 8/16-byte aligned: Lp, K multiples of VW
      for (int v = 0; v < LV; ++v) Nw[v * 32 + lane] = nsrc[v];
      const V* isrc = reinterpret_cast<const V*>(row + Lp);
      for (int v = 0; v < KV; ++v) NIw[v * 32 + lane] = isrc[v];
      const V* r2 = reinterpret_cast<const V*>(row + Lp + KP);
      const V* one = reinterpret_cast<const V*>(row + Lp + KP + Lp);
      for (int v = 0; v < LV; ++v) { R2l[(size_t)v * 32 + lane] = r2[v]; ONEl[(size_t)v * 32 + lane] = one[v]; }
    }
    __syncwarp();

    // canonical reduction of the base is not needed: Montgomery arithmetic works on [0, R)
    io.Y = R2l + lane;
    mont_call<K, M, MONT_MUL, true, true>(io);

    const int tsize = (1 << p.wbits) - 1;
    for (int v = 0; v < LV; ++v) tab[(size_t)v * 32 + lane] = Xw[v * 32 + lane];
    for (int d = 2; d <= tsize; ++d) {
      io.Y = tab + lane;
      mont_call<K, M, MONT_MUL, true, true>(io);
      V* dst = tab + (size_t)(d - 1) * LV * 32 + lane;
      for (int v = 0; v < LV; ++v) dst[(size_t)v * 32] = Xw[v * 32 + lane];
    }
    for (int v = 0; v < LV; ++v) Xw[v * 32 + lane] = ONEl[(size_t)v * 32 + lane];
    const uint8_t* dg = p.digits + gid * (unsigned long long)p.ndigits;
    if constexpr (CT) {
      // constant-time table access: every window's multiplier goes through ct_select into the
      // spare slot after the table, and io.Y stays there; digit 0 (index d - 1 wrapped around)
      // selects the lane's ONEl
      V* slot = tab + (size_t)tsize * LV * 32 + lane;
      io.Y = slot;
      for (int t = 0; t < p.ndigits; ++t) {
        if (t > 0)
          for (int s = 0; s < p.wbits; ++s) mont_call<K, M, MONT_SQR, true, true>(io);
        ct_select_lane<V, VW>(tab + lane, ONEl + lane, slot, tsize, LV, (uint32_t)dg[t] - 1u);
        mont_call<K, M, MONT_MUL, true, true>(io);
      }
    } else {
      for (int t = 0; t < p.ndigits; ++t) {
        if (t > 0)
          for (int s = 0; s < p.wbits; ++s) mont_call<K, M, MONT_SQR, true, true>(io);
        const int d = dg[t];
        io.Y = (d == 0) ? (ONEl + lane) : (tab + (size_t)(d - 1) * LV * 32 + lane);
        mont_call<K, M, MONT_MUL, true, true>(io);
      }
    }
    mont_call<K, M, MONT_REDC, true, true>(io);
    canonicalize<K, M>(io, 1);
    __syncwarp();

    for (int r = 0; r < cnt; ++r) {
      uint32_t* row = p.out + (first + (unsigned long long)r) * (unsigned long long)p.limbs;
      for (int l = lane; l < Lp; l += 32) {
        const int dst = (l / KP) * K + (l % KP);
        if ((l % KP) < K && dst < p.limbs) row[dst] = Xw32[((l / VW) * 32 + r) * VW + (l % VW)];
      }
    }
    __syncwarp();
  }
}

}  // namespace dkg
