// Fixed-modulus, fixed-exponent batched modular exponentiation: one big integer per thread,
// one persistent CTA per SM, every warp owns 32 independent instances at a time.
//
// Data layout (see DESIGN.md "Data layout"):
//  * shared memory, per warp: X (running value) and Q (Montgomery quotient blocks), each stored
//    limb-vector-major / lane-minor: vector v (VW = 4 or 2 limbs) of lane l at [(v*32 + l)] so that
//    one LDS.128/LDS.64 of a warp touches 32 consecutive vectors (conflict-free);
//  * shared memory, per CTA: the modulus N, its block inverse -N^-1 mod 2^(32K) (uniform:
//    broadcast loads);
//  * global scratch, per warp: the window table c^1..c^(2^w-1) in Montgomery form, same
//    vector-major / lane-minor layout, so a warp's table reads are 512-byte coalesced;
//  * bases / results in HBM are row-major [count][limbs] as the C ABI hands them over; the warp
//    transposes through shared memory on the way in and out.
#pragma once
#include <cuda_runtime.h>
#include "dkg_mont.cuh"
#include "dkg_ct_select.cuh"
#include "dkg_modexp_params.h"

namespace dkg {

template <int K> struct VecSel { using T = uint2; static constexpr int VW = 2; };
#define DKG_VEC4(K_) template <> struct VecSel<K_> { using T = uint4; static constexpr int VW = 4; };
DKG_VEC4(4) DKG_VEC4(8) DKG_VEC4(12) DKG_VEC4(16) DKG_VEC4(20) DKG_VEC4(24) DKG_VEC4(28) DKG_VEC4(32)
#undef DKG_VEC4

__device__ __forceinline__ void unpack(const uint4& v, uint32_t* r) { r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w; }
__device__ __forceinline__ void unpack(const uint2& v, uint32_t* r) { r[0] = v.x; r[1] = v.y; }
__device__ __forceinline__ void pack(uint4& v, const uint32_t* r) { v = make_uint4(r[0], r[1], r[2], r[3]); }
__device__ __forceinline__ void pack(uint2& v, const uint32_t* r) { v = make_uint2(r[0], r[1]); }

// explicit shared-space accesses (32-bit shared addresses): the IO object crosses a noinline call,
// where the compiler would otherwise lose the address space and emit generic LD/ST
__device__ __forceinline__ void lds_vec(uint4& v, uint32_t saddr) {
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr) : "memory");
}
__device__ __forceinline__ void lds_vec(uint2& v, uint32_t saddr) {
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(saddr) : "memory");
}
__device__ __forceinline__ void sts_vec(uint32_t saddr, const uint4& v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" :: "r"(saddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void sts_vec(uint32_t saddr, const uint2& v) {
  asm volatile("st.shared.v2.u32 [%0], {%1, %2};" :: "r"(saddr), "r"(v.x), "r"(v.y) : "memory");
}
__device__ __forceinline__ void ldg_vec(uint4& v, const uint4* p) {
  asm volatile("ld.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
}
__device__ __forceinline__ void stg_vec(uint4* p, const uint4& v) {
  asm volatile("st.global.v4.u32 [%0], {%1, %2, %3, %4};" :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void stg_vec(uint2* p, const uint2& v) {
  asm volatile("st.global.v2.u32 [%0], {%1, %2};" :: "l"(p), "r"(v.x), "r"(v.y) : "memory");
}
__device__ __forceinline__ void ldg_vec(uint2& v, const uint2* p) {
  asm volatile("ld.global.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
}

// one load through a generic address (shared or global window)
__device__ __forceinline__ void ld_generic(uint4& v, const char* p) {
  asm volatile("ld.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
}
__device__ __forceinline__ void ld_generic(uint2& v, const char* p) {
  asm volatile("ld.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
}

// IO policy of dkg::mont_mul for one thread of a warp.
//  xs      shared-space byte address of this lane's vector 0 of X (consecutive vectors of one
//          lane are 32 vectors apart); ns/nis: the CTA-uniform modulus and block inverse;
//  Qg      this lane's Montgomery-quotient blocks in the warp's global scratch (same
//          vector-major / lane-minor layout; L1/L2 resident, always read through the prefetch);
//  Y       multiplication operand in global memory, this lane's vector 0; like every other
//          lane-private array its vectors are 32 apart (uniform constants are kept lane-replicated
//          by the host for this reason): with ONE compile-time stride the prefetch inside the block
//          product needs no address arithmetic, only immediate offsets -- a run-time stride put
//          64-bit adds between the multiplies and made ptxas shuffle the accumulator through
//          ~40 IMAD.MOV per block product, all on the multiplier pipe.
//  PLN     per-lane modulus: ns/nis then address this lane's copy of N / -N^-1 (32 vectors apart),
//          as in the grouped kernel where every lane may have its own modulus.
//  SCHED   the pair schedule comes from a table in shared memory (sched_s, filled by the kernel
//          with fill_schedule) instead of being recomputed inside the block-product loop.
//  XG      X may live in GLOBAL memory instead of shared (xg != nullptr: this lane's vector 0 there,
//          same vector-major / lane-minor layout; xs is then unused).  The pair kernels of wide keys
//          keep the b component of the running pair there: with only a in shared memory twice as
//          many warps fit an SM.  Decided per call (run time), so a and b products share one instance.
template <class V, bool XG> struct XgField { __device__ __forceinline__ V* xg_get() const { return nullptr; } };
template <class V> struct XgField<V, true> { V* xg = nullptr; __device__ __forceinline__ V* xg_get() const { return xg; } };
template <int K, int M, bool PLN = false, bool SCHED_ = false, bool XG_ = false>
struct WarpIO : XgField<typename VecSel<kpad<K>>::T, XG_> {
  static constexpr bool SCHED = SCHED_;
  uint32_t sched_s = 0;     // shared-space address of the schedule table (SCHED only)
  __device__ __forceinline__ uint32_t sched_begin(int word_offset) const { return sched_s + 4u * (uint32_t)word_offset; }
  __device__ __forceinline__ uint32_t sched_next(uint32_t pos) const { return pos + 4u; }
  __device__ __forceinline__ uint32_t sched_word(uint32_t base, int i) const {
    uint32_t w;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w) : "r"(base + 4u * (uint32_t)i));
    return w;
  }
  // blocks sit in slots of KP = K + (K & 1) limbs (whole vectors; the pad limb of an odd K is zero)
  static constexpr int KP = kpad<K>;
  using V = typename VecSel<KP>::T;
  static constexpr int VW = VecSel<KP>::VW;
  static constexpr int KV = KP / VW;
  static constexpr uint32_t VB = sizeof(V);
  static constexpr uint32_t NSTRIDE = PLN ? 32u * VB : VB;
  uint32_t xs, ns, nis;
  V* Qg;
  const V* Y;
  uint32_t ss = 0;          // second shared-memory operand S (pair arithmetic), lane's vector 0
  const V* Y2 = nullptr;    // second global operand (same layout as Y)
  // (XG only: the member xg of the base class is X's address in global memory, or null)
  __device__ __forceinline__ bool x_global() const { return XG_ && this->xg_get() != nullptr; }

  // never true (a shared-space address is far below 2^32 - 1), but not provably so: guards the
  // pipe-balance ballast in mont_mul
  __device__ __forceinline__ bool never() const { return ns == 0xffffffffu; }
  // does any lane of the warp hold a non-zero v?  (all 32 lanes call the Montgomery product together)
  __device__ __forceinline__ bool any_lane(uint32_t v) const { return __any_sync(0xffffffffu, v != 0u); }
  __device__ __forceinline__ void load_x(int i, uint32_t (&r)[KP]) const {
    if (x_global()) {
#pragma unroll
      for (int q = 0; q < KV; q++) { V v; ldg_vec(v, this->xg_get() + (size_t)(i * KV + q) * 32); unpack(v, &r[q * VW]); }
      return;
    }
#pragma unroll
    for (int q = 0; q < KV; q++) { V v; lds_vec(v, xs + (uint32_t)(i * KV + q) * 32u * VB); unpack(v, &r[q * VW]); }
  }
  __device__ __forceinline__ void load_s(int i, uint32_t (&r)[KP]) const {
#pragma unroll
    for (int q = 0; q < KV; q++) { V v; lds_vec(v, ss + (uint32_t)(i * KV + q) * 32u * VB); unpack(v, &r[q * VW]); }
  }
  // block i of S (from_s) or X: one load sequence for both, the base selected
  __device__ __forceinline__ void load_xs(bool from_s, int i, uint32_t (&r)[KP]) const {
    if (!from_s && x_global()) { load_x(i, r); return; }
    const uint32_t base = from_s ? ss : xs;
#pragma unroll
    for (int q = 0; q < KV; q++) { V v; lds_vec(v, base + (uint32_t)(i * KV + q) * 32u * VB); unpack(v, &r[q * VW]); }
  }
  // top limb (K - 1) of block b of X
  __device__ __forceinline__ uint32_t x_top_limb(int b) const {
    constexpr int tv = (K - 1) / VW, te = (K - 1) % VW;
    if (x_global()) return reinterpret_cast<const uint32_t*>(this->xg_get() + (size_t)(b * KV + tv) * 32)[te];
    uint32_t w;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w) : "r"(xs + (uint32_t)(b * KV + tv) * 32u * VB + (uint32_t)te * 4u));
    return w;
  }
  // block i of 2*S (from_s) or 2*X: every limb shifted left by one, the bit shifted in is the top
  // bit of the limb below (of block i-1 for the first limb)
  __device__ __forceinline__ void load_xs2(bool from_s, int i, uint32_t (&r)[KP]) const {
    const uint32_t base = from_s ? ss : xs;   // (the doubled operand is never the global X: SQR runs on a, MUL2S doubles S)
    uint32_t prev = 0;
    if (i > 0) {
      constexpr int tv = (K - 1) / VW, te = (K - 1) % VW;   // top limb of block i - 1
      asm volatile("ld.shared.u32 %0, [%1];" : "=r"(prev) : "r"(base + (uint32_t)((i - 1) * KV + tv) * 32u * VB + (uint32_t)te * 4u));
    }
#pragma unroll
    for (int q = 0; q < KV; q++) { V v; lds_vec(v, base + (uint32_t)(i * KV + q) * 32u * VB); unpack(v, &r[q * VW]); }
#pragma unroll
    for (int p = K - 1; p > 0; p--) r[p] = __funnelshift_l(r[p - 1], r[p], 1);
    r[0] = __funnelshift_l(prev, r[0], 1);
  }
  __device__ __forceinline__ void load_y(int j, uint32_t (&r)[KP]) const {
#pragma unroll
    for (int q = 0; q < KV; q++) { V v; ldg_vec(v, Y + (size_t)(j * KV + q) * 32); unpack(v, &r[q * VW]); }
  }
  __device__ __forceinline__ void load_q(int i, uint32_t (&r)[KP]) const {
#pragma unroll
    for (int q = 0; q < KV; q++) { V v; ldg_vec(v, Qg + (size_t)(i * KV + q) * 32); unpack(v, &r[q * VW]); }
  }
  // Prefetch descriptor: the next y operand comes either from shared memory (an X block) or from
  // global memory (table entry / quotient block / the global X of the XG layouts).
  // ONE predicated load through a generic address.  With two predicated loads (ld.global / ld.shared,
  // exactly one of them on) into the same registers, ptxas sinks the shared-memory ones to the end of
  // the block product, where each of them -- predicated off or not -- waits on the scoreboard of the
  // global load still in flight to the same register (write after write): the L2 latency of every
  // global y operand was exposed once per block product (5 % of all warp stall samples on that one
  // instruction, profiles/r02_ncu_multi_opcodes.txt).
  // The load is unconditional: a step without a y operand (the quotient step, the end of the product)
  // reads a valid dummy (shared memory, short latency) into registers that are overwritten before
  // their next use -- no predicate to set up and to keep alive through the block product.
  struct Prefetch { const char* base; };
  __device__ __forceinline__ Prefetch prefetch_desc(int kind, int blk) const {
    Prefetch d;
    const bool xkind = kind == PAIR_XX || kind == PAIR_XX2 || kind == PAIR_SX2;   // y = a block of X
    const bool from_shared = xkind && !x_global();
    const bool none = !(xkind || kind == PAIR_XY || kind == PAIR_NQ || kind == PAIR_SY2);
    unsigned long long sgen;
    // (the dummy is block 0 of this lane's own second shared-memory operand -- kernels without one
    // point ss at X: no other thread writes there)
    const uint32_t sbase = none ? ss : xs;
    asm("cvta.shared.u64 %0, %1;" : "=l"(sgen) : "l"((unsigned long long)(sbase + (uint32_t)((none ? 0 : blk) * KV) * 32u * VB)));
    const V* g = kind == PAIR_XY ? Y : (kind == PAIR_SY2 ? Y2 : ((xkind && x_global()) ? this->xg_get() : Qg));
    const char* gb = reinterpret_cast<const char*>(g + (size_t)(blk * KV) * 32);
    d.base = (from_shared || none) ? reinterpret_cast<const char*>(sgen) : gb;
    return d;
  }
  __device__ __forceinline__ void prefetch_load(const Prefetch& d, int v, uint32_t (&r)[KP]) const {
    V val;
    ld_generic(val, d.base + (size_t)v * 32u * VB);
    unpack(val, &r[v * VW]);
  }
  __device__ __forceinline__ void load_n(int j, uint32_t (&r)[KP]) const {
#pragma unroll
    for (int q = 0; q < KV; q++) { V v; lds_vec(v, ns + (uint32_t)(j * KV + q) * NSTRIDE); unpack(v, &r[q * VW]); }
  }
  __device__ __forceinline__ void load_ninv(uint32_t (&r)[KP]) const {
#pragma unroll
    for (int q = 0; q < KV; q++) { V v; lds_vec(v, nis + (uint32_t)q * NSTRIDE); unpack(v, &r[q * VW]); }
  }
  __device__ __forceinline__ void store_q(int i, const uint32_t (&r)[KP]) const {
#pragma unroll
    for (int q = 0; q < KV; q++) { V v; pack(v, &r[q * VW]); stg_vec(Qg + (size_t)(i * KV + q) * 32, v); }
  }
  __device__ __forceinline__ void store_x(int i, const uint32_t (&r)[KP]) const {
    if (x_global()) {
#pragma unroll
      for (int q = 0; q < KV; q++) { V v; pack(v, &r[q * VW]); stg_vec(this->xg_get() + (size_t)(i * KV + q) * 32, v); }
      return;
    }
#pragma unroll
    for (int q = 0; q < KV; q++) { V v; pack(v, &r[q * VW]); sts_vec(xs + (uint32_t)(i * KV + q) * 32u * VB, v); }
  }
};


// limb l of a lane-private big integer stored vector-major in shared memory (base = lane's vector 0)
template <int VW>
__device__ __forceinline__ int sidx(int l) { return (l / VW) * 32 * VW + (l % VW); }

// Binary extended GCD with multi-bit shifts on four lane-private arrays of `Lp` limbs (limb l at
// [l * 32] from the given lane-offset pointers; global scratch or shared memory).  On entry u = a,
// on exit the returned pointer holds a^-1 mod N if *bad == 0.  Invariants: x1*a = u, x2*a = v.
static __device__ __noinline__ uint32_t* mod_inverse_arrays(uint32_t* pu, uint32_t* pv, uint32_t* px1, uint32_t* px2,
                                                     const uint32_t* Ns, uint32_t n0inv, int Lp, uint32_t* bad_out) {
  uint32_t nz = 0;
  for (int l = 0; l < Lp; ++l) {
    pv[l * 32] = Ns[l];
    px1[l * 32] = (l == 0) ? 1u : 0u;
    px2[l * 32] = 0u;
    nz |= pu[l * 32];
  }
  int len = Lp;
  int guard = 64 * Lp + 64;
  while (nz != 0 && guard-- > 0) {
    // 1. make u odd: shift out up to 32 zero bits at a time, dividing x1 by the same power of 2
    uint32_t u0 = pu[0];
    while ((u0 & 1u) == 0) {
      const int tz = u0 ? __ffs(u0) - 1 : 32;
      uint32_t lo = u0;
      for (int l = 0; l < len; ++l) {
        const uint32_t hi = (l + 1 < len) ? pu[(l + 1) * 32] : 0u;
        pu[l * 32] = (uint32_t)((((uint64_t)hi << 32) | lo) >> tz);
        lo = hi;
      }
      const uint32_t mask = tz == 32 ? 0xffffffffu : ((1u << tz) - 1u);
      const uint32_t m = (px1[0] * n0inv) & mask;
      uint64_t carry = 0;
      uint32_t prev = 0;
      for (int l = 0; l < Lp; ++l) {
        const uint64_t t = (uint64_t)px1[l * 32] + (uint64_t)m * Ns[l] + carry;
        const uint32_t cur = (uint32_t)t;
        carry = t >> 32;
        if (l > 0) px1[(l - 1) * 32] = (uint32_t)((((uint64_t)cur << 32) | prev) >> tz);
        prev = cur;
      }
      px1[(Lp - 1) * 32] = (uint32_t)(((carry << 32) | prev) >> tz);
      u0 = pu[0];
    }
    // 2. order: u >= v
    bool lt = false;
    for (int l = len - 1; l >= 0; --l) {
      const uint32_t a = pu[l * 32], b = pv[l * 32];
      if (a != b) { lt = a < b; break; }
    }
    if (lt) {
      uint32_t* t = pu; pu = pv; pv = t;
      t = px1; px1 = px2; px2 = t;
    }
    // 3. u -= v ; x1 = x1 - x2 (mod N)
    uint32_t borrow = 0;
    nz = 0;
    for (int l = 0; l < len; ++l) {
      const uint64_t d = (uint64_t)pu[l * 32] - pv[l * 32] - borrow;
      pu[l * 32] = (uint32_t)d;
      nz |= (uint32_t)d;
      borrow = (uint32_t)(d >> 63);
    }
    bool xlt = false;
    for (int l = Lp - 1; l >= 0; --l) {
      const uint32_t a = px1[l * 32], b = px2[l * 32];
      if (a != b) { xlt = a < b; break; }
    }
    const uint32_t addmask = xlt ? 0xffffffffu : 0u;
    int64_t c = 0;
    for (int l = 0; l < Lp; ++l) {
      const int64_t t = (int64_t)px1[l * 32] - (int64_t)px2[l * 32] + (int64_t)(Ns[l] & addmask) + c;
      px1[l * 32] = (uint32_t)t;
      c = t >> 32;
    }
    while (len > 1 && pu[(len - 1) * 32] == 0 && pv[(len - 1) * 32] == 0) --len;
  }
  // gcd is in v; invertible iff v == 1; the inverse is x2
  uint32_t bad = pv[0] ^ 1u;
  for (int l = 1; l < Lp; ++l) bad |= pv[l * 32];
  *bad_out = bad ? 1u : 0u;
  return px2;
}

// Modular inverse of the lane's value in X (shared memory, vector-major layout), work arrays in
// `g` (4 * Lp * 32 words of global scratch or shared memory, lane offset applied).
// Returns 0 if invertible (X <- a^-1 mod N), 1 otherwise (X unspecified).
template <int K, int M>
__device__ uint32_t mod_inverse_lane(uint32_t* X, const uint32_t* Ns, uint32_t n0inv, uint32_t* g) {
  constexpr int VW = VecSel<K>::VW;
  constexpr int Lp = K * M;
  for (int l = 0; l < Lp; ++l) g[l * 32] = X[sidx<VW>(l)];
  uint32_t bad = 0;
  const uint32_t* r = mod_inverse_arrays(g, g + Lp * 32, g + 2 * Lp * 32, g + 3 * Lp * 32, Ns, n0inv, Lp, &bad);
  for (int l = 0; l < Lp; ++l) X[sidx<VW>(l)] = r[l * 32];
  return bad;
}

// One out-of-line instance of the Montgomery product per shape, shared by every mode (square,
// multiply, reduce, doubled product, multiply-add): the hot loop stays inside the instruction cache.
template <int K, int M, bool PLN, bool SCHED, bool XG>
__device__ __noinline__ void mont_call_rt(const WarpIO<K, M, PLN, SCHED, XG> io, const int mode) {
  mont_mul<K, M>(io, mode);
}
template <int K, int M, int MODE, bool PLN = false, bool SCHED = false, bool XG = false>
__device__ __forceinline__ void mont_call(const WarpIO<K, M, PLN, SCHED, XG>& io) {
  mont_call_rt<K, M, PLN, SCHED, XG>(io, MODE);
}
// all threads of the CTA fill the schedule table (sched_offset<M>(kSchedModes) words at `tab`)
template <int M>
__device__ __forceinline__ void fill_schedule(uint32_t* tab) {
  const int n = sched_offset<M>(kSchedModes);
  for (int i = threadIdx.x; i < n; i += blockDim.x) tab[i] = sched_entry<M>(i);
}

// ct_select accessor for one lane of a warp's window table (vector-major / lane-minor, global
// memory; every pointer already offset by the lane): entry k, vector v at tab[(k * nvec + v) * 32]
template <class V, int VW>
struct LaneTable {
  const V* tab;
  const V* onev;   // the Montgomery one, same vector stride
  V* slot;         // the spare slot the selection goes to
  int nvec;
  __device__ __forceinline__ void one(int v, uint32_t (&r)[VW]) const { unpack(onev[(size_t)v * 32], r); }
  __device__ __forceinline__ void entry(int k, int v, uint32_t (&r)[VW]) const { unpack(tab[((size_t)k * nvec + v) * 32], r); }
  __device__ __forceinline__ void put(int v, const uint32_t (&r)[VW]) const { V x; pack(x, r); slot[(size_t)v * 32] = x; }
};
// Out of line: inlined, the scan's loads and masks raise the register demand of the whole kernel
// (and the spills of the widest shapes) at a point where most of its state is live.
template <class V, int VW>
__device__ __noinline__ void ct_select_lane(const V* tab, const V* onev, V* slot, int n, int nvec, uint32_t idx) {
  ct_select<VW>(LaneTable<V, VW>{tab, onev, slot, nvec}, n, nvec, idx);
}

// CT: constant-time table access (DESIGN.md §2.11), its own instantiation chosen by the host, so
// that the default one is not touched by it
template <int K, int M, bool CT = false>
__global__ void __launch_bounds__(DKG_MAX_THREADS, 1) modexp_fixed_kernel(const ModexpParams p) {
  using V = typename VecSel<K>::T;
  constexpr int VW = VecSel<K>::VW;
  constexpr int Lp = K * M;
  constexpr int LV = Lp / VW;  // vectors per big integer

  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint32_t* Ns32 = reinterpret_cast<uint32_t*>(smem_raw);  // N[Lp] then NINV[K]
  constexpr int UNI = ((Lp + K) * 4 + 15) / 16 * 16;       // bytes of the uniform area
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;

  for (int i = threadIdx.x; i < Lp + K; i += blockDim.x) Ns32[i] = p.consts[i];
  __syncthreads();

  V* Xw = reinterpret_cast<V*>(smem_raw + UNI) + (size_t)warp * LV * 32;
  uint32_t* Xw32 = reinterpret_cast<uint32_t*>(Xw);
  const V* Ns = reinterpret_cast<const V*>(Ns32);
  const V* NIs = reinterpret_cast<const V*>(Ns32 + Lp);
  const V* ONEg = reinterpret_cast<const V*>(p.consts + Lp + K + Lp);
  // lane-replicated copies of R^2 and R mod N ([v][lane], after the uniform constants)
  const V* R2rep = reinterpret_cast<const V*>(p.consts + Lp + K + 3 * Lp) + lane;
  const V* ONErep = R2rep + (size_t)LV * 32;

  const unsigned gwarp = blockIdx.x * nwarps + warp;
  uint32_t* scratch32 = p.scratch + (size_t)gwarp * p.scratch_per_warp;
  V* tab = reinterpret_cast<V*>(scratch32);  // entry d (1-based) at tab[((d-1)*LV + v)*32 + lane]
  V* Qg = reinterpret_cast<V*>(scratch32 + p.scratch_q_offset);  // quotient blocks, [v*32 + lane]

  WarpIO<K, M> io;
  io.xs = (uint32_t)__cvta_generic_to_shared(Xw + lane);
  io.ss = io.xs;   // (no second operand here: the prefetch's dummy reads go to X)
  io.ns = (uint32_t)__cvta_generic_to_shared(Ns);
  io.nis = (uint32_t)__cvta_generic_to_shared(NIs);
  io.Qg = Qg + lane; io.Y = nullptr;

  const unsigned long long ngroups = (p.run_if != nullptr && *p.run_if == 0u) ? 0ull : (p.count + 31ull) / 32ull;
  for (;;) {
    unsigned int g = 0;
    if (lane == 0) g = atomicAdd(p.counter, 1u);
    g = __shfl_sync(0xffffffffu, g, 0);
    if (g >= ngroups) break;
    const unsigned long long first = (unsigned long long)g * 32ull;
    const int cnt = (int)((p.count - first) < 32ull ? (p.count - first) : 32ull);

    // ---- load 32 rows, transposed into X (zero padded; idle lanes get the value 1) ----------
    for (int r = 0; r < 32; ++r) {
      const uint32_t* row = p.bases + (first + (unsigned long long)r) * (unsigned long long)p.in_limbs;
      for (int l = lane; l < Lp; l += 32) {
        uint32_t v = (r < cnt) ? (l < p.in_limbs ? row[l] : 0u) : (l == 0 ? 1u : 0u);
        Xw32[((l / VW) * 32 + r) * VW + (l % VW)] = v;
      }
    }
    __syncwarp();

    uint32_t st = 0;
    bool in_mont_form = false;
    if (p.negative) {
      // the batched inversion (dkg_batchinv.cuh) has left c^-1 * R for this group unless its
      // chain hit a non-invertible element; then every lane of the group inverts on its own
      uint32_t chain_bad = 1;
      if (p.inv_mont != nullptr) chain_bad = p.chain_status[(size_t)(g % p.nchain_warps) * 32 + lane];
      if (__any_sync(0xffffffffu, chain_bad != 0)) {
        st = mod_inverse_lane<K, M>(Xw32 + lane * VW, Ns32, p.n0inv, scratch32 + lane);
        __syncwarp();
      } else {
        const V* src = reinterpret_cast<const V*>(p.inv_mont + (size_t)g * Lp * 32) + lane;
        for (int v = 0; v < LV; ++v) Xw[v * 32 + lane] = src[(size_t)v * 32];
        in_mont_form = true;
      }
    }

    // ---- to Montgomery form: X <- X * R^2 / R ------------------------------------------------
    if (!in_mont_form) {
      io.Y = R2rep;
      mont_call<K, M, MONT_MUL>(io);
    }

    if (p.nops == 0) {
      for (int v = 0; v < LV; ++v) Xw[v * 32 + lane] = ONEg[v];
    } else {
      // ---- window table: tab[k] = c^(k+1), or the odd powers c^(2k+1) with c^2 in the slot after
      const int tn = p.tab_entries;
      for (int v = 0; v < LV; ++v) tab[(size_t)v * 32 + lane] = Xw[v * 32 + lane];
      if (tn > 1) {
        const V* step = tab + lane;   // multiply by c ...
        if (p.table_odd) {            // ... or by c^2
          V* c2 = tab + (size_t)tn * LV * 32 + lane;
          mont_call<K, M, MONT_SQR>(io);
          for (int v = 0; v < LV; ++v) { c2[(size_t)v * 32] = Xw[v * 32 + lane]; Xw[v * 32 + lane] = tab[(size_t)v * 32 + lane]; }
          step = c2;
        }
        io.Y = step;
        for (int k = 1; k < tn; ++k) {
          mont_call<K, M, MONT_MUL>(io);
          V* dst = tab + (size_t)k * LV * 32 + lane;
          for (int v = 0; v < LV; ++v) dst[(size_t)v * 32] = Xw[v * 32 + lane];
        }
      }
      // ---- left to right through the operation list (one list for the whole batch) -------------
      if constexpr (CT) {
        // constant-time table access (fixed windows only): the first value and every multiplier
        // come from ct_select into the spare slot after the table, so no address depends on a
        // digit (dkg_ct_select.cuh); io.Y stays on the slot
        V* slot = tab + (size_t)tn * LV * 32 + lane;
        ct_select_lane<V, VW>(tab + lane, ONErep, slot, tn, LV, p.ops[0] & 0xffu);
        for (int v = 0; v < LV; ++v) Xw[v * 32 + lane] = slot[(size_t)v * 32];
        io.Y = slot;
        for (int t = 1; t < p.nops; ++t) {
          const uint32_t op = p.ops[t];
          for (uint32_t s = op >> 8; s > 0; --s) mont_call<K, M, MONT_SQR>(io);
          ct_select_lane<V, VW>(tab + lane, ONErep, slot, tn, LV, op & 0xffu);
          mont_call<K, M, MONT_MUL>(io);
        }
      } else {
        {
          const V* src = tab + (size_t)(p.ops[0] & 0xffu) * LV * 32 + lane;
          for (int v = 0; v < LV; ++v) Xw[v * 32 + lane] = src[(size_t)v * 32];
        }
        for (int t = 1; t < p.nops; ++t) {
          const uint32_t op = p.ops[t];
          for (uint32_t s = op >> 8; s > 0; --s) mont_call<K, M, MONT_SQR>(io);
          const uint32_t idx = op & 0xffu;
          if (idx != 0xffu) {
            io.Y = idx == 0xfeu ? ONErep : tab + (size_t)idx * LV * 32 + lane;
            mont_call<K, M, MONT_MUL>(io);
          }
        }
      }
    }

    // ---- optional final plain multiplier (encryption epilogue), else leave Montgomery form ---
    if (p.final_mul != nullptr) {
      // stage the multipliers through the table area (entry 1) in lane layout
      __syncwarp();
      uint32_t* stage = scratch32;
      for (int r = 0; r < 32; ++r) {
        const uint32_t* row = p.final_mul + (first + (unsigned long long)r) * (unsigned long long)p.in_limbs;
        for (int l = lane; l < Lp; l += 32) {
          uint32_t v = (r < cnt && l < p.in_limbs) ? row[l] : 0u;
          stage[((l / VW) * 32 + r) * VW + (l % VW)] = v;
        }
      }
      __syncwarp();
      io.Y = tab + lane;
      mont_call<K, M, MONT_MUL>(io);   // (x R) * y / R = x y
    } else {
      mont_call<K, M, MONT_REDC>(io);
    }
    canonicalize<K, M>(io, p.final_mul != nullptr ? 2 : 1);
    __syncwarp();

    // ---- store rows ---------------------------------------------------------------------------
    for (int r = 0; r < cnt; ++r) {
      const uint32_t st_r = __shfl_sync(0xffffffffu, st, r);
      uint32_t* row = p.out + (first + (unsigned long long)r) * (unsigned long long)p.in_limbs;
      for (int l = lane; l < p.in_limbs; l += 32) {
        const uint32_t v = Xw32[((l / VW) * 32 + r) * VW + (l % VW)];
        row[l] = st_r ? 0u : v;
      }
    }
    if (p.status != nullptr && lane < cnt) p.status[first + lane] = (uint8_t)st;
    __syncwarp();
  }
}

}  // namespace dkg
