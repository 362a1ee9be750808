// Cooperative (warp-per-operand) modular exponentiation: the latency path for small batches.
//
// The throughput kernels (dkg_modexp.cuh, dkg_nsq.cuh, dkg_grouped.cuh) hold one big integer per
// THREAD, so one wave of 56 832 instances is also the latency of a single instance (0.74 s at
// 2048-bit N).  The reference decrypts ONE ciphertext per call in _decrypt_raw
// (distributed_keygen.py:314-382), ten in its own tests (test_distributed_keygen.py:161-185), and a
// compute_modulus round has a handful of surviving candidates (:1288-1329): for those sizes one
// integer is spread over the 32 lanes of a WARP here.
//
//  * A number of nb blocks of K limbs (K = 6 or 12, nb <= 16) lives with block p on lane p.
//  * Product: lane d forms the block anti-diagonal sum E_d = sum_{i+j=d} X_i * Y_j with the same
//    register-resident K x K block product as the throughput kernels (ColAcc / block_mac, all
//    IMAD.WIDE carry chains), operands read from shared memory.  The 2nb-1 diagonals have 1..nb
//    tiles; the spare lanes take a second..fourth chunk of the long ones (host-built plan,
//    tests/coop_model.py: make_plan) and hand their partial sums over with __shfl_sync.
//  * Carry resolution: E_d overlaps E_{d-1}, E_{d-2}; lane d fetches the overlapping limbs with
//    __shfl_up_sync, adds, passes its small carry up once and settles the remaining 0/1 ripple
//    with two __ballot_sync masks (generate / propagate) and one integer addition.
//  * Montgomery product in three such phases: T = X*Y, q = (T mod R) * (-N^-1) mod R (low
//    diagonals only), (T + q*N) / R.  R = 2^(32 K nb) >= 4N (>= 8N for the pair arithmetic), so no
//    conditional subtraction is needed between products.
//  * On top: the pair arithmetic modulo N^2 of dkg_nsq.cuh (same formulas, same bounds), with
//    negative exponents handled per instance by the almost-inverse (Kaliski) modulo N on lane
//    registers plus one Newton step in the pair domain -- no chains, exact per-element status;
//    and a grouped kernel (per-instance modulus and exponent, biprimality test) that derives
//    -N^-1 mod R, R mod N and R^2 mod N itself.
// Python model of every lane-level step: tests/coop_model.py.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "dkg_coop_params.h"
#include "dkg_mont.cuh"

namespace dkg {

namespace coop {

using sa = uint32_t;   // shared-space byte address (numbers live in shared memory; the arithmetic
                       // below crosses noinline calls, where generic pointers would lose LDS/STS)
__device__ __forceinline__ sa saddr(const void* p) { return (sa)__cvta_generic_to_shared(p); }

template <int K>
struct NoIO {
  static constexpr int VW = 2;
  struct Prefetch {};
  __device__ __forceinline__ void prefetch_load(const Prefetch&, int, uint32_t (&)[K]) const {}
};

template <int K>
__device__ __forceinline__ void lds(uint32_t (&r)[K], sa p) {
  if constexpr (K % 4 == 0) {
#pragma unroll
    for (int v = 0; v < K / 4; ++v)
      asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                   : "=r"(r[4 * v]), "=r"(r[4 * v + 1]), "=r"(r[4 * v + 2]), "=r"(r[4 * v + 3]) : "r"(p + 16u * v) : "memory");
  } else {
#pragma unroll
    for (int v = 0; v < K / 2; ++v)
      asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(r[2 * v]), "=r"(r[2 * v + 1]) : "r"(p + 8u * v) : "memory");
  }
}
template <int K>
__device__ __forceinline__ void sts(sa p, const uint32_t (&r)[K]) {
#pragma unroll
  for (int v = 0; v < K / 2; ++v)
    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" :: "r"(p + 8u * v), "r"(r[2 * v]), "r"(r[2 * v + 1]) : "memory");
}
__device__ __forceinline__ uint32_t lds1(sa p) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(p) : "memory");
  return v;
}

// this lane's entry of a plan table
struct LanePlan {
  int d, i0, i1, p0, p1, p2, rounds, ndiag;
  __device__ __forceinline__ void load(const CoopPlanTable& t, int lane) {
    d = t.d[lane]; i0 = t.i0[lane]; i1 = t.i1[lane];
    p0 = t.partner[0][lane]; p1 = t.partner[1][lane]; p2 = t.partner[2][lane];
    rounds = t.rounds; ndiag = t.ndiag;
  }
};

// E_d on the primary lanes (2K+2 limbs), zero elsewhere, for NS independent products at once.  X, Y
// (and the optional second pair of a stream, X2 != 0) are nb-block numbers in shared memory.  The
// streams share the lane plan; their block products and carry chains are independent, so ptxas
// interleaves them and one warp hides its own latencies (a single chain issues one dependent
// instruction every ~4.6 cycles).
template <int K, int NS>
__device__ __forceinline__ void product(uint32_t (&e)[NS][2 * K + 2], const LanePlan& lp, int lane, const sa (&X)[NS],
                                        const sa (&Y)[NS], const sa (&X2)[NS], const sa (&Y2)[NS]) {
  ColAcc<K> a[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) {
#pragma unroll
    for (int p = 0; p < 2 * K + 2; ++p) e[s][p] = 0;
    acc_load<K>(a[s], e[s]);
    acc_clear_side<K>(a[s]);
  }
  const NoIO<K> io;
  const typename NoIO<K>::Prefetch pf;
  for (int i = lp.i0; i < lp.i1; ++i) {
    uint32_t xb[NS][K], yb[NS][K];
    const uint32_t ox = (uint32_t)(i * K * 4), oy = (uint32_t)((lp.d - i) * K * 4);
#pragma unroll
    for (int s = 0; s < NS; ++s) { lds<K>(xb[s], X[s] + ox); lds<K>(yb[s], Y[s] + oy); }
#pragma unroll
    for (int s = 0; s < NS; ++s) block_mac<K>(a[s], xb[s], yb[s], io, pf);
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      if (X2[s] != 0) {
        lds<K>(xb[s], X2[s] + ox);
        lds<K>(yb[s], Y2[s] + oy);
        block_mac<K>(a[s], xb[s], yb[s], io, pf);
      }
    }
  }
  __syncwarp();
#pragma unroll
  for (int s = 0; s < NS; ++s) acc_merge<K>(a[s], e[s]);
  for (int r = 0; r < lp.rounds; ++r) {
    const int src = r == 0 ? lp.p0 : (r == 1 ? lp.p1 : lp.p2);
    const int from = src >= 0 ? src : lane;
    const uint32_t m = src >= 0 ? 0xffffffffu : 0u;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      uint32_t t[2 * K + 2];
#pragma unroll
      for (int k = 0; k < 2 * K + 2; ++k) t[k] = __shfl_sync(kCoopFull, e[s][k], from) & m;
      add_cc(e[s][0], t[0]);
#pragma unroll
      for (int k = 1; k < 2 * K + 1; ++k) addc_cc(e[s][k], t[k]);
      addc(e[s][2 * K + 1], t[2 * K + 1]);
    }
  }
  if (lane >= lp.ndiag) {
#pragma unroll
    for (int s = 0; s < NS; ++s) {
#pragma unroll
      for (int k = 0; k < 2 * K + 2; ++k) e[s][k] = 0;
    }
  }
}
template <int K>
__device__ __forceinline__ void product(uint32_t (&e)[2 * K + 2], const LanePlan& lp, int lane, sa X, sa Y, sa X2, sa Y2) {
  uint32_t ee[1][2 * K + 2];
  const sa x[1] = {X}, y[1] = {Y}, x2[1] = {X2}, y2[1] = {Y2};
  product<K, 1>(ee, lp, lane, x, y, x2, y2);
#pragma unroll
  for (int k = 0; k < 2 * K + 2; ++k) e[k] = ee[0][k];
}

// carry into every lane from generate / propagate masks; bit 32+ = carry out of lane 31
__device__ __forceinline__ uint64_t lookahead(uint32_t g, uint32_t p) {
  const uint64_t a = (uint64_t)(g | p), b = (uint64_t)g;
  return (a + b) ^ a ^ b;
}

// s (block `lane` of sum_d E_d W^d [+ addend]) from the diagonal sums: overlap limbs by shuffle,
// one explicit carry hop, then generate/propagate lookahead.
template <int K>
__device__ __forceinline__ void resolve(uint32_t (&s)[K], const uint32_t (&e)[2 * K + 2], const uint32_t* addend, int lane) {
  uint32_t mid[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    mid[k] = __shfl_up_sync(kCoopFull, e[K + k], 1);
    if (lane < 1) mid[k] = 0;
  }
  uint32_t h0 = __shfl_up_sync(kCoopFull, e[2 * K], 2), h1 = __shfl_up_sync(kCoopFull, e[2 * K + 1], 2);
  if (lane < 2) { h0 = 0; h1 = 0; }
  uint32_t c = 0;
#pragma unroll
  for (int k = 0; k < K; ++k) s[k] = e[k];
  add_cc(s[0], mid[0]);
#pragma unroll
  for (int k = 1; k < K; ++k) addc_cc(s[k], mid[k]);
  addc(c, 0);
  add_cc(s[0], h0);
  addc_cc(s[1], h1);
#pragma unroll
  for (int k = 2; k < K; ++k) addc_cc(s[k], 0);
  addc(c, 0);
  if (addend != nullptr) {
    add_cc(s[0], addend[0]);
#pragma unroll
    for (int k = 1; k < K; ++k) addc_cc(s[k], addend[k]);
    addc(c, 0);
  }
  uint32_t cin = __shfl_up_sync(kCoopFull, c, 1);
  if (lane < 1) cin = 0;
  uint32_t g = 0, ones = 0xffffffffu;
  add_cc(s[0], cin);
#pragma unroll
  for (int k = 1; k < K; ++k) addc_cc(s[k], 0);
  addc(g, 0);
#pragma unroll
  for (int k = 0; k < K; ++k) ones &= s[k];
  const uint32_t G = __ballot_sync(kCoopFull, g != 0);
  const uint32_t P = __ballot_sync(kCoopFull, ones == 0xffffffffu && g == 0);
  const uint32_t carry = (uint32_t)((lookahead(G, P) >> lane) & 1u);
  add_cc(s[0], carry);
#pragma unroll
  for (int k = 1; k < K - 1; ++k) addc_cc(s[k], 0);
  addc(s[K - 1], 0);
}

// s = x + y + (cin0 at lane 0) over the lanes; x, y must be zero on lanes >= nb.  Returns the carry
// out of block nb-1.
template <int K>
__device__ __forceinline__ uint32_t add(uint32_t (&s)[K], const uint32_t (&x)[K], const uint32_t (&y)[K], uint32_t cin0,
                                        int lane, int nb) {
  uint32_t carry = lane == 0 ? cin0 : 0u, ones = 0xffffffffu;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const uint64_t t = (uint64_t)x[k] + y[k] + carry;
    s[k] = (uint32_t)t;
    carry = (uint32_t)(t >> 32);
    ones &= s[k];
  }
  const uint32_t g = carry;
  const uint32_t G = __ballot_sync(kCoopFull, g != 0);
  const uint32_t P = __ballot_sync(kCoopFull, ones == 0xffffffffu && g == 0 && lane < nb);
  const uint64_t la = lookahead(G, P);
  carry = (uint32_t)((la >> lane) & 1u);
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const uint64_t t = (uint64_t)s[k] + carry;
    s[k] = (uint32_t)t;
    carry = (uint32_t)(t >> 32);
  }
  if (lane >= nb) {
#pragma unroll
    for (int k = 0; k < K; ++k) s[k] = 0;
  }
  return (uint32_t)((la >> nb) & 1u);
}

// s = x - y over the lanes (mod W^nb); returns 1 if x >= y (no borrow), else 0
template <int K>
__device__ __forceinline__ uint32_t sub(uint32_t (&s)[K], const uint32_t (&x)[K], const uint32_t (&y)[K], int lane, int nb) {
  uint32_t yc[K];
#pragma unroll
  for (int k = 0; k < K; ++k) yc[k] = lane < nb ? ~y[k] : 0u;
  return add<K>(s, x, yc, 1u, lane, nb);
}

// x > y over the lanes
template <int K>
__device__ __forceinline__ bool greater(const uint32_t (&x)[K], const uint32_t (&y)[K]) {
  int gt = 0, lt = 0;
#pragma unroll
  for (int k = K - 1; k >= 0; --k) {
    if (!gt && !lt) { gt = x[k] > y[k]; lt = x[k] < y[k]; }
  }
  return __ballot_sync(kCoopFull, gt) > __ballot_sync(kCoopFull, lt);
}
template <int K>
__device__ __forceinline__ bool is_zero(const uint32_t (&x)[K]) {
  uint32_t nz = 0;
#pragma unroll
  for (int k = 0; k < K; ++k) nz |= x[k];
  return __ballot_sync(kCoopFull, nz != 0) == 0u;
}
template <int K>
__device__ __forceinline__ void shr1(uint32_t (&x)[K], int lane) {
  uint32_t in = __shfl_down_sync(kCoopFull, x[0], 1);
  if (lane == 31) in = 0;
#pragma unroll
  for (int k = 0; k < K; ++k) x[k] = (x[k] >> 1) | ((k + 1 < K ? x[k + 1] : in) << 31);
}
template <int K>
__device__ __forceinline__ void shl1(uint32_t (&x)[K], int lane) {
  uint32_t in = __shfl_up_sync(kCoopFull, x[K - 1], 1);
  if (lane == 0) in = 0;
#pragma unroll
  for (int k = K - 1; k >= 0; --k) x[k] = (x[k] << 1) | ((k > 0 ? x[k - 1] : in) >> 31);
}

// x <- 2x mod n for x < n (one conditional subtraction)
template <int K>
__device__ __forceinline__ void double_mod(uint32_t (&x)[K], const uint32_t (&n)[K], int lane, int nb) {
  uint32_t t[K];
  shl1<K>(x, lane);
  if (sub<K>(t, x, n, lane, nb)) {
#pragma unroll
    for (int k = 0; k < K; ++k) x[k] = t[k];
  }
}

// Per-warp working set (passed BY VALUE across the noinline calls: it stays in registers).  All
// numbers are nb*K limbs in shared memory.
template <int K>
struct Warp {
  int lane, nb;
  LanePlan pf, pl;
  sa N;    // modulus
  sa NI;   // -N^-1 mod R
  sa T;    // scratch: T (low half of the product being reduced) | Q (quotient), 2*nb*K words per stream

  __device__ __forceinline__ sa Q() const { return T + (uint32_t)(nb * K * 4); }
  // quotient of the second stream of montmul2 (its T | Q area follows the first one)
  __device__ __forceinline__ sa Q2() const { return T + (uint32_t)(3 * nb * K * 4); }
  __device__ __forceinline__ void load_block(uint32_t (&r)[K], sa num) const {
    if (lane < nb) lds<K>(r, num + (uint32_t)(lane * K * 4));
    else {
#pragma unroll
      for (int k = 0; k < K; ++k) r[k] = 0;
    }
  }
  __device__ __forceinline__ void store_block(sa num, const uint32_t (&r)[K]) const {
    if (lane < nb) sts<K>(num + (uint32_t)(lane * K * 4), r);
  }
  // low nb blocks of X*Y -> out (registers, block `lane`); lanes >= nb hold garbage
  __device__ __forceinline__ void mul_low(uint32_t (&out)[K], sa X, sa Y) const {
    uint32_t e[2 * K + 2];
    product<K>(e, pl, lane, X, Y, 0, 0);
    resolve<K>(out, e, nullptr, lane);
  }
};

// One stream of a Montgomery product: out <- (X1*Y1 [+ X2*Y2]) / R mod N, or, with X1 == 0, the
// Montgomery reduction of the 2nb-block number already lying in the stream's T | Q area.  out may
// alias any operand of any stream (everything is read before anything is written).  The quotient q
// ((T + q N) / R exactly) is left in T + nb*K words.
struct Stream {
  sa out, X1, Y1, X2, Y2, T;
};

// NS independent Montgomery products modulo the same N in one instruction stream (NS = 2: the two
// products of a pair operation).  ONE instance of the three product phases per NS and kernel.
template <int K, int NS>
__device__ __forceinline__ void montmul_streams(const Warp<K>& w, const Stream (&st)[NS]) {
  const int lane = w.lane, nb = w.nb;
  const uint32_t qoff = (uint32_t)(nb * K * 4), boff = (uint32_t)(lane * K * 4);
  uint32_t e[NS][2 * K + 2], t[NS][K], r[NS][K];
  sa x1[NS], y1[NS], x2[NS], y2[NS], zero[NS], tt[NS], qq[NS], nn[NS], ni[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    x1[s] = st[s].X1 != 0 ? st[s].X1 : st[s].T; y1[s] = st[s].Y1; x2[s] = st[s].X2; y2[s] = st[s].Y2;
    zero[s] = 0; tt[s] = st[s].T; qq[s] = st[s].T + qoff; nn[s] = w.N; ni[s] = w.NI;
  }
  bool any_product = false;
#pragma unroll
  for (int s = 0; s < NS; ++s) any_product = any_product || st[s].X1 != 0;
  if (any_product) {   // (streams given as a ready T skip the first phase; never mixed in practice)
    product<K, NS>(e, w.pf, lane, x1, y1, x2, y2);
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      resolve<K>(t[s], e[s], nullptr, lane);
      if (lane < nb) sts<K>(tt[s] + boff, t[s]);
    }
  } else {
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      if (lane < 2 * nb) lds<K>(t[s], tt[s] + boff);
      else {
#pragma unroll
        for (int k = 0; k < K; ++k) t[s][k] = 0;
      }
    }
  }
  __syncwarp();
  product<K, NS>(e, w.pl, lane, tt, ni, zero, zero);
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    resolve<K>(r[s], e[s], nullptr, lane);
    if (lane < nb) sts<K>(qq[s] + boff, r[s]);
  }
  __syncwarp();
  product<K, NS>(e, w.pf, lane, qq, nn, zero, zero);
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    resolve<K>(r[s], e[s], t[s], lane);
    if (lane >= nb && lane < 2 * nb) sts<K>(st[s].out + (uint32_t)((lane - nb) * K * 4), r[s]);
  }
  __syncwarp();
}

template <int K>
__device__ __noinline__ void montmul(const Warp<K> w, sa out, sa X1, sa Y1, sa X2, sa Y2) {
  const Stream st[1] = {{out, X1, Y1, X2, Y2, w.T}};
  montmul_streams<K, 1>(w, st);
}
// two products at once; the second stream's scratch is w.T + 2*nb*K words, its quotient after it
template <int K>
__device__ __noinline__ void montmul2(const Warp<K> w, sa out0, sa X10, sa Y10, sa X20, sa Y20, sa out1, sa X11, sa Y11) {
  const Stream st[2] = {{out0, X10, Y10, X20, Y20, w.T}, {out1, X11, Y11, 0, 0, w.T + (uint32_t)(2 * w.nb * K * 4)}};
  montmul_streams<K, 2>(w, st);
}

// dst <- b2 - m kept in [0, R) congruent modulo N (pair_fixup of dkg_nsq.cuh): S = b2 + (R - m);
// if that passes R drop R, else add (-R mod N) and take N off once if that passes R.
template <int K>
__device__ __noinline__ void fixup(const Warp<K> w, sa dst, sa b2, sa m, sa dneg) {
  uint32_t x[K], y[K], s[K];
  w.load_block(x, b2);
  w.load_block(y, m);
  const uint32_t ge = sub<K>(s, x, y, w.lane, w.nb);   // b2 + ~m + 1: carry <=> S >= R
  if (!ge) {
    w.load_block(y, dneg);
    const uint32_t c2 = add<K>(x, s, y, 0u, w.lane, w.nb);
    if (c2) {
      w.load_block(y, w.N);
      sub<K>(s, x, y, w.lane, w.nb);
    } else {
#pragma unroll
      for (int k = 0; k < K; ++k) s[k] = x[k];
    }
  }
  w.store_block(dst, s);
  __syncwarp();
}

// Pair state (A, B) in shared memory plus scratch A2 (2A).
struct PairAddr {
  sa A, B, A2, dneg;
};

// (A, B) <- (A, B) * (C, D)
template <int K>
__device__ __noinline__ void pair_mul(const Warp<K> w, const PairAddr pr, sa C, sa D) {
  // B <- REDC(B c + A d) and A <- REDC(A c) (quotient m) in one interleaved instruction stream
  montmul2<K>(w, pr.B, pr.B, C, pr.A, D, pr.A, pr.A, C);
  fixup<K>(w, pr.B, pr.B, w.Q2(), pr.dneg);
}
template <int K>
__device__ __noinline__ void pair_sqr(const Warp<K> w, const PairAddr pr) {
  uint32_t x[K];
  w.load_block(x, pr.A);
  shl1<K>(x, w.lane);                      // A < 2N <= R/4: no bit is lost
  w.store_block(pr.A2, x);
  __syncwarp();
  // B <- REDC(2 A B) and A <- REDC(A^2) (quotient m) in one interleaved instruction stream
  montmul2<K>(w, pr.B, pr.A2, pr.B, 0, 0, pr.A, pr.A, pr.A);
  fixup<K>(w, pr.B, pr.B, w.Q2(), pr.dneg);
}

// Almost-inverse (Kaliski 1995) of the plain value in `src` modulo N, on lane registers:
//   u = N, v = a, r = 0, s = 1;  while v > 0: halve the even one / subtract the smaller from the
//   larger and halve, doubling the other cofactor;  ends with u = gcd and r = -a^-1 2^k (mod N).
// Then x = (N - r) 2^-k by one or two Montgomery reductions of (N - r) << (m - k).  Writes the
// inverse (< 2N) to dst and returns true, or returns false if gcd(a, N) != 1.
template <int K>
__device__ __noinline__ bool mod_inverse(const Warp<K> w, sa dst, sa src) {
  const int lane = w.lane, nb = w.nb;
  uint32_t u[K], v[K], r[K], s[K], t[K], nreg[K];
  w.load_block(nreg, w.N);
  w.load_block(v, src);
#pragma unroll
  for (int k = 0; k < K; ++k) { u[k] = nreg[k]; r[k] = 0; s[k] = 0; }
  if (lane == 0) s[0] = 1;
  int k2 = 0;
  while (!is_zero<K>(v)) {
    const uint32_t u0 = __shfl_sync(kCoopFull, u[0], 0), v0 = __shfl_sync(kCoopFull, v[0], 0);
    if ((u0 & 1u) == 0) { shr1<K>(u, lane); shl1<K>(s, lane); }
    else if ((v0 & 1u) == 0) { shr1<K>(v, lane); shl1<K>(r, lane); }
    else if (greater<K>(u, v)) {
      sub<K>(t, u, v, lane, nb);
#pragma unroll
      for (int k = 0; k < K; ++k) u[k] = t[k];
      shr1<K>(u, lane);
      add<K>(t, r, s, 0u, lane, nb);
#pragma unroll
      for (int k = 0; k < K; ++k) r[k] = t[k];
      shl1<K>(s, lane);
    } else {
      sub<K>(t, v, u, lane, nb);
#pragma unroll
      for (int k = 0; k < K; ++k) v[k] = t[k];
      shr1<K>(v, lane);
      add<K>(t, s, r, 0u, lane, nb);
#pragma unroll
      for (int k = 0; k < K; ++k) s[k] = t[k];
      shl1<K>(r, lane);
    }
    ++k2;
  }
  // u == 1 ?
  {
    uint32_t rest = 0;
#pragma unroll
    for (int k = 0; k < K; ++k) rest |= (lane == 0 && k == 0) ? (u[k] ^ 1u) : u[k];
    if (__ballot_sync(kCoopFull, rest != 0) != 0u) return false;
  }
  // r < 2N: bring below N, y = N - r
  if (sub<K>(t, r, nreg, lane, nb)) {
#pragma unroll
    for (int k = 0; k < K; ++k) r[k] = t[k];
  }
  sub<K>(t, nreg, r, lane, nb);     // y = N - r in (0, N]
  const int m = 32 * K * nb, L2 = 2 * nb * K;
  for (int pass = 0; pass < 2; ++pass) {
    int sh;
    if (k2 > m) { sh = 0; k2 -= m; }      // first y <- REDC(y) = y 2^-m
    else { sh = m - k2; k2 = 0; pass = 1; }
    // T = y << sh as 2nb blocks, through the warp's T | Q area
    if (lane < nb) sts<K>(w.T + (uint32_t)(lane * K * 4), t);
    else if (lane < 2 * nb) {
      uint32_t z[K];
#pragma unroll
      for (int k = 0; k < K; ++k) z[k] = 0;
      sts<K>(w.T + (uint32_t)(lane * K * 4), z);
    }
    __syncwarp();
    const int ws = sh >> 5, bs = sh & 31;
    uint32_t tb[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int g = lane * K + k - ws;
      const uint32_t hi = (g >= 0 && g < L2) ? lds1(w.T + (uint32_t)(g * 4)) : 0u;
      const uint32_t lo = (g - 1 >= 0 && g - 1 < L2) ? lds1(w.T + (uint32_t)((g - 1) * 4)) : 0u;
      tb[k] = bs ? ((hi << bs) | (lo >> (32 - bs))) : hi;
    }
    __syncwarp();
    if (lane < 2 * nb) sts<K>(w.T + (uint32_t)(lane * K * 4), tb);
    __syncwarp();
    montmul<K>(w, dst, 0, 0, 0, 0);
    w.load_block(t, dst);
  }
  return true;
}

}  // namespace coop

// ---- pair-arithmetic exponentiation, one instance per warp ------------------------------------------
template <int K, int THREADS>
__global__ void __launch_bounds__(THREADS) coop_nsq_kernel(const CoopNsqParams p) {
  using namespace coop;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint32_t* S = reinterpret_cast<uint32_t*>(smem_raw);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int nb = p.nb, Lc = nb * K;
  // CTA: the constants; per warp: A B A2 T0 Q0 T1 Q1 C D XA XB YA YB I0
  for (int i = threadIdx.x; i < kCoopNsqConsts * Lc; i += blockDim.x) S[i] = p.consts[i];
  __syncthreads();
  const uint32_t *cONEA = S + 5 * Lc;
  const sa c0 = saddr(S), LB = (uint32_t)(Lc * 4);
  const sa sN = c0, sNI = c0 + LB, sDNEG = c0 + 2 * LB, sR2A = c0 + 3 * LB, sR2B = c0 + 4 * LB, sONEA = c0 + 5 * LB,
           sONEB = c0 + 6 * LB, sTWOA = c0 + 7 * LB, sTWOB = c0 + 8 * LB, sPLAIN1 = c0 + 9 * LB, sZERO = c0 + 10 * LB;
  uint32_t* W = S + kCoopNsqConsts * Lc + (size_t)warp * kCoopNsqWarpBufs * Lc;
  uint32_t *A = W, *B = W + Lc, *C = W + 7 * Lc, *XA = W + 9 * Lc, *YA = W + 11 * Lc, *I0 = W + 13 * Lc;
  const sa w0 = saddr(W);
  const sa sA = w0, sB = w0 + LB, sA2 = w0 + 2 * LB, sT = w0 + 3 * LB, sC = w0 + 7 * LB, sD = w0 + 8 * LB,
           sXA = w0 + 9 * LB, sXB = w0 + 10 * LB, sYA = w0 + 11 * LB, sYB = w0 + 12 * LB, sI0 = w0 + 13 * LB;

  Warp<K> w;
  w.lane = lane; w.nb = nb; w.pf.load(p.full, lane); w.pl.load(p.low, lane);
  w.N = sN; w.NI = sNI; w.T = sT;
  PairAddr pr;
  pr.A = sA; pr.B = sB; pr.A2 = sA2; pr.dneg = sDNEG;

  const unsigned gwarp = blockIdx.x * nwarps + warp;
  uint32_t* tab = p.scratch + (size_t)gwarp * p.scratch_per_warp;   // entry k: a at 2k*Lc, b right after
  auto copy = [&](uint32_t* dst, const uint32_t* src, int n) {
    for (int l = lane; l < n; l += 32) dst[l] = src[l];
  };

  for (;;) {
    unsigned long long idx = 0;
    if (lane == 0) idx = atomicAdd(p.counter, 1u);
    idx = __shfl_sync(kCoopFull, idx, 0);
    if (idx >= p.count * (unsigned long long)p.nparties) break;
    const int party = (int)(idx / p.count);
    const unsigned long long ct = idx % p.count;
    const uint32_t* ops = p.ops[party];
    const int nops = p.nops[party], tn = p.tab_entries[party], table_odd = p.table_odd[party], negative = p.negative[party];
    copy(A, p.pairs_in + ct * (unsigned long long)(2 * Lc), 2 * Lc);   // A | B contiguous
    __syncwarp();
    bool ok = true;
    if (negative) { copy(I0, A, Lc); __syncwarp(); }
    pair_mul<K>(w, pr, sR2A, sR2B);             // into the Montgomery domain: x R
    if (negative) {
      // x^-1 = y0 (2 - x y0) with y0 = (x mod N)^-1 taken modulo N: one Newton step modulo N^2
      copy(XA, A, 2 * Lc); __syncwarp();        // XA | XB
      ok = mod_inverse<K>(w, sI0, sI0);
      if (ok) {
        copy(A, I0, Lc);
        for (int l = lane; l < Lc; l += 32) B[l] = 0;
        __syncwarp();
        pair_mul<K>(w, pr, sR2A, sR2B);         // P(y0)
        copy(YA, A, 2 * Lc); __syncwarp();
        pair_mul<K>(w, pr, sXA, sXB);           // P(x y0) = P(1 + t N)
        {
          uint32_t x[K], y[K], s[K];
          w.load_block(x, sTWOA);
          w.load_block(y, sA);
          sub<K>(s, x, y, lane, nb);            // (2 ONE_a + 2N) - z_a in (0, 4N)
          w.store_block(sA, s);
          __syncwarp();
        }
        fixup<K>(w, sB, sTWOB, sB, sDNEG);      // (2 ONE_b - 2R) - z_b
        pair_mul<K>(w, pr, sYA, sYB);           // P(x^-1)
      }
    }
    if (ok) {
      if (nops == 0) {
        copy(A, cONEA, 2 * Lc); __syncwarp();   // ONEA | ONEB contiguous
      } else {
        auto entry = [&](int k) -> uint32_t* { return tab + (size_t)k * 2 * Lc; };
        copy(entry(0), A, 2 * Lc);
        if (tn > 1) {
          int src = 0;
          if (table_odd) {                      // odd powers: multiply by c^2, kept after the last entry
            pair_sqr<K>(w, pr);
            copy(entry(tn), A, 2 * Lc);
            __syncwarp();
            copy(A, entry(0), 2 * Lc);
            src = tn;
          }
          __syncwarp();
          copy(C, entry(src), 2 * Lc);          // C | D contiguous
          __syncwarp();
          for (int k = 1; k < tn; ++k) {
            pair_mul<K>(w, pr, sC, sD);
            copy(entry(k), A, 2 * Lc);
          }
        }
        __syncwarp();
        // constant-time table access: scan every entry (and the Montgomery one for digit 0) under
        // a mask instead of reading entry `di` (see modexp_nsq_kernel)
        auto ct_select = [&](uint32_t* dst, uint32_t di) {
          const uint32_t m0 = 0u - (uint32_t)(di == 0xfeu);
          for (int l = lane; l < 2 * Lc; l += 32) {
            uint32_t acc = cONEA[l] & m0;
            for (int k = 0; k < tn; ++k) acc |= entry(k)[l] & (0u - (uint32_t)((uint32_t)k == di));
            dst[l] = acc;
          }
        };
        if (p.ct_table) ct_select(A, ops[0] & 0xffu);
        else copy(A, entry((int)(ops[0] & 0xffu)), 2 * Lc);
        __syncwarp();
        for (int t = 1; t < nops; ++t) {
          const uint32_t op = ops[t];
          for (uint32_t q = op >> 8; q > 0; --q) pair_sqr<K>(w, pr);
          const uint32_t di = op & 0xffu;
          if (p.ct_table) {
            ct_select(C, di);
            __syncwarp();
            pair_mul<K>(w, pr, sC, sD);
          } else if (di == 0xfeu) pair_mul<K>(w, pr, sONEA, sONEB);
          else if (di != 0xffu) {
            copy(C, entry((int)di), 2 * Lc);
            __syncwarp();
            pair_mul<K>(w, pr, sC, sD);
          }
        }
      }
      pair_mul<K>(w, pr, sPLAIN1, sZERO);       // out of the Montgomery domain
      copy(p.pairs_out + idx * (unsigned long long)(2 * Lc), A, 2 * Lc);
    } else {
      for (int l = lane; l < 2 * Lc; l += 32) p.pairs_out[idx * (unsigned long long)(2 * Lc) + l] = 0;
    }
    if (p.status != nullptr && lane == 0) p.status[idx] = ok ? 0 : 1;
    __syncwarp();
  }
}

// ---- share combination, one ciphertext per warp -------------------------------------------------------
// x = prod_j partial_j mod N^2 (Montgomery products on the plain inputs, one multiplication by
// R^shares at the end); y = x - 1; N | y and u = y / N from ONE Montgomery reduction of y modulo N:
// with q = y * (-N^-1) mod R,  (y + q N) / R = N  <=>  y = (R - q) N,  so u = R - q (u = 0: y = 0);
// m = u * theta^-1 mod N.
template <int K, int THREADS>
__global__ void __launch_bounds__(THREADS) coop_combine_kernel(const CoopCombineParams p) {
  using namespace coop;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint32_t* S = reinterpret_cast<uint32_t*>(smem_raw);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nb = p.nb, Lc = nb * K;
  for (int i = threadIdx.x; i < kCoopCombineConsts * Lc; i += blockDim.x) S[i] = p.consts[i];
  __syncthreads();
  const sa c0 = saddr(S), LB = (uint32_t)(Lc * 4);
  const sa sN2 = c0, sNI2 = c0 + LB, sRPOW = c0 + 2 * LB, sN = c0 + 3 * LB, sNIN = c0 + 4 * LB, sTHR = c0 + 5 * LB;
  uint32_t* W = S + kCoopCombineConsts * Lc + (size_t)warp * kCoopCombineWarpBufs * Lc;
  uint32_t *X = W, *Y = W + Lc;
  const sa w0 = saddr(W);
  const sa sX = w0, sY = w0 + LB, sT = w0 + 2 * LB, sU = w0 + 4 * LB;
  Warp<K> w2;   // modulo N^2
  w2.lane = lane; w2.nb = nb; w2.pf.load(p.full, lane); w2.pl.load(p.low, lane);
  w2.N = sN2; w2.NI = sNI2; w2.T = sT;
  Warp<K> w1 = w2;   // modulo N
  w1.N = sN; w1.NI = sNIN;
  uint32_t n2reg[K], nreg[K];
  w2.load_block(n2reg, sN2);
  w1.load_block(nreg, sN);

  for (;;) {
    unsigned long long idx = 0;
    if (lane == 0) idx = atomicAdd(p.counter, 1u);
    idx = __shfl_sync(kCoopFull, idx, 0);
    if (idx >= p.count) break;
    const uint32_t* row = p.partials + idx * (unsigned long long)p.l2;
    for (int l = lane; l < Lc; l += 32) X[l] = l < p.l2 ? row[l] : 0u;
    __syncwarp();
    for (int s = 1; s < p.shares; ++s) {
      row = p.partials + ((unsigned long long)s * p.count + idx) * (unsigned long long)p.l2;
      for (int l = lane; l < Lc; l += 32) Y[l] = l < p.l2 ? row[l] : 0u;
      __syncwarp();
      montmul<K>(w2, sX, sX, sY, 0, 0);
    }
    montmul<K>(w2, sX, sX, sRPOW, 0, 0);         // plain product modulo N^2, < 2 N^2
    uint32_t x[K], t[K], one[K];
    w2.load_block(x, sX);
    if (sub<K>(t, x, n2reg, lane, nb)) {
#pragma unroll
      for (int k = 0; k < K; ++k) x[k] = t[k];
    }
    bool bad = is_zero<K>(x);                    // x = 0: (0 - 1) % N != 0 in the reference
#pragma unroll
    for (int k = 0; k < K; ++k) one[k] = (lane == 0 && k == 0) ? 1u : 0u;
    sub<K>(t, x, one, lane, nb);                 // y = x - 1
    const bool y_zero = is_zero<K>(t);
    // y as a 2nb-block number in the T | Q area (high half zero), then its Montgomery reduction mod N
    if (lane < nb) sts<K>(sT + (uint32_t)(lane * K * 4), t);
    else if (lane < 2 * nb) {
      uint32_t z[K];
#pragma unroll
      for (int k = 0; k < K; ++k) z[k] = 0;
      sts<K>(sT + (uint32_t)(lane * K * 4), z);
    }
    __syncwarp();
    montmul<K>(w1, sU, 0, 0, 0, 0);              // U <- (y + q N) / R, q in w1.Q()
    w1.load_block(x, sU);
    uint32_t diff = 0;
#pragma unroll
    for (int k = 0; k < K; ++k) diff |= x[k] ^ nreg[k];
    const bool is_n = __ballot_sync(kCoopFull, diff != 0) == 0u;
    bad = bad || !(is_n || y_zero);
    // u = R - q  (0 when y = 0)
    uint32_t q[K], nq[K], zero[K];
    w1.load_block(q, w1.Q());
#pragma unroll
    for (int k = 0; k < K; ++k) { nq[k] = lane < nb ? ~q[k] : 0u; zero[k] = 0; }
    add<K>(t, nq, zero, 1u, lane, nb);
    if (y_zero) {
#pragma unroll
      for (int k = 0; k < K; ++k) t[k] = 0;
    }
    w1.store_block(sU, t);
    __syncwarp();
    montmul<K>(w1, sU, sU, sTHR, 0, 0);          // u * theta^-1 mod N, < 2N
    w1.load_block(x, sU);
    if (sub<K>(t, x, nreg, lane, nb)) {
#pragma unroll
      for (int k = 0; k < K; ++k) x[k] = t[k];
    }
    if (bad) {
#pragma unroll
      for (int k = 0; k < K; ++k) x[k] = 0;
    }
    w1.store_block(sU, x);
    __syncwarp();
    uint32_t* o = p.out + idx * (unsigned long long)p.ln;
    const uint32_t* U = W + 4 * Lc;
    for (int l = lane; l < p.ln; l += 32) o[l] = U[l];
    if (p.status != nullptr && lane == 0) p.status[idx] = bad ? 2 : 0;
    __syncwarp();
  }
}

// ---- grouped exponentiation (per-instance modulus and exponent), one instance per warp ---------------
// CT: constant-time table access (DESIGN.md §2.11), its own instantiation chosen by the host
template <int K, int THREADS, bool CT = false>
__global__ void __launch_bounds__(THREADS) coop_grouped_kernel(const CoopGroupedParams p) {
  using namespace coop;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int nb = p.nb, Lc = nb * K;
  // per warp: N NI X T Q Y R2 ONE U
  uint32_t* W = reinterpret_cast<uint32_t*>(smem_raw) + (size_t)warp * 9 * Lc;
  uint32_t *N = W, *X = W + 2 * Lc, *Y = W + 5 * Lc, *ONE = W + 7 * Lc;
  const sa w0 = saddr(W), LB = (uint32_t)(Lc * 4);
  const sa sN = w0, sNI = w0 + LB, sX = w0 + 2 * LB, sT = w0 + 3 * LB, sY = w0 + 5 * LB, sR2 = w0 + 6 * LB,
           sONE = w0 + 7 * LB, sU = w0 + 8 * LB;
  Warp<K> w;
  w.lane = lane; w.nb = nb; w.pf.load(p.full, lane); w.pl.load(p.low, lane);
  w.N = sN; w.NI = sNI; w.T = sT;
  const unsigned gwarp = blockIdx.x * nwarps + warp;
  uint32_t* tab = p.scratch + (size_t)gwarp * p.scratch_per_warp;   // entry k (value x^(k+1)) at k*Lc
  auto copy = [&](uint32_t* dst, const uint32_t* src, int n) {
    for (int l = lane; l < n; l += 32) dst[l] = src[l];
  };
  const unsigned long long count = p.groups * (unsigned long long)p.per_group;
  const int m = 32 * Lc;

  for (;;) {
    unsigned long long idx = 0;
    if (lane == 0) idx = atomicAdd(p.counter, 1u);
    idx = __shfl_sync(kCoopFull, idx, 0);
    if (idx >= count) break;
    const unsigned long long g = idx / (unsigned long long)p.per_group;
    const uint32_t* mod = p.moduli + g * (unsigned long long)p.limbs;
    const uint32_t* base = p.bases + idx * (unsigned long long)p.limbs;
    for (int l = lane; l < Lc; l += 32) {
      N[l] = l < p.limbs ? mod[l] : 0u;
      X[l] = l < p.limbs ? base[l] : 0u;
    }
    __syncwarp();
    uint32_t nreg[K], x[K], t[K];
    w.load_block(nreg, sN);
    // ---- -N^-1 mod R by Newton: inv <- inv (2 - N inv), precision doubling from 32 bits
    {
      const uint32_t n0 = N[0];
      uint32_t inv0 = n0;
#pragma unroll
      for (int i = 0; i < 5; ++i) inv0 *= 2u - n0 * inv0;
#pragma unroll
      for (int k = 0; k < K; ++k) x[k] = (lane == 0 && k == 0) ? inv0 : 0u;
      w.store_block(sNI, x);
      __syncwarp();
      uint32_t zero[K], nt[K], u[K];
#pragma unroll
      for (int k = 0; k < K; ++k) zero[k] = 0;
      for (int prec = 32; prec < m; prec *= 2) {
        w.mul_low(t, sN, sNI);                          // N inv mod R
#pragma unroll
        for (int k = 0; k < K; ++k) nt[k] = lane < nb ? ~t[k] : 0u;
        add<K>(u, nt, zero, 3u, lane, nb);              // 2 - t = ~t + 3
        w.store_block(sU, u);
        __syncwarp();
        w.mul_low(t, sNI, sU);
        __syncwarp();
        w.store_block(sNI, t);
        __syncwarp();
      }
      w.load_block(t, sNI);
#pragma unroll
      for (int k = 0; k < K; ++k) nt[k] = lane < nb ? ~t[k] : 0u;
      add<K>(x, nt, zero, 1u, lane, nb);                // negate
      w.store_block(sNI, x);
      __syncwarp();
    }
    // ---- R mod N: 2^(n-1) doubled m - n + 1 times with a conditional subtraction each
    {
      uint32_t nz = 0;
      int top_bit = 0;   // bit length within this lane's block
#pragma unroll
      for (int k = 0; k < K; ++k) {
        nz |= nreg[k];
        if (nreg[k]) top_bit = 32 * k + (32 - __clz(nreg[k]));
      }
      const uint32_t lanes_nz = __ballot_sync(kCoopFull, nz != 0);
      const int top_lane = 31 - __clz(lanes_nz);
      top_bit = __shfl_sync(kCoopFull, top_bit, top_lane);
      const int nbits = top_lane * 32 * K + top_bit;
      const int b = nbits - 1;
#pragma unroll
      for (int k = 0; k < K; ++k) x[k] = (nbits > 1 && lane == b / (32 * K) && k == (b % (32 * K)) / 32) ? (1u << (b % 32)) : 0u;
      for (int i = 0; i < m - b; ++i) double_mod<K>(x, nreg, lane, nb);   // N == 1: stays 0
      w.store_block(sONE, x);
      // R^2 mod N: 2^o R by doublings, then e Montgomery squarings, m = 2^e * o
      int e = 0, o = m;
      while ((o & 1) == 0) { o >>= 1; ++e; }
      for (int i = 0; i < o; ++i) double_mod<K>(x, nreg, lane, nb);
      w.store_block(sR2, x);
      __syncwarp();
      for (int i = 0; i < e; ++i) montmul<K>(w, sR2, sR2, sR2, 0, 0);
    }
    // ---- exponentiation: fixed windows, every window multiplies
    montmul<K>(w, sX, sX, sR2, 0, 0);                   // x R
    const int tn = (1 << p.wbits) - 1;
    copy(tab, X, Lc);
    copy(Y, X, Lc);
    __syncwarp();
    for (int k = 1; k < tn; ++k) {
      montmul<K>(w, sX, sX, sY, 0, 0);
      copy(tab + (size_t)k * Lc, X, Lc);
    }
    __syncwarp();
    const uint32_t* ex = p.exps + g * (unsigned long long)p.exp_limbs;
    if constexpr (CT) {
      // constant-time table access: from ONE, every window scans all entries and ONE (digit 0)
      // under a mask into Y, lane-strided as in coop_nsq_kernel, and multiplies by Y; the digit
      // comes from shifts and masks (the conditions are on bit positions only)
      auto digit = [&](int tdig) -> uint32_t {
        const int lowbit = p.wbits * (p.ndigits - 1 - tdig);
        const int wi = lowbit / 32;
        const uint64_t lo = wi < p.exp_limbs ? ex[wi] : 0u, hi = wi + 1 < p.exp_limbs ? ex[wi + 1] : 0u;
        return (uint32_t)((hi << 32 | lo) >> (lowbit % 32)) & ((1u << p.wbits) - 1u);
      };
      copy(X, ONE, Lc);
      for (int td = 0; td < p.ndigits; ++td) {
        if (td > 0)
          for (int q = 0; q < p.wbits; ++q) montmul<K>(w, sX, sX, sX, 0, 0);
        const uint32_t dg = digit(td), di = dg - 1u, m0 = 0u - (uint32_t)(dg == 0u);
        for (int l = lane; l < Lc; l += 32) {
          uint32_t acc = ONE[l] & m0;
          for (int k = 0; k < tn; ++k) acc |= tab[(size_t)k * Lc + l] & (0u - (uint32_t)((uint32_t)k == di));
          Y[l] = acc;
        }
        __syncwarp();
        montmul<K>(w, sX, sX, sY, 0, 0);
      }
    } else {
      auto digit = [&](int tdig) -> uint32_t {
        const int lowbit = p.wbits * (p.ndigits - 1 - tdig);
        uint32_t v = 0;
        for (int bb = 0; bb < p.wbits; ++bb) {
          const int bit = lowbit + bb;
          if (bit < 32 * p.exp_limbs && ((ex[bit / 32] >> (bit % 32)) & 1u)) v |= 1u << bb;
        }
        return v;
      };
      {
        const uint32_t d0 = digit(0);
        if (d0) copy(X, tab + (size_t)(d0 - 1) * Lc, Lc); else copy(X, ONE, Lc);
        __syncwarp();
      }
      for (int td = 1; td < p.ndigits; ++td) {
        for (int q = 0; q < p.wbits; ++q) montmul<K>(w, sX, sX, sX, 0, 0);
        const uint32_t dg = digit(td);
        if (dg) { copy(Y, tab + (size_t)(dg - 1) * Lc, Lc); __syncwarp(); montmul<K>(w, sX, sX, sY, 0, 0); }
        else montmul<K>(w, sX, sX, sONE, 0, 0);
      }
    }
    // ---- out of the Montgomery domain, canonical residue
    {
#pragma unroll
      for (int k = 0; k < K; ++k) x[k] = (lane == 0 && k == 0) ? 1u : 0u;
      w.store_block(sY, x);
      __syncwarp();
      montmul<K>(w, sX, sX, sY, 0, 0);
      w.load_block(x, sX);
      if (sub<K>(t, x, nreg, lane, nb)) {
#pragma unroll
        for (int k = 0; k < K; ++k) x[k] = t[k];
      }
      w.store_block(sX, x);
      __syncwarp();
    }
    uint32_t* o = p.out + idx * (unsigned long long)p.limbs;
    for (int l = lane; l < p.limbs; l += 32) o[l] = X[l];
    __syncwarp();
  }
}

}  // namespace dkg
