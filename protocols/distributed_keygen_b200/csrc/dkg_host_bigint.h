// Host-side helpers that derive the per-key Montgomery constants when a context is created
// (once per key; never on the data path).  Plain schoolbook on little-endian uint32 limbs.
#pragma once
#include <stdint.h>
#include <vector>

namespace dkg_host {

using Limbs = std::vector<uint32_t>;

inline int bit_length(const uint32_t* a, int n) {
  for (int i = n - 1; i >= 0; --i)
    if (a[i]) return 32 * i + (32 - __builtin_clz(a[i]));
  return 0;
}

inline bool geq(const Limbs& a, const Limbs& b) {  // same length
  for (int i = (int)a.size() - 1; i >= 0; --i)
    if (a[i] != b[i]) return a[i] > b[i];
  return true;
}

inline void sub_inplace(Limbs& a, const Limbs& b) {
  uint64_t borrow = 0;
  for (size_t i = 0; i < a.size(); ++i) {
    uint64_t d = (uint64_t)a[i] - b[i] - borrow;
    a[i] = (uint32_t)d;
    borrow = d >> 63;
  }
}

// 2^bits mod n (n odd or any n > 0), n given on `len` limbs.
inline Limbs pow2_mod(size_t bits, const Limbs& n) {
  const size_t len = n.size();
  Limbs x(len, 0);
  x[0] = 1;
  if (!geq(n, x) || (bit_length(n.data(), (int)len) == 1)) {  // n == 1 (n == 0 is rejected earlier)
    x[0] = 0;
    return x;
  }
  // jump: 2^k for k < bitlen(n) needs no reduction
  const size_t nb = (size_t)bit_length(n.data(), (int)len);
  size_t k = bits < nb - 1 ? bits : nb - 1;
  x[0] = 0;
  x[k / 32] = 1u << (k % 32);
  for (; k < bits; ++k) {
    uint32_t carry = 0;
    for (size_t i = 0; i < len; ++i) {
      uint32_t nc = x[i] >> 31;
      x[i] = (x[i] << 1) | carry;
      carry = nc;
    }
    if (carry || geq(x, n)) sub_inplace(x, n);
  }
  return x;
}

// -a mod 2^(32 a.size())
inline Limbs negate(const Limbs& a) {
  Limbs r(a.size());
  uint64_t carry = 1;
  for (size_t i = 0; i < a.size(); ++i) {
    uint64_t t = (uint64_t)(~a[i]) + carry;
    r[i] = (uint32_t)t;
    carry = t >> 32;
  }
  return r;
}

// a^2 by schoolbook, without leading zero limbs (at least one limb)
inline Limbs square(const Limbs& a) {
  const size_t n = a.size();
  Limbs r(2 * n, 0);
  for (size_t i = 0; i < n; ++i) {
    uint64_t carry = 0;
    for (size_t j = 0; j < n; ++j) {
      uint64_t t = (uint64_t)a[i] * a[j] + r[i + j] + carry;
      r[i + j] = (uint32_t)t;
      carry = t >> 32;
    }
    r[i + n] = (uint32_t)carry;
  }
  while (r.size() > 1 && r.back() == 0) r.pop_back();
  return r;
}

// -n^-1 mod 2^(32*K) for odd n (Hensel lifting, one limb at a time)
inline Limbs neg_inv_block(const Limbs& n, int K) {
  // 32-bit inverse of n[0] by Newton
  uint32_t n0 = n[0];
  uint32_t inv0 = n0;  // correct to 3 bits
  for (int i = 0; i < 5; ++i) inv0 *= 2u - n0 * inv0;
  Limbs inv(K, 0), p(K, 0);  // p = n * inv mod 2^(32K), kept up to date
  auto nl = [&](int i) -> uint32_t { return i < (int)n.size() ? n[i] : 0u; };
  for (int i = 0; i < K; ++i) {
    // want p == 1 (mod 2^(32(i+1))): cancel limb i of (p - 1)
    uint32_t target = (i == 0) ? (1u - p[0]) : (0u - p[i]);
    uint32_t d = target * inv0;
    inv[i] = d;
    uint64_t carry = 0;
    for (int j = 0; i + j < K; ++j) {
      uint64_t t = (uint64_t)d * nl(j) + p[i + j] + carry;
      p[i + j] = (uint32_t)t;
      carry = t >> 32;
    }
  }
  return negate(inv);
}

// (a + b) mod n and (a - b) mod n for a, b < n (same length)
inline Limbs addmod(const Limbs& a, const Limbs& b, const Limbs& n) {
  Limbs r(a.size());
  uint64_t c = 0;
  for (size_t i = 0; i < a.size(); ++i) {
    uint64_t t = (uint64_t)a[i] + b[i] + c;
    r[i] = (uint32_t)t;
    c = t >> 32;
  }
  if (c || geq(r, n)) sub_inplace(r, n);
  return r;
}
inline Limbs submod(const Limbs& a, const Limbs& b, const Limbs& n) {
  Limbs r = a;
  if (!geq(a, b)) {
    uint64_t c = 0;
    for (size_t i = 0; i < r.size(); ++i) {
      uint64_t t = (uint64_t)r[i] + n[i] + c;
      r[i] = (uint32_t)t;
      c = t >> 32;
    }
  }
  sub_inplace(r, b);
  return r;
}

// a * b mod n by shift-and-add (only used for tiny one-off constants)
inline Limbs mulmod_slow(const Limbs& a, const Limbs& b, const Limbs& n) {
  const size_t len = n.size();
  Limbs r(len, 0);
  const int bits = bit_length(b.data(), (int)len);
  for (int k = bits - 1; k >= 0; --k) {
    uint32_t carry = 0;
    for (size_t i = 0; i < len; ++i) {
      uint32_t nc = r[i] >> 31;
      r[i] = (r[i] << 1) | carry;
      carry = nc;
    }
    if (carry || geq(r, n)) sub_inplace(r, n);
    if ((b[k / 32] >> (k % 32)) & 1u) {
      uint64_t c = 0;
      for (size_t i = 0; i < len; ++i) {
        uint64_t t = (uint64_t)r[i] + a[i] + c;
        r[i] = (uint32_t)t;
        c = t >> 32;
      }
      if (c || geq(r, n)) sub_inplace(r, n);
    }
  }
  return r;
}

// a = q * n + r by bit-serial long division (a: any length, n: n.size() limbs, n > 0);
// q has a.size() limbs, r has n.size() limbs.  One-off constants only.
inline void divmod_slow(const Limbs& a, const Limbs& n, Limbs* q, Limbs* r) {
  const size_t len = n.size();
  q->assign(a.size(), 0);
  r->assign(len, 0);
  const int abits = bit_length(a.data(), (int)a.size());
  for (int k = abits - 1; k >= 0; --k) {
    uint32_t carry = (a[k / 32] >> (k % 32)) & 1u;
    for (size_t i = 0; i < len; ++i) {
      const uint32_t nc = (*r)[i] >> 31;
      (*r)[i] = ((*r)[i] << 1) | carry;
      carry = nc;
    }
    if (carry || geq(*r, n)) {
      sub_inplace(*r, n);
      (*q)[k / 32] |= 1u << (k % 32);
    }
  }
}

}  // namespace dkg_host
