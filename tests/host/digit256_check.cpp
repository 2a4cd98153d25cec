// Host-side check of K1's radix-256 digit fast path (standardize.cu): the fma-with-magic-constant rounding and the
// PRMT / XOR byte packing of ozaki_store_slices256 must give the int8 digits of a plain balanced radix-256
// decomposition of the exactly rounded fixed-point integer q = rint(c * mul), mul = 2^39 / (row scale).  The device
// helpers are pasted in by tests/test_digit256_host.py (DIGIT_SNIPPET) with host stand-ins for the intrinsics.
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#define __device__
#define __forceinline__ inline
#define MCD_OZAKI_MAX_SLICES 8
static inline uint32_t __byte_perm(uint32_t a, uint32_t b, uint32_t s) {
  uint8_t src[8];
  std::memcpy(src, &a, 4);
  std::memcpy(src + 4, &b, 4);
  uint32_t r = 0;
  for (int i = 0; i < 4; ++i) {
    const int n = (s >> (4 * i)) & 0xf;
    uint8_t v = src[n & 7];
    if (n & 8) v = (v & 0x80) ? 0xff : 0;
    r |= (uint32_t)v << (8 * i);
  }
  return r;
}
static inline uint32_t __funnelshift_r(uint32_t lo, uint32_t hi, uint32_t sh) {
  return (uint32_t)((((uint64_t)hi << 32) | lo) >> (sh & 31));
}
static inline long long __double_as_longlong(double d) {
  long long r;
  std::memcpy(&r, &d, 8);
  return r;
}
static inline long long __double2ll_rn(double d) { return llrint(d); }
#include DIGIT_SNIPPET

constexpr int NSL = 5;

// q = the exact product c * mul rounded once to the nearest integer, ties to even
static long long exact_rint(double c, double mul) {
  const double p = c * mul, err = std::fma(c, mul, -p), fl = std::floor(p);
  if (p - fl == 0.5) return (long long)(err > 0 ? fl + 1 : err < 0 ? fl : std::rint(p));
  return (long long)std::rint(p);
}

// plain balanced radix-256 digits by repeated division: d_t in [-128, 127] for t > 0, the rest in d_0
static void reference_digits(long long q, int d[NSL]) {
  long long r = q;
  for (int t = NSL - 1; t > 0; --t) {
    long long m = ((r % 256) + 256) % 256;  // floor mod
    if (m >= 128) m -= 256;
    d[t] = (int)m;
    r = (r - m) / 256;
  }
  d[0] = (int)r;
}

static long bad = 0, lead_pos = 0, lead_neg = 0;

static void check4(const double (&c)[4], double mul) {
  const unsigned long long B = 0x8080808080808080ull & ((1ull << (8 * NSL)) - 1ull);
  const double magic = 6755399441055744.0 + (double)B;
  uint32_t lo[4], hi[4];
  int dref[4][NSL];
  for (int i = 0; i < 4; ++i) {
    ozaki_bits<NSL>(c[i], mul, magic, lo[i], hi[i]);
    const long long q = exact_rint(c[i], mul);
    reference_digits(q, dref[i]);
    if (dref[i][0] < -64 || dref[i][0] > 64) ++bad;  // |q| <= 2^38
    lead_pos += dref[i][0] == 64;
    lead_neg += dref[i][0] == -64;
    int dgen[MCD_OZAKI_MAX_SLICES];  // the generic kernels' helper agrees too
    ozaki_digits256((double)q, NSL, dgen);
    for (int t = 0; t < NSL; ++t) bad += dgen[t] != dref[i][t];
  }
  int8_t out[NSL * 16];
  std::memset(out, 0x55, sizeof out);
  ozaki_store_slices256<NSL, 0>(lo, hi, out, 16);
  for (int sl = 0; sl < NSL; ++sl)
    for (int i = 0; i < 4; ++i) bad += out[sl * 16 + i] != (int8_t)dref[i][sl];
}

int main() {
  const double top = ldexp(1.0, 8 * NSL - 1);  // 2^39
  // random rows: c * mul = y * 2^39 with |y| < 0.5, mul = 2^39 times a row factor in [1, 2) and a power of two
  for (long it = 0; it < 1000000; ++it) {
    const double mul = ldexp(1.0 + drand48(), (rand() % 5) + 8 * NSL - 3);
    double c[4];
    for (int i = 0; i < 4; ++i) {
      c[i] = (drand48() - 0.5) * 0.99999 * ldexp(1.0, -(rand() % 5)) * top / mul;
      if (it % 97 == 0 && i == 0) c[i] = 0.0;
      if (it % 89 == 0 && i == 1) c[i] = std::floor(c[i] * mul) / mul;          // exact integers and
      if (it % 83 == 0 && i == 2) c[i] = (std::floor(c[i] * mul) + 0.5) / mul;  // exact ties
      if (std::fabs(c[i] * mul) > ldexp(1.0, 8 * NSL - 2)) c[i] = 0.0;
    }
    check4(c, mul);
  }
  // edges with mul = 2^39: +-(0.5 - ulp) rounds to +-2^38 (leading digit +-64), 0, exact powers of two
  const double half_minus = std::nextafter(0.5, 0.0);
  const double edges[] = {half_minus, -half_minus, 0.0, -0.0, 0.25, -0.25, 0x1p-39, -0x1p-39, 0x1p-40, -0x1p-40,
                          0x1p-41, 0x1p-8, -0x1p-16, 0x1p-24, -0x1p-32, 0.375, -0.4999999};
  const int ne = sizeof edges / sizeof edges[0];
  for (int a = 0; a < ne; ++a)
    for (int b = 0; b < ne; ++b) {
      const double c[4] = {edges[a], edges[b], edges[(a + b) % ne], edges[(a + 2 * b + 1) % ne]};
      check4(c, top);
    }
  if (lead_pos == 0 || lead_neg == 0) ++bad;  // the leading digit must reach +-64
  std::printf("radix-256 digit bits: %ld mismatches (leading digit +64: %ld, -64: %ld)\n", bad, lead_pos, lead_neg);
  return bad != 0;
}
