// K1 -- per-cell standardisation (HBM-bound streaming kernel).
//
// Replaces the per-operand half of cosine_similarity_np (reference
// src/MaCroDNA/macrodna.py:24-25): for every cell row x[0..G) compute
//   mean = sum(x)/G,  c = x - mean,  norm = sqrt(sum(c^2))
// once, instead of twice per (RNA, DNA) pair as the reference does.
//
// Layout: X is cells x genes row-major (macrodna.py:93-94 hand-off), so one cell is
// one contiguous vector.  A group of T threads owns one row and keeps it in
// registers between the mean pass and the norm pass, so HBM sees exactly one read
// (8 B/element) and one write (8 B/element FP64 centred rows, or 4 B/element for the
// two fp16 slices of the tcgen05 path).  Loads/stores are 128-bit and coalesced; reductions are warp
// shuffles plus one shared-memory hop.
#include "mcd_internal.cuh"

#include <cuda_fp16.h>

#include <cstdlib>

namespace {

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Sum over the T threads that own one row.  `red` has BLOCK/32 doubles.
template <int T, int BLOCK>
__device__ __forceinline__ double group_sum(double v, double* red) {
  v = warp_sum(v);
  if (T == 32) return v;
  constexpr int WPG = T / 32;  // warps per row group
  const int warp = threadIdx.x >> 5;
  __syncthreads();  // protect `red` reuse between the two reductions
  if ((threadIdx.x & 31) == 0) red[warp] = v;
  __syncthreads();
  const int g0 = (warp / WPG) * WPG;
  double s = 0.0;
#pragma unroll
  for (int w = 0; w < WPG; ++w) s += red[g0 + w];
  return s;
}

// Max over the T threads that own one row (same protocol as group_sum).
template <int T, int BLOCK>
__device__ __forceinline__ double group_max(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  if (T == 32) return v;
  constexpr int WPG = T / 32;
  const int warp = threadIdx.x >> 5;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[warp] = v;
  __syncthreads();
  const int g0 = (warp / WPG) * WPG;
  double s = 0.0;
#pragma unroll
  for (int w = 0; w < WPG; ++w) s = fmax(s, red[g0 + w]);
  return s;
}

// A zero-variance cell must standardise to EXACTLY zero (reference: its correlations are exactly 0.0, SURVEY
// App. B), but sum/G need not reproduce the constant bit for bit, which would leave a row of identical rounding
// residues with a non-zero norm.  A row whose centred sum of squares is at rounding level relative to its mean
// (every residue below 2^-45 |mean|: nothing but the rounding of the mean) is therefore declared zero-variance:
// norm 0, unit row / digits / centred row all zero.
__device__ __forceinline__ bool flat_row(double ss, double mean, int G) {
  const double r = mean * 0x1p-45;
  return ss <= (double)G * r * r;
}

// Integer-slice operand of the int8 tensor-core path (corr_ozaki.cu).  y (|y| < 0.5) is rounded to the
// fixed-point integer q = rint(y * 2^(7*nsl-1)) and written as nsl balanced radix-128 digits d_t in [-64, 63],
//   q = sum_t d_t * 128^(nsl-1-t)      (t = 0 is the most significant slice).
// The products of two such digit vectors are exact in the tensor core's int32 accumulators.
// ys = y * 2^(7 nsl - 1), already scaled by the caller (one multiply by a per-row power of two).
__device__ __forceinline__ void ozaki_digits(double ys, int nsl, int d[MCD_OZAKI_MAX_SLICES]) {
  const long long q = __double2ll_rn(ys);  // |q| <= 2^(7 nsl - 2)
  // Adding 64 to every 7-bit field turns the balanced digits into plain bit fields: q + B = sum (d_t + 64) 128^..
  const unsigned long long B = (0x0102040810204081ull << 6) & ((1ull << (7 * nsl)) - 1ull);
  const unsigned long long qb = (unsigned long long)q + B;
#pragma unroll
  for (int t = 0; t < MCD_OZAKI_MAX_SLICES; ++t)
    d[t] = (t < nsl) ? (int)((qb >> (7 * (nsl - 1 - t))) & 127ull) - 64 : 0;
}

// Radix-256 form (nsl <= 7): q = rint(y * 2^(8 nsl - 1)) as nsl balanced digits d_t in [-128, 127], the leading one
// in [-64, 64] (|q| <= 2^(8 nsl - 2)).  Adding 128 to every byte makes them plain bytes: q + B = sum (d_t + 128) 256^..
__device__ __forceinline__ void ozaki_digits256(double ys, int nsl, int d[MCD_OZAKI_MAX_SLICES]) {
  const long long q = __double2ll_rn(ys);
  const unsigned long long B = 0x8080808080808080ull & ((1ull << (8 * nsl)) - 1ull);
  const unsigned long long qb = (unsigned long long)q + B;
#pragma unroll
  for (int t = 0; t < MCD_OZAKI_MAX_SLICES; ++t)
    d[t] = (t < nsl) ? (int)((qb >> (8 * (nsl - 1 - t))) & 255ull) - 128 : 0;
}

// digits of either radix, RB chosen at compile time (the generic kernels are instantiated per radix)
template <int RB>
__device__ __forceinline__ void ozaki_digits_of(double ys, int nsl, int d[MCD_OZAKI_MAX_SLICES]) {
  if constexpr (RB == 8)
    ozaki_digits256(ys, nsl, d);
  else
    ozaki_digits(ys, nsl, d);
}

// Split-precision operand for the tcgen05 path: y (|y| <= 1, a unit-norm centred value) is scaled by
// 2^8 and written as fp16 hi + fp16 lo (22 significant bits; the scale keeps `lo` out of the fp16
// subnormal range for every |y| > 5e-4).  hi*hi + hi*lo + lo*hi reproduces the product to ~2^-22.
__device__ __forceinline__ void split_fp16x2(double y, uint16_t& s0, uint16_t& s1) {
  const double ys = y * 256.0;
  const __half h0 = __double2half(ys);
  const double r = ys - (double)__half2float(h0);
  const __half h1 = __double2half(r);
  s0 = __half_as_ushort(h0);
  s1 = __half_as_ushort(h1);
}

// T threads per row, NV double2 per thread (row capacity 2*T*NV elements), VEC = 128-bit loads legal.
// gidx != nullptr: gene gather -- element g of the standardised row is X[row, gidx[g]] (the host only computes
// the index arrays of the gene intersection, macrodna.py:89-91; the data never gets re-indexed on the host).
// The row is then read with scattered 8-byte loads, but it is L1/L2 resident while its CTA works on it.
// RB: radix bits of the digit output (oz.rb), a template parameter so that each radix compiles to its own kernel.
template <int T, int NV, bool VEC, int RB>
__global__ void __launch_bounds__((T > 512 ? T : 512), 1)
standardize_rows(const double* __restrict__ X, const int* __restrict__ gidx, int64_t ncells, int G, int64_t ldx,
                 double* __restrict__ Y,
                 int64_t ldk, uint16_t* __restrict__ S, uint16_t* __restrict__ S_lo, int64_t ldk16,
                 double* __restrict__ norms, int* __restrict__ flags, const mcd_ozaki_out oz) {
  constexpr int BLOCK = (T > 512 ? T : 512);
  constexpr int ROWS = BLOCK / T;
  __shared__ double red[BLOCK / 32];
  const int t = threadIdx.x % T;
  const int64_t row = (int64_t)blockIdx.x * ROWS + threadIdx.x / T;
  const bool live = row < ncells;
  const double* x = X + (live ? row : 0) * ldx;

  double2 v[NV];
  double sum = 0.0;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int e = 2 * (t + k * T);
    double2 d = make_double2(0.0, 0.0);
    if (live) {
      if (gidx != nullptr) {
        if (e < G) d.x = __ldg(x + __ldg(gidx + e));
        if (e + 1 < G) d.y = __ldg(x + __ldg(gidx + e + 1));
      } else if (e + 1 < G) {
        if (VEC) {
          d = __ldcs(reinterpret_cast<const double2*>(x + e));
        } else {
          d.x = __ldcs(x + e);
          d.y = __ldcs(x + e + 1);
        }
      } else if (e < G) {
        d.x = __ldcs(x + e);
      }
    }
    v[k] = d;
    sum += d.x + d.y;
  }
  sum = group_sum<T, BLOCK>(sum, red);
  const double mean = sum / (double)G;

  double ss = 0.0;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int e = 2 * (t + k * T);
    double cx = (e < G) ? v[k].x - mean : 0.0;
    double cy = (e + 1 < G) ? v[k].y - mean : 0.0;
    v[k] = make_double2(cx, cy);
    ss += cx * cx + cy * cy;
  }
  ss = group_sum<T, BLOCK>(ss, red);
  const bool flat = flat_row(ss, mean, G);
  if (flat) ss = 0.0;  // zero-variance cell: norm 0, every output below becomes exactly zero
  const double nrm = sqrt(ss);
  double amax = 0.0;
  if (oz.digits != nullptr) {  // uniform over the block
#pragma unroll
    for (int k = 0; k < NV; ++k) amax = fmax(amax, fmax(fabs(v[k].x), fabs(v[k].y)));
    amax = group_max<T, BLOCK>(amax, red);
  }
  if (!live) return;
  if (t == 0) {
    norms[row] = nrm;
    if (!isfinite(sum) || !isfinite(ss)) atomicOr(flags, 1);
  }
  if (oz.digits != nullptr) {
    // unit row u = c / nrm scaled by 2^e so that max|u| * 2^e lies in [0.25, 0.5)
    const double inv = (nrm > 0.0 && isfinite(nrm)) ? 1.0 / nrm : 0.0;
    const double umax = amax * inv;
    int ex = 0;
    if (umax > 0.0 && isfinite(umax)) (void)frexp(umax, &ex);  // umax = f * 2^ex, f in [0.5, 1)
    const int e = -ex - 1;
    if (t == 0) oz.scale[row] = scalbn(1.0, -e);
    // one multiplier per row: 1/nrm times the exact power of two 2^(e + rb nsl - 1)  (bit-identical to scaling
    // the rounded quotient afterwards: a power-of-two factor commutes with rounding)
    const double mul = inv * scalbn(1.0, e + RB * oz.nsl - 1);
    int8_t* o = oz.digits + row * oz.ldk8;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int g = 2 * (t + k * T);
      if (g < G) {
        int d0[MCD_OZAKI_MAX_SLICES], d1[MCD_OZAKI_MAX_SLICES];
        ozaki_digits_of<RB>(v[k].x * mul, oz.nsl, d0);
        ozaki_digits_of<RB>((g + 1 < G) ? v[k].y * mul : 0.0, oz.nsl, d1);
#pragma unroll
        for (int sl = 0; sl < MCD_OZAKI_MAX_SLICES; ++sl)
          if (sl < oz.nsl)  // g is even and ldk8 a multiple of 64: aligned 2-byte store
            *reinterpret_cast<uint16_t*>(o + sl * oz.slice_stride + g) =
                (uint16_t)((uint32_t)(d0[sl] & 0xff) | ((uint32_t)(d1[sl] & 0xff) << 8));
      }
    }
    const int64_t g2 = (G + 1) & ~1;
    for (int sl = 0; sl < oz.nsl; ++sl)
      for (int64_t c = g2 + 2 * t; c < oz.ldk8; c += 2 * T)
        *reinterpret_cast<uint16_t*>(o + sl * oz.slice_stride + c) = 0;
  }

  if (Y != nullptr) {
    double* y = Y + row * ldk;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int e = 2 * (t + k * T);
      if (e + 1 < G) {
        *reinterpret_cast<double2*>(y + e) = flat ? make_double2(0.0, 0.0) : v[k];  // ldk % 16 == 0 -> aligned
      } else if (e < G) {
        y[e] = flat ? 0.0 : v[k].x;
      }
    }
    for (int64_t c = G + t; c < ldk; c += T) y[c] = 0.0;
  }
  if (S != nullptr) {
    const double inv = nrm > 0.0 ? 1.0 / nrm : 0.0;
    uint16_t* s0 = S + row * ldk16;
    uint16_t* s1 = S_lo + row * ldk16;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int e = 2 * (t + k * T);
      if (e < G) {
        uint16_t a0, a1, b0 = 0, b1 = 0;
        split_fp16x2(v[k].x * inv, a0, a1);
        if (e + 1 < G) split_fp16x2(v[k].y * inv, b0, b1);
        // e is even and ldk16 is a multiple of 64: 4-byte aligned pair store (pad column is zero)
        *reinterpret_cast<uint32_t*>(s0 + e) = (uint32_t)a0 | ((uint32_t)b0 << 16);
        *reinterpret_cast<uint32_t*>(s1 + e) = (uint32_t)a1 | ((uint32_t)b1 << 16);
      }
    }
    const int64_t g2 = (G + 1) & ~1;
    for (int64_t c = g2 + 2 * t; c < ldk16; c += 2 * T) {
      *reinterpret_cast<uint32_t*>(s0 + c) = 0u;
      *reinterpret_cast<uint32_t*>(s1 + c) = 0u;
    }
  }
}

// ---- digit-slice fast path (the default precision mode) ---------------------------------------------------------
// Same arithmetic as the digit branch of standardize_rows, restructured so that the kernel stays on the HBM
// roofline instead of the issue slots (ncu of the generic kernel: 128 instructions per element, 47 % of the copy
// bandwidth):
//   * a thread owns 4 CONSECUTIVE genes per sweep (one 256-bit ld.global.cs, LDG.256), so the four digits of one
//     slice form one 32-bit word and a warp stores 128 contiguous bytes per slice;
//   * NSL is a template parameter: every field offset is an immediate;
//   * rounding to the fixed-point integer and adding the field bias is ONE fma with the constant
//     1.5 * 2^52 + B (B = 64 in every 7-bit field): the low mantissa bits of the result are q + B
//     (NSL <= 7: |q + B| < 2^51; 8 slices need 56 bits and keep cvt.rni.s64);
//   * bytes are packed with PRMT, and  ((w & 0x7f7f7f7f) + 0x40404040) ^ 0x80808080  turns the four biased
//     fields d + 64 into the int8 digits d  (no carry can cross a byte: d + 128 <= 191);
//   * radix-256 digits (RB = 8) are whole bytes of q + B (B = 128 in every byte): PRMT and one XOR, see
//     ozaki_store_slices256.
template <int NSL>
__device__ __forceinline__ void ozaki_bits(double c, double mul, double magic, uint32_t& lo, uint32_t& hi) {
  if (NSL <= 7) {
    const long long b = __double_as_longlong(fma(c, mul, magic));
    lo = (uint32_t)b;
    hi = (uint32_t)((unsigned long long)b >> 32);
  } else {
    const unsigned long long B = (0x0102040810204081ull << 6) & ((1ull << (7 * NSL)) - 1ull);
    const unsigned long long qb = (unsigned long long)__double2ll_rn(c * mul) + B;
    lo = (uint32_t)qb;
    hi = (uint32_t)(qb >> 32);
  }
}

template <int OFF>
__device__ __forceinline__ uint32_t ozaki_field(uint32_t lo, uint32_t hi) {  // low 7 bits = field at bit OFF
  if constexpr (OFF == 0)
    return lo;
  else if constexpr (OFF + 7 <= 32)
    return lo >> OFF;
  else if constexpr (OFF >= 32)
    return hi >> (OFF - 32);
  else
    return __funnelshift_r(lo, hi, OFF);
}

template <int NSL, int SL>
__device__ __forceinline__ void ozaki_store_slices(const uint32_t (&lo)[4], const uint32_t (&hi)[4], int8_t* o,
                                                   int64_t slice_stride) {
  if constexpr (SL < NSL) {
    constexpr int OFF = 7 * (NSL - 1 - SL);
    const uint32_t w01 = __byte_perm(ozaki_field<OFF>(lo[0], hi[0]), ozaki_field<OFF>(lo[1], hi[1]), 0x0040);
    const uint32_t w23 = __byte_perm(ozaki_field<OFF>(lo[2], hi[2]), ozaki_field<OFF>(lo[3], hi[3]), 0x0040);
    const uint32_t w = __byte_perm(w01, w23, 0x5410);
    *reinterpret_cast<uint32_t*>(o + SL * slice_stride) = ((w & 0x7f7f7f7fu) + 0x40404040u) ^ 0x80808080u;
    ozaki_store_slices<NSL, SL + 1>(lo, hi, o, slice_stride);
  }
}

// Radix-256 digits (NSL <= 6, the magic constant then carries B = 0x80 in every byte): the digit of slice SL is byte
// 8 (NSL-1-SL) of q + B, so PRMT gathers it from the four genes as it stands and  ^ 0x80808080  turns the biased
// bytes d + 128 into the int8 digits d.  No masks, no field shifts.
template <int NSL, int SL>
__device__ __forceinline__ void ozaki_store_slices256(const uint32_t (&lo)[4], const uint32_t (&hi)[4], int8_t* o,
                                                      int64_t slice_stride) {
  if constexpr (SL < NSL) {
    constexpr int BYTE = NSL - 1 - SL;  // byte of the 64-bit q + B
    constexpr uint32_t SEL = (uint32_t)(BYTE & 3) | ((uint32_t)(4 + (BYTE & 3)) << 4);
    const uint32_t w01 = BYTE < 4 ? __byte_perm(lo[0], lo[1], SEL) : __byte_perm(hi[0], hi[1], SEL);
    const uint32_t w23 = BYTE < 4 ? __byte_perm(lo[2], lo[3], SEL) : __byte_perm(hi[2], hi[3], SEL);
    *reinterpret_cast<uint32_t*>(o + SL * slice_stride) = __byte_perm(w01, w23, 0x5410) ^ 0x80808080u;
    ozaki_store_slices256<NSL, SL + 1>(lo, hi, o, slice_stride);
  }
}

// T threads per row, NV4 sweeps of 4 genes per thread (row capacity 4*T*NV4 >= ldk8), digit output only.
// vec: X is 32-byte aligned and ldx a multiple of 4 (256-bit loads legal).
// Everything of the digit pass behind the load: v holds the row slice of this thread (4 consecutive genes per k),
// sum its partial sum.  Shared by the one-row-per-launch-CTA kernel and the persistent streaming kernel below.
template <int T, int NV4, int NSL, int RB>
__device__ __forceinline__ void digits_row_finish(double (&v)[NV4][4], double sum, int t, int64_t row, bool live, int G,
                                                  double* __restrict__ norms, int* __restrict__ flags,
                                                  const mcd_ozaki_out& oz, double* red) {
  constexpr int BLOCK = 512;
  sum = group_sum<T, BLOCK>(sum, red);
  const double mean = sum / (double)G;

  double ss = 0.0, amax = 0.0;
#pragma unroll
  for (int k = 0; k < NV4; ++k) {
    const int e = 4 * (t + k * T);
    if (e + 3 < G) {  // whole group inside the row: no per-gene masks
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const double c = v[k][i] - mean;
        v[k][i] = c;
        ss = fma(c, c, ss);
        amax = (fabs(c) > amax) ? fabs(c) : amax;  // non-finite rows are flagged below: no NaN handling needed
      }
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const double c = (e + i < G) ? v[k][i] - mean : 0.0;
        v[k][i] = c;
        ss = fma(c, c, ss);
        amax = (fabs(c) > amax) ? fabs(c) : amax;
      }
    }
  }
  ss = group_sum<T, BLOCK>(ss, red);
  if (flat_row(ss, mean, G)) ss = 0.0;  // zero-variance cell: norm 0 -> mul 0 -> all digits zero
  amax = group_max<T, BLOCK>(amax, red);
  if (!live) return;
  const double nrm = sqrt(ss);
  if (t == 0) {
    norms[row] = nrm;
    if (!isfinite(sum) || !isfinite(ss)) atomicOr(flags, 1);
  }
  // unit row u = c / nrm scaled by 2^e so that max|u| * 2^e lies in [0.25, 0.5)
  const double inv = (nrm > 0.0 && isfinite(nrm)) ? 1.0 / nrm : 0.0;
  const double umax = amax * inv;
  int ex = 0;
  if (umax > 0.0 && isfinite(umax)) (void)frexp(umax, &ex);
  const int sh = -ex - 1;
  if (t == 0) oz.scale[row] = scalbn(1.0, -sh);
  static_assert(RB == 7 || (RB == 8 && NSL <= 6), "radix-256 digits need B < 2^51");
  const double mul = inv * scalbn(1.0, sh + RB * NSL - 1);
  const unsigned long long B = RB == 8 ? 0x8080808080808080ull >> (64 - 8 * NSL)
                                       : (0x0102040810204081ull << 6) & ((1ull << (7 * NSL)) - 1ull);
  const double magic = 6755399441055744.0 + (double)B;  // 1.5 * 2^52 + B, exact (B < 2^51 when NSL <= 7)
  int8_t* o = oz.digits + row * oz.ldk8 + 4 * t;
  const int ldk8 = (int)oz.ldk8;
#pragma unroll
  for (int k = 0; k < NV4; ++k) {
    const int g = 4 * (t + k * T);
    if (g < ldk8) {  // genes in [G, ldk8) are zero digits (c = 0 there)
      uint32_t lo[4], hi[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) ozaki_bits<NSL>(v[k][i], mul, magic, lo[i], hi[i]);
      if constexpr (RB == 8)
        ozaki_store_slices256<NSL, 0>(lo, hi, o + 4 * k * T, oz.slice_stride);
      else
        ozaki_store_slices<NSL, 0>(lo, hi, o + 4 * k * T, oz.slice_stride);
    }
  }
}


template <int T, int NV4, int NSL, int RB>
__global__ void __launch_bounds__(512, 1)
standardize_digits(const double* __restrict__ X, const int* __restrict__ gidx, int64_t ncells, int G, int64_t ldx,
                   int vec, double* __restrict__ norms, int* __restrict__ flags, const mcd_ozaki_out oz) {
  constexpr int BLOCK = 512;
  constexpr int ROWS = BLOCK / T;
  __shared__ double red[BLOCK / 32];
  const int t = threadIdx.x % T;
  const int64_t row = (int64_t)blockIdx.x * ROWS + threadIdx.x / T;
  const bool live = row < ncells;
  const double* x = X + (live ? row : 0) * ldx;

  double v[NV4][4];
  double sum = 0.0;
#pragma unroll
  for (int k = 0; k < NV4; ++k) {
    const int e = 4 * (t + k * T);
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    if (live && e < G) {
      if (gidx != nullptr) {
        a0 = __ldg(x + __ldg(gidx + e));
        if (e + 1 < G) a1 = __ldg(x + __ldg(gidx + e + 1));
        if (e + 2 < G) a2 = __ldg(x + __ldg(gidx + e + 2));
        if (e + 3 < G) a3 = __ldg(x + __ldg(gidx + e + 3));
      } else if (vec && e + 3 < G) {
        asm volatile("ld.global.cs.v4.f64 {%0, %1, %2, %3}, [%4];"
                     : "=d"(a0), "=d"(a1), "=d"(a2), "=d"(a3)
                     : "l"(x + e));
      } else {
        a0 = __ldcs(x + e);
        if (e + 1 < G) a1 = __ldcs(x + e + 1);
        if (e + 2 < G) a2 = __ldcs(x + e + 2);
        if (e + 3 < G) a3 = __ldcs(x + e + 3);
      }
    }
    v[k][0] = a0;
    v[k][1] = a1;
    v[k][2] = a2;
    v[k][3] = a3;
    sum += (a0 + a1) + (a2 + a3);
  }
  digits_row_finish<T, NV4, NSL, RB>(v, sum, t, row, live, G, norms, flags, oz, red);
}

// Persistent streaming form for long rows (T = 512: one row per CTA at a time).  The one-row-per-CTA kernel above
// runs load -> reduce -> store strictly one after the other on an SM (one 512-thread CTA of 128 registers is all
// that fits), so HBM reads pause while a row is being reduced and stored: 73 % of the copy peak at C5.  Here a CTA
// loops over rows and the NEXT row is already on its way into shared memory -- one 1-D bulk copy (TMA,
// cp.async.bulk) of the whole row, completion on an mbarrier -- while the current row is reduced, turned into digit
// slices and stored from registers.  Same thread <-> gene mapping and the same arithmetic as above: bit-identical.
// Needs X 16-byte aligned, ldx and G even (bulk copies move multiples of 16 bytes) and no gene gather.
template <int NV4, int NSL, int RB>
__global__ void __launch_bounds__(512, 1)
standardize_digits_stream(const double* __restrict__ X, int64_t ncells, int G, int64_t ldx, double* __restrict__ norms,
                          int* __restrict__ flags, const mcd_ozaki_out oz) {
  constexpr int T = 512;
  extern __shared__ __align__(128) unsigned char k1_smem[];
  double* buf = reinterpret_cast<double*>(k1_smem);  // [G] the row in flight
  __shared__ double red[T / 32];
  __shared__ __align__(8) unsigned long long bar;
  const int t = threadIdx.x;
  const uint32_t bar_a = (uint32_t)__cvta_generic_to_shared(&bar);
  const uint32_t buf_a = (uint32_t)__cvta_generic_to_shared(buf);
  const uint32_t bytes = (uint32_t)G * 8u;
  int64_t row = blockIdx.x;
  if (t == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (row < ncells) {
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(bytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(buf_a),
                   "l"(X + row * ldx), "r"(bytes), "r"(bar_a)
                   : "memory");
    }
  }
  __syncthreads();
  uint32_t phase = 0;
  for (; row < ncells; row += gridDim.x) {
    // wait for the row
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "K1_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra K1_DONE;\n"
        "bra K1_WAIT;\n"
        "K1_DONE:\n"
        "}\n" ::"r"(bar_a),
        "r"(phase)
        : "memory");
    phase ^= 1u;
    double v[NV4][4];
    double sum = 0.0;
#pragma unroll
    for (int k = 0; k < NV4; ++k) {
      const int e = 4 * (t + k * T);
      double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
      if (e + 3 < G) {
        const double2 lo = *reinterpret_cast<const double2*>(buf + e);
        const double2 hi = *reinterpret_cast<const double2*>(buf + e + 2);
        a0 = lo.x, a1 = lo.y, a2 = hi.x, a3 = hi.y;
      } else if (e < G) {
        a0 = buf[e];
        if (e + 1 < G) a1 = buf[e + 1];
        if (e + 2 < G) a2 = buf[e + 2];
      }
      v[k][0] = a0;
      v[k][1] = a1;
      v[k][2] = a2;
      v[k][3] = a3;
      sum += (a0 + a1) + (a2 + a3);
    }
    __syncthreads();  // every thread has its slice: the buffer is free for the next row
    const int64_t nxt = row + gridDim.x;
    if (t == 0 && nxt < ncells) {
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(bytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(buf_a),
                   "l"(X + nxt * ldx), "r"(bytes), "r"(bar_a)
                   : "memory");
    }
    digits_row_finish<T, NV4, NSL, RB>(v, sum, t, row, true, G, norms, flags, oz, red);
  }
}

template <int T, int NV4, int NSL, int RB>
int launch_digits_fmt(mcd_context* h, const double* X, const int* gidx, int64_t ncells, int G, int64_t ldx, double* norms,
                      const mcd_ozaki_out& oz) {
  constexpr int ROWS = 512 / T;
  const unsigned grid = (unsigned)((ncells + ROWS - 1) / ROWS);
  const int vec = ((reinterpret_cast<uintptr_t>(X) & 31) == 0) && ((ldx & 3) == 0);
  if (T == 512 && gidx == nullptr && !h->opt.k1_no_stream && (reinterpret_cast<uintptr_t>(X) & 15) == 0 && (ldx & 1) == 0 &&
      (G & 1) == 0 && ncells >= 2 * (int64_t)h->sm_count) {
    // long rows, plenty of them: persistent CTAs with the next row prefetched by a bulk copy
    const size_t smem = ((size_t)G * 8 + 127) / 128 * 128;
    const unsigned pgrid = (unsigned)h->sm_count;
    MCD_CUDA(h, cudaFuncSetAttribute(standardize_digits_stream<NV4, NSL, RB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)smem));
    standardize_digits_stream<NV4, NSL, RB><<<pgrid, 512, smem, h->stream>>>(X, ncells, G, ldx, norms, h->d_flags, oz);
    MCD_LAUNCH_CHECK(h, "standardize_digits_stream");
    return MCD_OK;
  }
  standardize_digits<T, NV4, NSL, RB><<<grid, 512, 0, h->stream>>>(X, gidx, ncells, G, ldx, vec, norms, h->d_flags, oz);
  MCD_LAUNCH_CHECK(h, "standardize_digits");
  return MCD_OK;
}

// the digit formats the fast path is compiled for: radix 128 x 6 or 8 slices, radix 256 x 5 (mcd_ozaki_format)
bool fast_digit_format(const mcd_ozaki_out& oz) {
  return (oz.rb == 7 && (oz.nsl == 6 || oz.nsl == 8)) || (oz.rb == 8 && oz.nsl == 5);
}

template <int T, int NV4>
int launch_digits(mcd_context* h, const double* X, const int* gidx, int64_t ncells, int G, int64_t ldx, double* norms,
                  const mcd_ozaki_out& oz) {
  if (oz.rb == 8) return launch_digits_fmt<T, NV4, 5, 8>(h, X, gidx, ncells, G, ldx, norms, oz);
  if (oz.nsl == 6) return launch_digits_fmt<T, NV4, 6, 7>(h, X, gidx, ncells, G, ldx, norms, oz);
  return launch_digits_fmt<T, NV4, 8, 7>(h, X, gidx, ncells, G, ldx, norms, oz);
}

// Rows longer than the register-resident capacity: one 512-thread block per row, three sweeps
// (the row stays L2-resident between sweeps; declared as a 3-read variant in DESIGN.md).
template <int RB>
__global__ void __launch_bounds__(512)
standardize_rows_long(const double* __restrict__ X, const int* __restrict__ gidx, int64_t ncells, int64_t G,
                      int64_t ldx, double* __restrict__ Y,
                      int64_t ldk, uint16_t* __restrict__ S, uint16_t* __restrict__ S_lo, int64_t ldk16,
                      double* __restrict__ norms, int* __restrict__ flags, const mcd_ozaki_out oz) {
  __shared__ double red[16];
  const int64_t row = blockIdx.x;
  const double* x = X + row * ldx;
  auto at = [&](int64_t e) { return gidx != nullptr ? x[gidx[e]] : x[e]; };
  double sum = 0.0;
  for (int64_t e = threadIdx.x; e < G; e += 512) sum += at(e);
  sum = group_sum<512, 512>(sum, red);
  const double mean = sum / (double)G;
  double ss = 0.0;
  for (int64_t e = threadIdx.x; e < G; e += 512) {
    const double c = at(e) - mean;
    ss += c * c;
  }
  ss = group_sum<512, 512>(ss, red);
  const bool flat = flat_row(ss, mean, (int)(G < 2147483647 ? G : 2147483647));
  if (flat) ss = 0.0;
  const double nrm = sqrt(ss);
  if (threadIdx.x == 0) {
    norms[row] = nrm;
    if (!isfinite(sum) || !isfinite(ss)) atomicOr(flags, 1);
  }
  const double inv = nrm > 0.0 ? 1.0 / nrm : 0.0;
  if (Y != nullptr) {
    double* y = Y + row * ldk;
    for (int64_t e = threadIdx.x; e < ldk; e += 512) y[e] = (e < G && !flat) ? at(e) - mean : 0.0;
  }
  if (oz.digits != nullptr) {
    double amax = 0.0;
    for (int64_t e = threadIdx.x; e < G; e += 512) amax = fmax(amax, fabs(at(e) - mean));
    amax = group_max<512, 512>(amax, red);
    const double inv1 = (nrm > 0.0 && isfinite(nrm)) ? 1.0 / nrm : 0.0;
    const double umax = amax * inv1;
    int ex = 0;
    if (umax > 0.0 && isfinite(umax)) (void)frexp(umax, &ex);
    const int sh = -ex - 1;
    if (threadIdx.x == 0) oz.scale[row] = scalbn(1.0, -sh);
    const double mul = inv1 * scalbn(1.0, sh + RB * oz.nsl - 1);
    int8_t* o = oz.digits + row * oz.ldk8;
    for (int64_t e = threadIdx.x; e < oz.ldk8; e += 512) {
      int d[MCD_OZAKI_MAX_SLICES];
      ozaki_digits_of<RB>(e < G ? (at(e) - mean) * mul : 0.0, oz.nsl, d);
#pragma unroll
      for (int sl = 0; sl < MCD_OZAKI_MAX_SLICES; ++sl)
        if (sl < oz.nsl) o[sl * oz.slice_stride + e] = (int8_t)d[sl];
    }
  }
  if (S != nullptr) {
    uint16_t* s0 = S + row * ldk16;
    uint16_t* s1 = S_lo + row * ldk16;
    for (int64_t e = threadIdx.x; e < ldk16; e += 512) {
      uint16_t a0 = 0, a1 = 0;
      if (e < G) split_fp16x2((at(e) - mean) * inv, a0, a1);
      s0[e] = a0;
      s1[e] = a1;
    }
  }
}

template <int T, int NV>
int launch_t(mcd_context* h, bool vec, const double* X, const int* gidx, int64_t ncells, int G, int64_t ldx, double* Y,
             int64_t ldk,
             uint16_t* S, uint16_t* S_lo, int64_t ldk16, double* norms, const mcd_ozaki_out& oz) {
  constexpr int BLOCK = (T > 512 ? T : 512);
  constexpr int ROWS = BLOCK / T;
  const int64_t grid = (ncells + ROWS - 1) / ROWS;
  // radix-256 digits come here only off the fast path (mcd_launch_standardize): scalar loads suffice
  if (oz.digits != nullptr && oz.rb == 8)
    standardize_rows<T, NV, false, 8><<<(unsigned)grid, BLOCK, 0, h->stream>>>(X, gidx, ncells, G, ldx, Y, ldk, S, S_lo,
                                                                              ldk16, norms, h->d_flags, oz);
  else if (vec)
    standardize_rows<T, NV, true, 7><<<(unsigned)grid, BLOCK, 0, h->stream>>>(X, gidx, ncells, G, ldx, Y, ldk, S, S_lo,
                                                                             ldk16, norms, h->d_flags, oz);
  else
    standardize_rows<T, NV, false, 7><<<(unsigned)grid, BLOCK, 0, h->stream>>>(X, gidx, ncells, G, ldx, Y, ldk, S, S_lo,
                                                                              ldk16, norms, h->d_flags, oz);
  MCD_LAUNCH_CHECK(h, "standardize_rows");
  return MCD_OK;
}

}  // namespace

int mcd_launch_standardize(mcd_context* h, const double* X, int64_t ncells, int64_t G, int64_t ldx, double* centred,
                           int64_t ldk, uint16_t* slices, uint16_t* slices_lo, int64_t ldk16, double* norms,
                           const int* gidx, const mcd_ozaki_out* ozaki) {
  if (ncells == 0) return MCD_OK;
  mcd_ozaki_out oz{};
  if (ozaki != nullptr) oz = *ozaki;
  const bool vec = ((reinterpret_cast<uintptr_t>(X) & 15) == 0) && ((ldx & 1) == 0);
  const int g = (int)G;
  if (oz.digits != nullptr && centred == nullptr && slices == nullptr && fast_digit_format(oz) &&
      oz.ldk8 <= 24576 && (oz.ldk8 & 3) == 0 && (oz.slice_stride & 3) == 0 &&
      (reinterpret_cast<uintptr_t>(oz.digits) & 3) == 0 && !h->opt.k1_generic) {
    const int64_t cap = oz.ldk8;  // the sweeps also write the zero padding up to ldk8
    if (cap <= 256) return launch_digits<32, 2>(h, X, gidx, ncells, g, ldx, norms, oz);
    if (cap <= 1024) return launch_digits<128, 2>(h, X, gidx, ncells, g, ldx, norms, oz);
    if (cap <= 4096) return launch_digits<512, 2>(h, X, gidx, ncells, g, ldx, norms, oz);
    if (cap <= 8192) return launch_digits<512, 4>(h, X, gidx, ncells, g, ldx, norms, oz);
    if (cap <= 12288) return launch_digits<512, 6>(h, X, gidx, ncells, g, ldx, norms, oz);
    if (cap <= 16384) return launch_digits<512, 8>(h, X, gidx, ncells, g, ldx, norms, oz);
    if (cap <= 20480) return launch_digits<512, 10>(h, X, gidx, ncells, g, ldx, norms, oz);
    return launch_digits<512, 12>(h, X, gidx, ncells, g, ldx, norms, oz);
  }
  if (G <= 256) return launch_t<32, 4>(h, vec, X, gidx, ncells, g, ldx, centred, ldk, slices, slices_lo, ldk16, norms, oz);
  if (G <= 1024) return launch_t<128, 4>(h, vec, X, gidx, ncells, g, ldx, centred, ldk, slices, slices_lo, ldk16, norms, oz);
  if (G <= 4096) return launch_t<512, 4>(h, vec, X, gidx, ncells, g, ldx, centred, ldk, slices, slices_lo, ldk16, norms, oz);
  if (G <= 8192) return launch_t<512, 8>(h, vec, X, gidx, ncells, g, ldx, centred, ldk, slices, slices_lo, ldk16, norms, oz);
  if (G <= 12288) return launch_t<512, 12>(h, vec, X, gidx, ncells, g, ldx, centred, ldk, slices, slices_lo, ldk16, norms, oz);
  if (G <= 16384) return launch_t<512, 16>(h, vec, X, gidx, ncells, g, ldx, centred, ldk, slices, slices_lo, ldk16, norms, oz);
  if (G <= 20480) return launch_t<512, 20>(h, vec, X, gidx, ncells, g, ldx, centred, ldk, slices, slices_lo, ldk16, norms, oz);
  if (G <= 24576) return launch_t<512, 24>(h, vec, X, gidx, ncells, g, ldx, centred, ldk, slices, slices_lo, ldk16, norms, oz);
  if (oz.digits != nullptr && oz.rb == 8)
    standardize_rows_long<8><<<(unsigned)ncells, 512, 0, h->stream>>>(X, gidx, ncells, G, ldx, centred, ldk, slices,
                                                                     slices_lo, ldk16, norms, h->d_flags, oz);
  else
    standardize_rows_long<7><<<(unsigned)ncells, 512, 0, h->stream>>>(X, gidx, ncells, G, ldx, centred, ldk, slices,
                                                                     slices_lo, ldk16, norms, h->d_flags, oz);
  MCD_LAUNCH_CHECK(h, "standardize_rows_long");
  return MCD_OK;
}
