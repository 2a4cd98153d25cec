// K2c -- FP64-equivalent correlation contraction on the int8 tcgen05 tensor cores (sm_100a).
//
// Replaces the RNA x DNA double loop of the reference (src/MaCroDNA/macrodna.py:103-107) with an
// error-free ("Ozaki scheme") integer GEMM.  K1 writes every unit-norm centred row as nsl balanced
// digit slices of rb bits (int8, standardize.cu::ozaki_digits / ozaki_digits256):
//     x = 2^-(rb nsl - 1) * sum_t d_t 2^(rb (nsl-1-t)),   d_t in [-64, 63] (rb = 7) or [-128, 127] (rb = 8).
// A dot product then splits into digit-slice products that the tensor core evaluates EXACTLY
// (int8 x int8 -> int32, no rounding anywhere):
//     <x, y> = 2^(2 - 2 rb) * sum_g 2^(-rb g) ACC_g,    ACC_g = sum_{t+t'=g} sum_k d_t[k] d'_t'[k],
// truncated at g < nsl (the dropped groups are below the digit resolution).  All products of one
// significance group g share ONE int32 accumulator in TMEM (the caller keeps |ACC_g| < 2^31:
// mcd_ozaki_exact), the FP64 combination of the groups happens once per output in the epilogue.
// Radix 128: nsl = 6 (21 products) gives ~1e-12 absolute, nsl = 8 (36 products) is at the level of an FP64
// GEMM's own rounding.  Radix 256: nsl = 5 (15 products) carries 40 bits, ~5e-12 absolute.
//
// Structure: persistent kernel, CTA PAIRS (cluster of 2, tcgen05 cta_group::2) on 256 x 256 output tiles:
//   * each CTA stages 128 rows of the RNA tile and 128 rows of the DNA tile per digit slice (8 KB tiles,
//     K-major, 64-byte swizzle) with cp.async.bulk.tensor.3d (.cta_group::2: both CTAs' loads complete on
//     the LEADER's mbarrier); ring of 12 "units" (unit = A_t + B_t of one k-block of 64 genes);
//   * the leader CTA's warp 1 issues tcgen05.mma.cta_group::2.kind::i8 (M256 N256 K32): each SM multiplies
//     its own 128 RNA rows with all 256 DNA columns, reading half of the DNA operand from its peer's shared
//     memory -- per MMA each SM's smem port moves 8 KB per 128 clk instead of 12 KB (cta_group::1);
//   * TMEM holds exactly two 256-column int32 accumulators per CTA (512 columns), so a tile is worked
//     in ceil(nsl/2) PASSES over the genes, pass p accumulating the groups 2p and 2p+1 (least significant
//     pass first); after each pass the epilogue warps of both CTAs drain the accumulators, fold them into
//     the FP64 partial sum kept in C, and the last pass applies the reference's scaling
//     nn / (1e-10 + nn), nn = |r_i| |d_j| (macrodna.py:25 on unit vectors) and writes C and C^T.
// Pass p needs the digit slices 0 .. 2p+1 of both operands, so the three passes of nsl = 6 stream 4 + 8 + 12
// slice tiles per k-block for 3 + 7 + 11 products.
#include <cuda.h>

#include <cstdlib>
#include <type_traits>

#include "mcd_internal.cuh"

namespace {

constexpr int TM = 256;                 // pair-tile rows (128 per CTA)
constexpr int TN = 256;                 // pair-tile columns (each CTA stages 128 of them)
constexpr int HALF = 128;
constexpr int BK = 64;                  // int8 elements = 64 bytes = one swizzle-64B row
constexpr int UMMA_K = 32;
constexpr int TILE_BYTES = HALF * BK;   // 8 KB: one digit slice of one operand half
constexpr int UNIT_BYTES = 2 * TILE_BYTES;
#ifndef MCD_OZ_UNITS
#define MCD_OZ_UNITS 12
#endif
#ifndef MCD_OZ_BAND
#define MCD_OZ_BAND 6
#endif
constexpr int UNITS = MCD_OZ_UNITS;
constexpr int SMEM_BYTES = UNITS * UNIT_BYTES + 1024 /*align*/ + 512 /*barriers*/;
constexpr int NUM_THREADS = 320;        // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue
constexpr int EPI_WARPS = 8;
constexpr int TMEM_COLS = 512;
constexpr int BAND_M = MCD_OZ_BAND;

// instruction descriptor, kind::i8: D = S32 (bits 4-5 = 2), A = B = signed int8 (bits 7-9, 10-12 = 1),
// both K-major, N >> 3 at bit 17, M >> 4 at bit 24
constexpr uint32_t IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(TN >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// one elected lane of a converged warp arrives (the producer warp runs warp-uniformly, see umma_i8_2cta_pred)
__device__ __forceinline__ void mbar_expect_tx_elect(uint32_t bar, uint32_t bytes) {
  asm volatile(
      "{\n"
      ".reg .pred q;\n"
      "elect.sync _|q, 0xffffffff;\n"
      "@q mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n"
      "}\n" ::"r"(bar),
      "r"(bytes)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "OZ_WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra OZ_WAIT_DONE;\n"
      "bra OZ_WAIT_LOOP;\n"
      "OZ_WAIT_DONE:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_smem_addr, uint32_t cta) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(cta));
  return r;
}
// 3-D tile load (genes, rows, slice); the completion bytes go to `bar`, a shared::cluster address that may
// belong to the peer CTA of the pair (.cta_group::2)
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int x, int y, int z) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], "
      "[%2];" ::"r"(dst),
      "l"(map), "r"(bar), "r"(x), "r"(y), "r"(z)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_elect(uint32_t dst, const CUtensorMap* map, uint32_t bar, int x, int y,
                                                  int z) {
  asm volatile(
      "{\n"
      ".reg .pred q;\n"
      "elect.sync _|q, 0xffffffff;\n"
      "@q cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
      "%4, %5}], [%2];\n"
      "}\n" ::"r"(dst),
      "l"(map), "r"(bar), "r"(x), "r"(y), "r"(z)
      : "memory");
}
// K-major operand tile, 64-byte swizzle: rows of 64 B, 8-row groups 512 B apart (SBO), descriptor version 1
// (Blackwell), layout type 4 = SWIZZLE_64B.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t addr) {
  uint64_t d = 0;
  d |= (uint64_t)((addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;           // leading byte offset (unused: one MMA's K extent stays inside a swizzle row)
  d |= (uint64_t)(512 >> 4) << 32;  // stride byte offset
  d |= (uint64_t)1 << 46;           // version
  d |= (uint64_t)4 << 61;           // SWIZZLE_64B
  return d;
}
__device__ __forceinline__ void umma_i8_2cta(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(da), "l"(db), "r"(idesc), "r"(accum)
      : "memory");
}
// arrives (once the MMAs issued so far have retired) on the barrier at this smem offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
      "h"((uint16_t)3)
      : "memory");
}
// The MMA warp runs its loops WARP-UNIFORMLY (all 32 lanes: ring slots, phases and descriptors then live in uniform
// registers) and only the tcgen05 instructions themselves are predicated on one elected lane (elect.sync).  Inside an
// `if (lane == 0)` region the compiler cannot prove the descriptors uniform and wraps every UTCIMMA in an
// ELECT / R2UR.BROADCAST waterfall loop (~20 instructions + local-memory slot lookups per MMA).
__device__ __forceinline__ void umma_i8_2cta_pred(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc,
                                                  uint32_t accum) {
  asm volatile(
      "{\n"
      ".reg .pred p, q;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "elect.sync _|q, 0xffffffff;\n"
      "@q tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(da), "l"(db), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void umma_commit_pair_pred(uint32_t bar) {
  asm volatile(
      "{\n"
      ".reg .pred q;\n"
      "elect.sync _|q, 0xffffffff;\n"
      "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n"
      "}\n" ::"r"(bar),
      "h"((uint16_t)3)
      : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  __syncwarp();
  asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}

// Tile order: bands of BAND_M tile-rows, column-major inside a band, so the ~74 pair tiles in flight touch
// ~8 RNA panels x ~9 DNA panels and advance through the genes together (operand panels are read from HBM about
// once per wave and served to the other pairs from L2).
__device__ __forceinline__ void decode_tile(int t, int tiles_m, int tiles_n, int& tm, int& tn) {
  const int per_band = BAND_M * tiles_n;
  const int band = t / per_band;
  const int rem = t - band * per_band;
  const int hb = min(BAND_M, tiles_m - band * BAND_M);
  tn = rem / hb;
  tm = band * BAND_M + (rem - tn * hb);
}

// Order in which one pass loads the digit-slice units of a k-block, and the MMA schedule that goes with it.
// A pass accumulates the significance groups g_lo = nload - ng (and g_lo + 1 when ng = 2) from the units
// 0 .. nload-1; group g is the sum of the products (A unit t) x (B unit g - t).
//   mode 0: units in index order, the whole k-block is waited for, multiplied group by group and freed together.
//   mode 1: units walked from both ends (step a brings a, gh - a and, with two groups, gh - a - 1): every product is
//           issued at the first step that has both its units and a unit goes back to the producer as soon as its
//           last product is issued, while the rest of the k-block is still being multiplied -- the 12-unit ring
//           then covers ~1.7 k-blocks of load latency in the heaviest pass (6 units per k-block) instead of 1.
// Evaluated at compile time: the issuer is fully unrolled per (nload, ng, mode).
struct PassPlan {
  int nunits = 0, nsteps = 0, nprod = 0;
  int ord[8] = {};  // load order: ord[k] = unit id
  int pos[8] = {};  // inverse
  unsigned wait_mask[8] = {};  // per step: units that must have landed (not waited for before)
  unsigned free_mask[8] = {};  // per step: units whose last product was issued in this step
  int step_end[8] = {};        // per step: end index into prod_*
  int prod_a[16] = {}, prod_b[16] = {}, prod_g[16] = {};  // products: A unit, B unit, accumulator (0 / 1)
  int prod_first[16] = {};                                // first product of its accumulator in the k-block
};

__host__ __device__ constexpr PassPlan make_pass_plan(int nload, int ng, int mode) {
  PassPlan pl;
  const int gh = nload - 1;
  const int gl = nload - ng;
  const bool two = ng == 2;
  pl.nunits = nload;
  unsigned seen = 0;
  int n = 0;
  for (int a = 0; a <= gh; ++a) {
    const int cand[3] = {a, mode ? gh - a : -1, (mode && two) ? gh - a - 1 : -1};
    for (int c = 0; c < 3; ++c) {
      const int x = cand[c];
      if (x >= 0 && x <= gh && !((seen >> x) & 1u)) {
        seen |= 1u << x;
        pl.pos[x] = n;
        pl.ord[n++] = x;
      }
    }
  }
  unsigned have = 0, freed = 0, started = 0;
  unsigned done[2] = {0, 0};
  int np = 0, ns = 0;
  const int total = (gh + 1) + (two ? gl + 1 : 0);
  for (int a = 0; a <= gh && np < total; ++a) {
    unsigned set = have;
    for (int x = 0; x <= gh; ++x)
      if (mode == 0 || x <= a || x >= gh - a - (two ? 1 : 0)) set |= 1u << x;
    pl.wait_mask[ns] = set & ~have;
    have = set;
    for (int gi = 0; gi < ng; ++gi) {
      const int g = gl + gi;
      for (int t = 0; t <= g; ++t) {
        if (!((done[gi] >> t) & 1u) && ((have >> t) & 1u) && ((have >> (g - t)) & 1u)) {
          done[gi] |= 1u << t;
          pl.prod_a[np] = t;
          pl.prod_b[np] = g - t;
          pl.prod_g[np] = gi;
          pl.prod_first[np] = ((started >> gi) & 1u) ? 0 : 1;
          started |= 1u << gi;
          ++np;
        }
      }
    }
    unsigned fm = 0;  // a unit is finished once every product it takes part in has been issued
    for (int x = 0; x <= gh; ++x) {
      if ((freed >> x) & 1u) continue;
      bool fin = true;
      for (int gi = 0; gi < ng; ++gi) {
        const int g = gl + gi;
        if (g - x >= 0) {
          if (!((done[gi] >> x) & 1u)) fin = false;        // product (x, g - x)
          if (!((done[gi] >> (g - x)) & 1u)) fin = false;  // product (g - x, x)
        }
      }
      if (fin) fm |= 1u << x;
    }
    freed |= fm;
    pl.free_mask[ns] = fm;
    pl.step_end[ns] = np;
    ++ns;
  }
  pl.nsteps = ns;
  pl.nprod = np;
  return pl;
}

template <int NLOAD, int NG, int MODE>
__host__ __device__ constexpr uint32_t packed_load_order() {
  constexpr PassPlan pl = make_pass_plan(NLOAD, NG, MODE);
  uint32_t r = 0;
  for (int k = 0; k < NLOAD; ++k) r |= (uint32_t)pl.ord[k] << (4 * k);
  return r;
}
// nibble k = the unit loaded k-th in a k-block of this pass (the producer's view of the plan)
__device__ __forceinline__ uint32_t load_order(int nload, int ng, int mode) {
  if (mode == 0) return 0x76543210u;
  switch (nload * 2 + ng) {
    case 2 * 2 + 2: { constexpr uint32_t o = packed_load_order<2, 2, 1>(); return o; }
    case 4 * 2 + 2: { constexpr uint32_t o = packed_load_order<4, 2, 1>(); return o; }
    case 6 * 2 + 2: { constexpr uint32_t o = packed_load_order<6, 2, 1>(); return o; }
    case 8 * 2 + 2: { constexpr uint32_t o = packed_load_order<8, 2, 1>(); return o; }
    case 3 * 2 + 1: { constexpr uint32_t o = packed_load_order<3, 1, 1>(); return o; }
    case 5 * 2 + 1: { constexpr uint32_t o = packed_load_order<5, 1, 1>(); return o; }
    default: { constexpr uint32_t o = packed_load_order<7, 1, 1>(); return o; }
  }
}

template <int NLOAD, int NG, int MODE>
struct PlanOf {
  static constexpr PassPlan pl = make_pass_plan(NLOAD, NG, MODE);
};
// compile-time loop: every index into the plan is a constant expression (a run-time index would force the plan
// into local memory)
template <int B, int E, class F>
__device__ __forceinline__ void static_for(F&& f) {
  if constexpr (B < E) {
    f(std::integral_constant<int, B>{});
    static_for<B + 1, E>(f);
  }
}

// One pass of the MMA issuer over all k-blocks, fully unrolled -- the ring slot of every unit is a register.
template <int NLOAD, int NG, int MODE>
__device__ __forceinline__ void mma_pass(const int num_kb, int& u, uint32_t& phase, const uint32_t smem_base,
                                         const uint32_t tmem_base, const uint32_t full_bar, const uint32_t empty_bar) {
  using P = PlanOf<NLOAD, NG, MODE>;
#pragma unroll 1
  for (int kb = 0; kb < num_kb; ++kb) {
    uint32_t slot[NLOAD], ph[NLOAD];  // unit x of this k-block was loaded pos[x]-th after slot u
    static_for<0, NLOAD>([&](auto X) {
      constexpr int x = decltype(X)::value;
      constexpr int pos = P::pl.pos[x];
      int sidx = u + pos;
      ph[x] = phase;
      if (sidx >= UNITS) {
        sidx -= UNITS;
        ph[x] ^= 1u;
      }
      slot[x] = (uint32_t)sidx;
    });
    static_for<0, P::pl.nsteps>([&](auto ST) {
      constexpr int st = decltype(ST)::value;
      static_for<0, NLOAD>([&](auto X) {
        constexpr int x = decltype(X)::value;
        constexpr bool need = (P::pl.wait_mask[st] >> x) & 1u;
        if constexpr (need) mbar_wait(full_bar + 8 * slot[x], ph[x]);
      });
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      constexpr int p_begin = st == 0 ? 0 : P::pl.step_end[st == 0 ? 0 : st - 1];
      constexpr int p_end = P::pl.step_end[st];
      static_for<p_begin, p_end>([&](auto PI) {
        constexpr int pi = decltype(PI)::value;
        constexpr int ua = P::pl.prod_a[pi], ub = P::pl.prod_b[pi], gi = P::pl.prod_g[pi];
        constexpr bool first = P::pl.prod_first[pi] != 0;
        const uint32_t tmem_d = tmem_base + gi * TN;
        const uint64_t da = make_smem_desc(smem_base + slot[ua] * UNIT_BYTES);
        const uint64_t db = make_smem_desc(smem_base + slot[ub] * UNIT_BYTES + TILE_BYTES);
#pragma unroll
        for (int ks = 0; ks < BK / UMMA_K; ++ks) {
          const uint64_t adv = (uint64_t)((ks * UMMA_K) >> 4);  // +32 B per k-step inside the swizzle row
          umma_i8_2cta_pred(tmem_d, da + adv, db + adv, IDESC, (kb != 0 || !first || ks != 0) ? 1u : 0u);
        }
      });
      static_for<0, NLOAD>([&](auto X) {  // finished units go back to the producer (both CTAs) once the MMAs retire
        constexpr int x = decltype(X)::value;
        constexpr bool fin = (P::pl.free_mask[st] >> x) & 1u;
        if constexpr (fin) umma_commit_pair_pred(empty_bar + 8 * slot[x]);
      });
    });
    u += NLOAD;
    if (u >= UNITS) {
      u -= UNITS;
      phase ^= 1u;
    }
  }
}

template <int MODE>
__device__ __forceinline__ void mma_pass_dispatch(int nload, int ngroups, const int num_kb, int& u, uint32_t& phase,
                                                  const uint32_t smem_base, const uint32_t tmem_base,
                                                  const uint32_t full_bar, const uint32_t empty_bar) {
  switch (nload * 2 + ngroups) {  // groups 2ps (and 2ps+1) from the slices 0 .. nload-1
    case 2 * 2 + 2: mma_pass<2, 2, MODE>(num_kb, u, phase, smem_base, tmem_base, full_bar, empty_bar); break;
    case 4 * 2 + 2: mma_pass<4, 2, MODE>(num_kb, u, phase, smem_base, tmem_base, full_bar, empty_bar); break;
    case 6 * 2 + 2: mma_pass<6, 2, MODE>(num_kb, u, phase, smem_base, tmem_base, full_bar, empty_bar); break;
    case 8 * 2 + 2: mma_pass<8, 2, MODE>(num_kb, u, phase, smem_base, tmem_base, full_bar, empty_bar); break;
    case 3 * 2 + 1: mma_pass<3, 1, MODE>(num_kb, u, phase, smem_base, tmem_base, full_bar, empty_bar); break;
    case 5 * 2 + 1: mma_pass<5, 1, MODE>(num_kb, u, phase, smem_base, tmem_base, full_bar, empty_bar); break;
    default: mma_pass<7, 1, MODE>(num_kb, u, phase, smem_base, tmem_base, full_bar, empty_bar); break;
  }
}

struct OzParams {
  int64_t M, N;
  int num_kb;
  int nsl;
  int rb;  // radix bits of the digits (7 or 8)
  int tiles_m, tiles_n;
  const double* sA;
  const double* sB;
  const double* nA;
  const double* nB;
  double* C;
  int64_t ldc;
  double* Ct;
  int64_t ldct;
  unsigned int* wave_counter;  // zeroed before the launch
  int align_mode;              // 0 free-running, 1 align the producers per wave, 2 per wave and pass
  int plan_mode;               // PassPlan mode
};

__global__ void __launch_bounds__(NUM_THREADS, 1)
corr_ozaki_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const OzParams p) {
  extern __shared__ unsigned char smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + UNITS * UNIT_BYTES;
  const uint32_t full_bar = bar_base;                 // [UNITS]  (used in the leader: both CTAs' TMA bytes land here)
  const uint32_t empty_bar = bar_base + 8 * UNITS;    // [UNITS]  (one per CTA: multicast commit)
  const uint32_t tfull_bar = bar_base + 16 * UNITS;   // accumulators complete (one per CTA: multicast commit)
  const uint32_t tempty_bar = tfull_bar + 8;          // accumulators drained (leader: 2 x EPI_WARPS arrivals)
  const uint32_t tmem_slot = tempty_bar + 8;

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);  // provably warp-uniform for the compiler
  const int lane = threadIdx.x & 31;
  uint32_t cta_rank;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(cta_rank));
  const bool leader = cta_rank == 0;
  const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;
  const int num_tiles = p.tiles_m * p.tiles_n;
  const int npass = (p.nsl + 1) >> 1;

  if (warp == 0 && lane == 0) {
    for (int u = 0; u < UNITS; ++u) {
      mbar_init(full_bar + 8 * u, 1);
      mbar_init(empty_bar + 8 * u, 1);
    }
    mbar_init(tfull_bar, 1);
    mbar_init(tempty_bar, 2 * EPI_WARPS);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
  }
  if (warp == 1) {  // the same warp of both CTAs allocates the pair's TMEM (all 512 columns, 1 CTA per SM)
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  cluster_sync_all();  // both CTAs' barriers are initialised before any remote completion / arrival
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));
  tmem_base = __shfl_sync(0xffffffffu, tmem_base, 0);

  if (warp == 0) {
    // ===================== TMA producer (both CTAs; warp-uniform loops, one elected lane issues) ==========
    {
      int u = 0;
      uint32_t phase = 0;
      unsigned int wave_target = 0;
      for (int tile = pair; tile < num_tiles; tile += num_pairs) {
        // Wave alignment.  The ~74 pair tiles of a wave share 8 RNA and ~9 DNA panels, but only the k-window all
        // of them are currently working in fits L2 (1.8 MB of distinct digits per k-block).  Free-running pairs
        // drift apart over the waves and every pair then streams its panels from HBM by itself (ncu: 755 GB of
        // DRAM reads, L2 hit rate 45 %).  So the leaders' producers start each wave together; inside a wave the
        // pairs keep each other in step (whoever is ahead takes the DRAM misses, the others hit L2 and catch up).
        // All CTAs are co-resident (grid <= #SMs, 1 CTA/SM), so the spin cannot deadlock.
        const int wave = (tile - pair) / num_pairs;
        const unsigned int wave_pairs = (unsigned int)min(num_pairs, num_tiles - wave * num_pairs);
        auto align = [&]() {
          wave_target += wave_pairs;
          if (lane == 0) {
            asm volatile("red.relaxed.gpu.global.add.u32 [%0], 1;" ::"l"(p.wave_counter) : "memory");
            unsigned int seen;
            do {
              asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(p.wave_counter) : "memory");
              if ((int)(seen - wave_target) < 0) __nanosleep(200);
            } while ((int)(seen - wave_target) < 0);
          }
          __syncwarp();
        };
        if (leader && tile != pair && p.align_mode >= 1) align();
        int tm, tn;
        decode_tile(tile, p.tiles_m, p.tiles_n, tm, tn);
        const int row0 = tm * TM + (int)cta_rank * HALF;
        const int col0 = tn * TN + (int)cta_rank * HALF;
        for (int ps = npass - 1; ps >= 0; --ps) {
          const int nload = min(p.nsl, 2 * ps + 2);  // slices 0 .. nload-1 take part in the groups 2ps, 2ps+1
          if (leader && ps != npass - 1 && p.align_mode >= 2) align();  // also re-align at every pass
          const uint32_t order = load_order(nload, min(2, p.nsl - 2 * ps), p.plan_mode);
          for (int kb = 0; kb < p.num_kb; ++kb) {
            for (int k = 0; k < nload; ++k) {
              const int t = (int)((order >> (4 * k)) & 15u);  // units are loaded in the order the MMA plan needs them
              mbar_wait(empty_bar + 8 * u, phase ^ 1);
              const uint32_t fb_leader = map_to_cta(full_bar + 8 * u, 0);
              if (leader) mbar_expect_tx_elect(full_bar + 8 * u, 2 * UNIT_BYTES);  // own + peer's A_t and B_t tiles
              const uint32_t dst = smem_base + u * UNIT_BYTES;
              tma_load_3d_elect(dst, &map_a, fb_leader, kb * BK, row0, t);
              tma_load_3d_elect(dst + TILE_BYTES, &map_b, fb_leader, kb * BK, col0, t);
              if (++u == UNITS) {
                u = 0;
                phase ^= 1;
              }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA; warp-uniform loops, lane 0 issues) =====================
    if (leader) {
      int u = 0;
      uint32_t phase = 0;
      uint32_t tphase = 0;
      for (int tile = pair; tile < num_tiles; tile += num_pairs) {
        for (int ps = npass - 1; ps >= 0; --ps) {
          const int nload = min(p.nsl, 2 * ps + 2);
          const int ngroups = min(2, p.nsl - 2 * ps);
          mbar_wait(tempty_bar, tphase ^ 1);  // both CTAs' epilogue warps drained the previous pass
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          if (p.plan_mode == 0)
            mma_pass_dispatch<0>(nload, ngroups, p.num_kb, u, phase, smem_base, tmem_base, full_bar, empty_bar);
          else
            mma_pass_dispatch<1>(nload, ngroups, p.num_kb, u, phase, smem_base, tmem_base, full_bar, empty_bar);
          umma_commit_pair_pred(tfull_bar);  // both accumulators of this pass complete
          tphase ^= 1;
        }
      }
    }
  } else {
    // ===================== epilogue (warps 2..9 of both CTAs) =====================
    const int quad = warp & 3;         // TMEM lane quadrant this warp may access
    const int half = (warp - 2) >> 2;  // which 128-column half of the tile
    const uint32_t tempty_leader = map_to_cta(tempty_bar, 0);
    double* const P = p.C ? p.C : p.Ct;  // where the FP64 partial sums live between passes
    const bool p_is_c = p.C != nullptr;
    const bool c_vec = p_is_c && ((p.ldc & 1) == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0);
    uint32_t tphase = 0;
    for (int tile = pair; tile < num_tiles; tile += num_pairs) {
      int tm, tn;
      decode_tile(tile, p.tiles_m, p.tiles_n, tm, tn);
      const int64_t row = (int64_t)tm * TM + (int64_t)cta_rank * HALF + quad * 32 + lane;
      const bool row_ok = row < p.M;
      const double na = row_ok ? p.nA[row] : 0.0;
      const double sa = row_ok ? p.sA[row] : 0.0;
      for (int ps = npass - 1; ps >= 0; --ps) {
        const int g_lo = 2 * ps;
        const bool two = p.nsl - g_lo >= 2;
        const bool first = ps == npass - 1, last = ps == 0;
        const double w0 = scalbn(1.0, -p.rb * g_lo), w1 = scalbn(1.0, -p.rb * (g_lo + 1));
        const double fin = scalbn(1.0, 2 - 2 * p.rb);
        mbar_wait(tfull_bar, tphase);
        tphase ^= 1;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + half * HALF;
#pragma unroll 1
        for (int c = 0; c < HALF / 32; ++c) {
          uint32_t r0[32], r1[32];
          tmem_ld32(taddr + c * 32, r0);
          if (two) tmem_ld32(taddr + TN + c * 32, r1);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (row_ok) {
            const int64_t col0 = (int64_t)tn * TN + half * HALF + c * 32;
            if (p_is_c && c_vec && col0 + 32 <= p.N) {
              // whole 32-column chunk inside the matrix: 128-bit accesses, all partial-sum loads issued up front
              double2* prow = reinterpret_cast<double2*>(P + row * p.ldc + col0);
              double2 acc[16];
              if (!first) {
#pragma unroll
                for (int q2 = 0; q2 < 16; ++q2) acc[q2] = prow[q2];
              }
#pragma unroll
              for (int q2 = 0; q2 < 16; ++q2) {
                double v0 = (double)(int)r0[2 * q2] * w0, v1 = (double)(int)r0[2 * q2 + 1] * w0;
                if (two) {
                  v0 += (double)(int)r1[2 * q2] * w1;
                  v1 += (double)(int)r1[2 * q2 + 1] * w1;
                }
                if (!first) {
                  v0 += acc[q2].x;
                  v1 += acc[q2].y;
                }
                if (last) {
                  const int64_t col = col0 + 2 * q2;
                  const double nn0 = na * __ldg(p.nB + col), nn1 = na * __ldg(p.nB + col + 1);
                  v0 = v0 * (sa * __ldg(p.sB + col) * fin) * (nn0 / (1e-10 + nn0));
                  v1 = v1 * (sa * __ldg(p.sB + col + 1) * fin) * (nn1 / (1e-10 + nn1));
                  if (p.Ct) {
                    p.Ct[col * p.ldct + row] = v0;
                    p.Ct[(col + 1) * p.ldct + row] = v1;
                  }
                }
                prow[q2] = make_double2(v0, v1);
              }
            } else {
#pragma unroll
            for (int q = 0; q < 32; ++q) {
              const int64_t col = col0 + q;
              if (col < p.N) {
                double v = (double)(int)r0[q] * w0;
                if (two) v += (double)(int)r1[q] * w1;
                const int64_t pi = p_is_c ? row * p.ldc + col : col * p.ldct + row;
                if (!first) v += P[pi];
                if (last) {
                  const double nn = na * __ldg(p.nB + col);
                  // <u_i, u_j> * nn/(1e-10+nn) == dot(xc, yc)/(1e-10 + |xc||yc|)  (macrodna.py:25)
                  v = v * (sa * __ldg(p.sB + col) * fin) * (nn / (1e-10 + nn));
                  if (p.C) p.C[row * p.ldc + col] = v;
                  if (p.Ct) p.Ct[col * p.ldct + row] = v;
                } else {
                  P[pi] = v;
                }
              }
            }
            }
          }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(tempty_leader);
      }
    }
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  cluster_sync_all();  // no CTA leaves while its peer may still read its operand tiles / arrive on its barriers
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TMEM_COLS) : "memory");
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  }
  return fn;
}

// 3-D map over the digit slices [nsl, rows, ldk8] (K-major): box = 64 bytes x 128 rows x 1 slice, 64 B swizzle,
// rows / genes beyond the extents read as zero digits.
bool make_map(CUtensorMap* map, const int8_t* base, int64_t rows, int64_t ldk8, int64_t slice_stride, int nsl) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return false;
  cuuint64_t dims[3] = {(cuuint64_t)ldk8, (cuuint64_t)rows, (cuuint64_t)nsl};
  cuuint64_t strides[2] = {(cuuint64_t)ldk8, (cuuint64_t)slice_stride};
  cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)HALF, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<int8_t*>(base), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace

int mcd_launch_corr_ozaki(mcd_context* h, const int8_t* A, int64_t a_stride, int64_t M, const int8_t* B,
                          int64_t b_stride, int64_t N, int64_t ldk8, int nsl, int rb, const double* sA, const double* sB,
                          const double* nA, const double* nB, double* C, int64_t ldc, double* Ct, int64_t ldct) {
  if (M == 0 || N == 0) return MCD_OK;
  if ((reinterpret_cast<uintptr_t>(A) & 15) || (reinterpret_cast<uintptr_t>(B) & 15) || (ldk8 % BK) != 0 ||
      (a_stride & 15) || (b_stride & 15) || (rb != 7 && rb != 8) || nsl < 2 || nsl > (rb == 8 ? 7 : MCD_OZAKI_MAX_SLICES))
    return mcd_fail(h, MCD_ERR_INVALID,
                    "corr_ozaki: operands must be 16-byte aligned, ldk8 a multiple of 64, 2..8 slices of 7 bits or 2..7 of 8");
  if (!mcd_ozaki_exact(nsl, rb, ldk8))
    return mcd_fail(h, MCD_ERR_UNSUPPORTED, "corr_ozaki: too many genes for exact int32 accumulation");
  CUtensorMap ma, mb;
  if (!make_map(&ma, A, M, ldk8, a_stride, nsl) || !make_map(&mb, B, N, ldk8, b_stride, nsl))
    return mcd_fail(h, MCD_ERR_CUDA, "cuTensorMapEncodeTiled failed");
  OzParams p;
  p.M = M;
  p.N = N;
  p.num_kb = (int)(ldk8 / BK);
  p.nsl = nsl;
  p.rb = rb;
  p.tiles_m = (int)((M + TM - 1) / TM);
  p.tiles_n = (int)((N + TN - 1) / TN);
  p.sA = sA;
  p.sB = sB;
  p.nA = nA;
  p.nB = nB;
  p.C = C;
  p.ldc = ldc;
  p.Ct = Ct;
  p.ldct = ldct;
  p.wave_counter = reinterpret_cast<unsigned int*>(h->d_flags + 8);
  p.align_mode = h->opt.ozaki_align;
  p.plan_mode = h->opt.ozaki_plan;
  MCD_CUDA(h, cudaMemsetAsync(p.wave_counter, 0, sizeof(unsigned int), h->stream));
  MCD_CUDA(h, cudaFuncSetAttribute(corr_ozaki_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  const int64_t tiles = (int64_t)p.tiles_m * p.tiles_n;
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = h->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  // the wave alignment spins on peers, so every CTA pair of the grid must be resident at once
  cfg.gridDim = dim3(h->sm_count & ~1);
  int resident_pairs = 0;
  MCD_CUDA(h, cudaOccupancyMaxActiveClusters(&resident_pairs, corr_ozaki_kernel, &cfg));
  if (resident_pairs < 1) return mcd_fail(h, MCD_ERR_CUDA, "corr_ozaki_kernel: no CTA pair can be resident");
  int64_t max_pairs = h->sm_count / 2;
  if (resident_pairs < max_pairs) max_pairs = resident_pairs;
  const int grid = 2 * (int)(tiles < max_pairs ? tiles : max_pairs);
  cfg.gridDim = dim3(grid);
  MCD_CUDA(h, cudaLaunchKernelEx(&cfg, corr_ozaki_kernel, ma, mb, p));
  h->launches++;
  return MCD_OK;
}
