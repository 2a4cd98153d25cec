// K3 -- exact rectangular assignment on the GPU.
//
// Replaces one `ilp` call of the reference (src/MaCroDNA/macrodna.py:27-84): maximise
// sum_i W[i, col(i)] over injective maps of n "persons" (rows) into m >= n "objects"
// (columns).  The Gurobi model there is a totally unimodular assignment polytope, so the
// exact LAP optimum is the ILP optimum.
//
// Algorithm (all FP64, exact complementary slackness -- no epsilon in the final answer):
//   phase A  Jacobi forward auction.  Every unassigned person finds the best and second-best
//            value  W[i,j] - price[j]  of its row, bids  price += best - second  (the "naive"
//            eps = 0 increment, which keeps exact CS: the bidder is indifferent between its object
//            and its runner-up), one winner per object, evicted owners rejoin the bidder list.
//            * candidate lists: a full row sweep also keeps the person's top-128 objects and the
//              129th value as a bound.  Prices only ever rise, so every unlisted object stays below
//              that bound; while the list's own second-best is still >= the bound, the list's top-2
//              ARE the row's top-2 and the bid needs 128 gathers instead of an m-long sweep
//              (18x fewer row sweeps at 10k x 50k, identical trajectory).
//            * wide rounds (> TAIL_NU bidders) run in a persistent cooperative kernel over the
//              whole grid; the narrow rounds (~93 % of all rounds, a handful of bidders each) run
//              in ONE CTA, where a round is a few hundred cycles of L1/L2 latency instead of two
//              grid barriers.
//            * n == m (every object must be sold) degenerates into price wars, so it is preceded by
//              eps-scaling phases (eps = range/4, /16, ... >= 1e-6*range) whose only product is the
//              price vector the final eps = 0 phase starts from -- valid for square problems because
//              every object ends up assigned.  For n < m all prices start at 0 and an object once
//              assigned stays assigned, so unassigned objects keep price 0 = the minimum: the
//              rectangular optimality condition holds by construction.
//   phase B  whatever the auction leaves (exact ties give zero increments -> no progress) is
//            finished by shortest-augmenting-path (Jonker-Volgenant/Dijkstra) steps that start from
//            the auction's dual-feasible prices/profits and tight partial matching.
//
// Bound: HBM bandwidth for the row sweeps (8 B per object), L2/launch latency for the narrow rounds.
#include <type_traits>

#include "mcd_internal.cuh"

namespace {

constexpr int LAP_THREADS = 256;   // wide kernel CTA
constexpr int LAP_WARPS = LAP_THREADS / 32;
constexpr int TAIL_THREADS = 512;  // narrow kernel CTA
constexpr int TAIL_WARPS = TAIL_THREADS / 32;
constexpr int TAIL_NU = 128;       // bidder count at which the single-CTA kernel takes over
constexpr int JV_THREADS = 1024;
#ifndef MCD_LIST_K
#define MCD_LIST_K 128
#endif
constexpr int LIST_K = MCD_LIST_K;  // candidate objects kept per person
constexpr int CAND_T = 4;          // per-thread candidates kept during a row sweep
constexpr int MAX_PHASES = 48;
constexpr int MAX_GRID_SLOTS = 4096;  // >= cooperative grid size
constexpr double NEG_INF = -1.0e300;  // finite sentinel: inputs are finite correlations
// A bid on an OWNED object must raise its price by more than this to be applied (2^-46: costs are correlations, O(1),
// so this is ~60 ulps of a price).  Exact ties (duplicated cells) give increments of 0 or of a few ulps of rounding
// noise; the latter used to count as progress, and two tied persons could swap an object back and forth until the
// round guard (264 000 rounds on a resampled replicate).  Treated as "no increment", such bidders stall and go to the
// shortest-augmenting-path kernel, which is exact from any dual-feasible state.
constexpr double GAMMA_TIE = 1.4210854715202004e-14;

// Grid-wide barrier for the persistent wide kernel (launched with cudaLaunchCooperativeKernel so
// all CTAs are co-resident).  One monotonic counter; each CTA's thread 0 arrives with a RELEASE
// reduction (MEMBAR.ALL.GPU + REDG) and spins on a relaxed gpu-scope load.  There is deliberately
// no acquire fence: on sm_100a every gpu-scope acquire (ld.acquire, fence.acq_rel, __threadfence,
// cooperative_groups grid.sync) ends in CCTL.IVALL, a whole-L1 invalidate that ncu showed costing
// ~4x the actual wait in this latency-bound round loop.  Instead every load of state that other
// CTAs mutate goes through ldm() = ld.global.cg (L2, the coherence point), so there is no stale L1
// line to drop.  The cost matrix W is immutable during the kernel and keeps the cached path.
struct GridBarrier {
  unsigned int* counter;
  unsigned int target;
  // split form: between arrive() and wait() a CTA may do work that nobody needs before the NEXT barrier (one
  // outstanding barrier per CTA: the single monotonic counter cannot tell generations apart otherwise)
  __device__ __forceinline__ void arrive() {
    __syncthreads();
    if (threadIdx.x == 0) {
      target += gridDim.x;
      asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(counter) : "memory");
    }
  }
  __device__ __forceinline__ void wait() {
    if (threadIdx.x == 0) {
      unsigned int seen;
      do {
        asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(counter) : "memory");
      } while ((int)(seen - target) < 0);
    }
    __syncthreads();
  }
  __device__ __forceinline__ void sync() {
    arrive();
    wait();
  }
};

// load of inter-CTA mutable state: L2-coherent, never served from a stale L1 line
template <typename T>
__device__ __forceinline__ T ldm(const T* p) {
  return __ldcg(p);
}

struct LapCtrl {
  int cnt[2];       // bidder-list lengths (double buffered)
  int progress[2];  // successful bids per round (double buffered by round parity)
  int cur;          // which list is current
  int stalled;      // phase A ended with bidders it cannot place (exact ties / guard) -> augmentation kernel
  double wmin, wmax;
  int finished;     // the final (eps = 0) phase has run: later auction launches are no-ops
  int in_tail;      // the wide kernel stopped with <= TAIL_NU bidders: the narrow kernel continues the phase
  double eps;       // eps of the phase in flight (handed from the wide kernel to the narrow kernel)
  int nfail[2];     // bidders whose candidate list failed this round (double buffered by round parity)
  int nhold[2];     // bidders that sat the round out because their list is being rebuilt (same buffering)
  unsigned int barrier[MAX_PHASES];  // one GridBarrier counter per wide-kernel launch
  // asynchronous wide kernel: next never-bid person, live count of unassigned persons, stop flag
  unsigned int aq_head, aq_tail;
  int a_active, a_stop, a_parked, a_guard;
  unsigned long long a_bids;
  unsigned long long a_t0;
  unsigned long long a_hops;
  int a_tie;       // an exact tie was met (two equal best values, or a bid that cannot raise a price)
  int a_fallback;  // ... so the step is redone by the round-synchronous kernel
  int sap_cnt[3];  // lap_sap_kernel: frontier lengths of rounds t, t + 1 (being appended) and t + 2 (being cleared)
};

struct LapState {
  const double* W;
  int n, m;
  int64_t ldw;
  int vec;     // 128-bit loads of W rows legal
  int list_k;  // min(LIST_K, m)
  double* price;             // [m]
  int* owner;                // [m]
  unsigned long long* key;   // [m] winning bid per object in the wide kernel
  double* profit;            // [n]
  int* col4row;              // [n]  (caller's output)
  int* bj;                   // [n] bid object per list slot
  double* gam;               // [n] bid increment per list slot
  double* bval;              // [n] bidder's value (W - price) of the object it bids on, per list slot
  int* un[2];                // [n] bidder lists
  int* lj;                   // [n * LIST_K] candidate objects
  double* lw;                // [n * LIST_K] their costs W[i, j]
  double* lbound;            // [n] no unlisted object is worth more than this to person i -- stored as the
                             //     order-preserving 64-bit key of the double (lb_store / lb_load): the chunks of a
                             //     cooperative rebuild fold their bounds in with one atomic max each
  int* lvalid;               // [n] 0 = never built, v >= 1 = usable from wide-kernel round v - 1 on
  int* fail;                 // [2][n] persons whose candidate list could not certify the top-2 (per round parity)
  int max_chunks;            // no-list mode: upper bound on CTAs sharing one row
  int chunk_waves;           // list rebuilds: at most this many chunks per CTA per round
  int* done;                 // [n] chunks finished per list slot
  double* pv1;               // [grid slots] partial best / second / objects of split rows
  double* pv2;
  int* pj1;
  int* pj2;
  double* pbound;            // [grid slots] chunk bounds of cooperative list rebuilds
  // augmentation scratch
  double* sp;                // [m] shortest path cost
  int* pred;                 // [m]
  int* sc_col;               // [n + 1] scanned columns in scan order
  double* sc_val;            // [n + 1] their path cost when scanned
  int* sap_r;                // [2][n] lap_sap_kernel frontier (double buffered by round parity): owner row,
  double* sap_d;             // [2][n]   distance of the owned column that improved,
  double* sap_p;             // [2][n]   and the owner's profit
  LapCtrl* ctrl;
  mcd_lap_counters* counters;
  const int* flags;  // [0] != 0: non-finite data was seen upstream -> every solver kernel is a no-op
  long long max_rounds;
  long long tail_budget;  // narrow rounds after which a phase with <= MH_BUDGET_NU bidders goes to augmenting paths
  // eps-scaling phases (eps > 0) only produce start prices for the next phase, which restarts with everybody
  // unassigned: such a phase may end early -- once at most scale_cut_nu persons are still bidding, or after
  // scale_tail_rounds narrow rounds (the last few persons of a phase are one long dependent eviction chain).
  int scale_cut_nu;
  long long scale_tail_rounds;
  int prefetch_rows;  // symmetric cluster tail: L2 prefetch of the likely next bidder's cost row
  ulonglong2* pw;     // [m] asynchronous wide kernel: {price bits, owner as u32} per object, updated by 128-bit CAS
  // Classes of similar persons (identical cost rows: copies of one resampled DNA cell).  pcls[i] = class id of
  // person i (persons with equal ids are copies), NULL = every person is its own class; ocls[j] = class of the
  // person that owns object j (-1 = free).  A bidder never bids against its own copies: objects held by its class
  // are skipped (swapping two copies changes nothing, and a bid between them has increment exactly 0 -- the auction
  // would stall on every duplicated cell).  What this leaves open -- copies holding objects at different profit
  // levels -- is closed by lap_class_equalize_kernel before the augmentation kernel / the certificate.
  //   clevel[t] = lowest profit any member of class t has settled at so far (order-preserving key).  While copies sit
  //   at different levels, an object held by a copy at a HIGH level is under-priced from the class's point of view
  //   (a copy at the low level would rather have it): a bidder of another class must raise its price at least to the
  //   class level to take it, otherwise the owner raises it there itself and keeps it (class_defends()).
  const int* pcls;
  int* ocls;
  unsigned long long* clevel;
};

struct Top2 {
  double v1, v2;
  int j1, j2;
};

// Written with non-short-circuit operators and selects: these run inside one-warp dependent chains, where a
// divergent double-compare branch costs more than the few redundant instructions.
__device__ __forceinline__ bool better(double va, int ja, double vb, int jb) {
  return (va > vb) | ((va == vb) & (ja < jb));
}
__device__ __forceinline__ void top2_push(Top2& t, double v, int j) {
  const bool b1 = better(v, j, t.v1, t.j1), b2 = better(v, j, t.v2, t.j2);
  const double nv2 = b1 ? t.v1 : (b2 ? v : t.v2);
  const int nj2 = b1 ? t.j1 : (b2 ? j : t.j2);
  t.v1 = b1 ? v : t.v1;
  t.j1 = b1 ? j : t.j1;
  t.v2 = nv2;
  t.j2 = nj2;
}
// in-thread variant: candidates arrive in increasing j, so strict '>' keeps the smallest index on ties
__device__ __forceinline__ void top2_push_seq(Top2& t, double v, int j) {
  const bool b1 = v > t.v1, b2 = v > t.v2;
  const double nv2 = b1 ? t.v1 : (b2 ? v : t.v2);
  const int nj2 = b1 ? t.j1 : (b2 ? j : t.j2);
  t.v1 = b1 ? v : t.v1;
  t.j1 = b1 ? j : t.j1;
  t.v2 = nv2;
  t.j2 = nj2;
}
__device__ __forceinline__ void top2_merge(Top2& a, const Top2& b) {
  top2_push(a, b.v1, b.j1);
  top2_push(a, b.v2, b.j2);
}
// ---- warp-level selection through redux.sync ------------------------------------------------------------
// The narrow rounds are one dependent chain, and ncu's source view put most of the working warp's time into the
// shuffle-and-branch top-2 butterfly (5 levels x 6 shuffles x two branchy double compares).  An arg-max over the warp
// is three integer warp reductions instead: the doubles are mapped to order-preserving 64-bit keys, the high
// words, the low words among the lanes that tie on the high word, and the object index among the lanes that tie on
// both are reduced with redux.sync.  Same total order as better(): larger value first, smaller index on ties.
__device__ __forceinline__ unsigned long long f64_sortable(double v) {
  const long long b = __double_as_longlong(v + 0.0);  // -0.0 -> +0.0: equal doubles get equal keys
  return (unsigned long long)(b ^ ((b >> 63) | (long long)0x8000000000000000ull));
}
__device__ __forceinline__ double sortable_f64(unsigned long long k) {
  const unsigned long long b = (k & 0x8000000000000000ull) ? (k ^ 0x8000000000000000ull) : ~k;
  return __longlong_as_double((long long)b);
}
// candidate-list bound of person i (see LapState::lbound)
__device__ __forceinline__ unsigned long long* lb_keys(const LapState& s) {
  return reinterpret_cast<unsigned long long*>(s.lbound);
}
__device__ __forceinline__ void lb_store(const LapState& s, int i, double b) { lb_keys(s)[i] = f64_sortable(b); }
// every lane returns the best key, its index, and the lane that held it
__device__ __forceinline__ void warp_argmax_key(unsigned long long key, int j, unsigned long long& kbest, int& jbest,
                                                int& wlane) {
  const unsigned hi = (unsigned)(key >> 32), lo = (unsigned)key;
  const unsigned mh = __reduce_max_sync(0xffffffffu, hi);
  const bool c1 = hi == mh;
  const unsigned ml = __reduce_max_sync(0xffffffffu, c1 ? lo : 0u);
  const bool c2 = c1 && lo == ml;
  const unsigned mj = __reduce_min_sync(0xffffffffu, c2 ? (unsigned)j : 0xffffffffu);  // j = -1 (nothing) loses ties
  kbest = ((unsigned long long)mh << 32) | ml;
  jbest = (int)mj;
  wlane = __ffs(__ballot_sync(0xffffffffu, c2 && (unsigned)j == mj)) - 1;
}
// Top-2 over the warp of per-lane sorted pairs (objects are distinct across lanes): the best is the best of the
// lanes' firsts; the runner-up is the best of {the winner lane's second, the other lanes' firsts}.
__device__ __forceinline__ Top2 top2_warp_reduce(Top2 t) {
  const int lane = threadIdx.x & 31;
  const unsigned long long k1 = f64_sortable(t.v1), k2 = f64_sortable(t.v2);
  unsigned long long kb1, kb2;
  int jb1, jb2, w1, w2;
  warp_argmax_key(k1, t.j1, kb1, jb1, w1);
  warp_argmax_key(lane == w1 ? k2 : k1, lane == w1 ? t.j2 : t.j1, kb2, jb2, w2);
  Top2 r;
  r.v1 = sortable_f64(kb1);
  r.j1 = jb1;
  r.v2 = sortable_f64(kb2);
  r.j2 = jb2;
  return r;
}

__device__ __forceinline__ unsigned long long pack_bid(double gamma, int person) {
  // increments are >= 0: the float32 bit pattern is monotone; person id breaks ties deterministically
  const float g = (float)gamma;
  return ((unsigned long long)__float_as_uint(g) << 32) | (unsigned)(person + 1);
}

// ------------------------------------------------------------------------------------------------
// Bids from the candidate list (one warp) and from a full row sweep that rebuilds the list (one CTA)
// ------------------------------------------------------------------------------------------------

// COHERENT = true: prices / lists may have been written by other SMs in this launch (wide kernel) -> ld.cg.
template <bool COHERENT>
__device__ __forceinline__ bool list_bid(const LapState& s, int i, int lane, Top2& out) {
  const int K = s.list_k;
  const int mycls = s.pcls != nullptr ? __ldg(s.pcls + i) : -2;  // -2 never equals an owner class (>= -1)
  const int* lj = s.lj + (int64_t)i * LIST_K;
  const double* lw = s.lw + (int64_t)i * LIST_K;
  // everything that depends only on i is requested up front: the bid is two dependent memory latencies
  // (list, then the prices of its objects), not four
  const int valid = COHERENT ? ldm(&s.lvalid[i]) : s.lvalid[i];
  const double b = sortable_f64(COHERENT ? ldm(lb_keys(s) + i) : lb_keys(s)[i]);
  int js[LIST_K / 32];
  double ws[LIST_K / 32];
#pragma unroll
  for (int q = 0; q < LIST_K / 32; ++q) {
    const int e = lane + 32 * q;
    js[q] = -1;
    ws[q] = NEG_INF;
    if (e < K) {
      js[q] = COHERENT ? ldm(lj + e) : lj[e];
      ws[q] = COHERENT ? ldm(lw + e) : lw[e];
    }
  }
  Top2 t{NEG_INF, NEG_INF, -1, -1};
  out = t;
  if (!valid) return false;  // never built: the slots hold garbage, do not touch them
  double ps[LIST_K / 32];
  int oc[LIST_K / 32];
#pragma unroll
  for (int q = 0; q < LIST_K / 32; ++q) {
    ps[q] = 0.0;
    oc[q] = -1;
    if (js[q] >= 0) {
      ps[q] = COHERENT ? ldm(s.price + js[q]) : s.price[js[q]];
      if (s.pcls != nullptr) oc[q] = COHERENT ? ldm(s.ocls + js[q]) : s.ocls[js[q]];  // same latency as the price
    }
  }
#pragma unroll
  for (int q = 0; q < LIST_K / 32; ++q)
    if (js[q] >= 0 && oc[q] != mycls) top2_push(t, ws[q] - ps[q], js[q]);  // objects of the bidder's own copies: skipped
  t = top2_warp_reduce(t);
  out = t;
  if (K == s.m) return true;  // every object is listed
  return t.j2 >= 0 && t.v2 >= b;
}

// A winning bid (increment gam) of person i on object j held by `prev`: if prev's class has settled lower than
// prev's own profit by more than gam, the object changes hands too cheaply -- a copy of prev at the class level would
// still prefer it at the new price, and nobody would ever tell it.  Returns the amount the owner must raise the price
// by to defend the object (> gam), or 0 when the bid stands.  COHERENT as in list_bid.
template <bool COHERENT>
__device__ __forceinline__ double class_defends(const LapState& s, int i, int prev, double gam) {
  if (s.pcls == nullptr || prev < 0) return 0.0;
  const int tp = __ldg(s.pcls + prev);
  if (tp == __ldg(s.pcls + i)) return 0.0;
  const double lvl = sortable_f64(ldm(s.clevel + tp));  // written by atomics (L2): never through a stale L1 line
  const double need = (COHERENT ? ldm(s.profit + prev) : s.profit[prev]) - lvl;
  return need > gam ? need : 0.0;
}
__device__ __forceinline__ void class_settle(const LapState& s, int i, double profit) {
  if (s.pcls != nullptr) atomicMin(s.clevel + __ldg(s.pcls + i), f64_sortable(profit));
}

// Whole-row sweep by an NT-thread CTA: exact top-2 of W[i,:] - price, and the person's new candidate
// list (top list_k by current value) with its bound.  Returns the top-2 in every thread.
// smem: cand_v[NT*CAND_T] doubles, cand_j[NT*CAND_T] ints, red[NT/32] doubles.
template <int NT, bool COHERENT>
__device__ Top2 full_scan_build(const LapState& s, int i, double* cand_v, int* cand_j, double* red,
                                bool set_valid = true) {
  constexpr int NC = NT * CAND_T;
  const int tid = threadIdx.x;
  const double* w = s.W + (int64_t)i * s.ldw;
  double tv[CAND_T];
  int tj[CAND_T];
#pragma unroll
  for (int q = 0; q < CAND_T; ++q) tv[q] = NEG_INF, tj[q] = 0x7fffffff;
  double lb = NEG_INF;  // largest value this thread dropped
  auto push = [&](double v, int j) {
    if (better(v, j, tv[CAND_T - 1], tj[CAND_T - 1])) {
      lb = fmax(lb, tv[CAND_T - 1]);
      tv[CAND_T - 1] = v;
      tj[CAND_T - 1] = j;
#pragma unroll
      for (int q = CAND_T - 1; q > 0; --q) {
        if (better(tv[q], tj[q], tv[q - 1], tj[q - 1])) {
          const double xv = tv[q];
          tv[q] = tv[q - 1];
          tv[q - 1] = xv;
          const int xj = tj[q];
          tj[q] = tj[q - 1];
          tj[q - 1] = xj;
        }
      }
    } else {
      lb = fmax(lb, v);
    }
  };
  if (s.vec) {
    constexpr int S = 2 * NT;
    int j = 2 * tid;
    for (; j + 3 * S + 1 < s.m; j += 4 * S) {  // 4 independent 128-bit loads in flight per thread
      double2 wv[4], pv[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) wv[u] = __ldg(reinterpret_cast<const double2*>(w + j + u * S));
#pragma unroll
      for (int u = 0; u < 4; ++u)
        pv[u] = COHERENT ? ldm(reinterpret_cast<const double2*>(s.price + j + u * S))
                         : *reinterpret_cast<const double2*>(s.price + j + u * S);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        push(wv[u].x - pv[u].x, j + u * S);
        push(wv[u].y - pv[u].y, j + u * S + 1);
      }
    }
    for (; j < s.m; j += S) {
      push(__ldg(w + j) - (COHERENT ? ldm(s.price + j) : s.price[j]), j);
      if (j + 1 < s.m) push(__ldg(w + j + 1) - (COHERENT ? ldm(s.price + j + 1) : s.price[j + 1]), j + 1);
    }
  } else {
    for (int j = tid; j < s.m; j += NT) push(__ldg(w + j) - (COHERENT ? ldm(s.price + j) : s.price[j]), j);
  }
#pragma unroll
  for (int q = 0; q < CAND_T; ++q) {
    cand_v[tid * CAND_T + q] = tv[q];
    cand_j[tid * CAND_T + q] = tj[q];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) lb = fmax(lb, __shfl_xor_sync(0xffffffffu, lb, o));
  if ((tid & 31) == 0) red[tid >> 5] = lb;
  __syncthreads();
  // bitonic sort of the NC candidates, descending by (value, -index)
  for (int k = 2; k <= NC; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int idx = tid; idx < NC; idx += NT) {
        const int ixj = idx ^ j;
        if (ixj > idx) {
          const double va = cand_v[idx], vb = cand_v[ixj];
          const int ja = cand_j[idx], jb = cand_j[ixj];
          const bool a_first = better(va, ja, vb, jb);
          const bool desc = (idx & k) == 0;
          if (desc ? !a_first : a_first) {
            cand_v[idx] = vb;
            cand_v[ixj] = va;
            cand_j[idx] = jb;
            cand_j[ixj] = ja;
          }
        }
      }
      __syncthreads();
    }
  }
  double bound = NEG_INF;
#pragma unroll
  for (int q = 0; q < NT / 32; ++q) bound = fmax(bound, red[q]);
  const int K = s.list_k;
  if (K < NC) bound = fmax(bound, cand_v[K]);  // (K+1)-th candidate, NEG_INF filler if there is none
  for (int q = tid; q < K; q += NT) {
    const int j = cand_j[q];
    s.lj[(int64_t)i * LIST_K + q] = j;
    s.lw[(int64_t)i * LIST_K + q] = __ldg(w + j);
  }
  if (tid == 0) {
    lb_store(s, i, bound);
    if (set_valid) s.lvalid[i] = 1;
  }
  Top2 t;
  t.v1 = cand_v[0];
  t.j1 = cand_j[0];
  const bool has2 = s.m > 1;
  t.v2 = has2 ? cand_v[1] : NEG_INF;
  t.j2 = has2 ? cand_j[1] : -1;
  __syncthreads();  // cand_* may be reused by the caller's next sweep
  return t;
}


// warp-wide arg-max of (v, j) with the smaller index winning ties; every lane returns the winner
__device__ __forceinline__ void warp_argmax(double& v, int& j) {
  unsigned long long kb;
  int jb, w;
  warp_argmax_key(f64_sortable(v), j, kb, jb, w);
  v = sortable_f64(kb);
  j = jb;
}

// Same contract as chunk_scan_build below for kc <= 16 (many short chunks), without the shared-memory sort:
// every lane keeps its top-2 and the largest value it dropped, every warp hands its best 4 to the CTA by four
// shuffle arg-max rounds, warp 0 picks the chunk's kc from those NT/32 * 4 (<= 32) candidates.  Whatever a warp
// or the CTA does not pass on only raises the bound, so the certificate stays valid (it is merely a little
// weaker than the exact chunk top-kc).  All loads of a chunk of <= 8 * 2 * NT objects are issued before the
// first use: a chunk costs one memory latency.
template <int NT>
__device__ Top2 chunk_scan_select(const LapState& s, int i, int j0, int j1, int c, int kc, double* s_cv, int* s_cj,
                                  double* s_wb, double* bound_out) {
  static_assert(NT / 32 * 4 <= 32, "one candidate per lane of warp 0");
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const double* w = s.W + (int64_t)i * s.ldw;
  Top2 t{NEG_INF, NEG_INF, -1, -1};
  double lb = NEG_INF;
  auto push = [&](double v, int j) {
    if (v > t.v1) {
      lb = fmax(lb, t.v2);
      t.v2 = t.v1, t.j2 = t.j1, t.v1 = v, t.j1 = j;
    } else if (v > t.v2) {
      lb = fmax(lb, t.v2);
      t.v2 = v, t.j2 = j;
    } else {
      lb = fmax(lb, v);
    }
  };
  if (s.vec) {  // j0 is even
    constexpr int S = 2 * NT;
    for (int j = j0 + 2 * tid; j < j1; j += 8 * S) {
      double2 wv[8], pv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int jj = j + u * S;
        wv[u] = make_double2(NEG_INF, NEG_INF);
        pv[u] = make_double2(0.0, 0.0);
        if (jj + 1 < j1) {
          wv[u] = __ldg(reinterpret_cast<const double2*>(w + jj));
          pv[u] = ldm(reinterpret_cast<const double2*>(s.price + jj));
        } else if (jj < j1) {
          wv[u].x = __ldg(w + jj);
          pv[u].x = ldm(s.price + jj);
        }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int jj = j + u * S;
        if (jj < j1) push(wv[u].x - pv[u].x, jj);
        if (jj + 1 < j1) push(wv[u].y - pv[u].y, jj + 1);
      }
    }
  } else {
    for (int j = j0 + tid; j < j1; j += NT) push(__ldg(w + j) - ldm(s.price + j), j);
  }
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    double bv = t.v1;
    int bj = t.j1;
    warp_argmax(bv, bj);
    if (bj >= 0 && bj == t.j1) {
      t.v1 = t.v2, t.j1 = t.j2;
      t.v2 = NEG_INF, t.j2 = -1;
    }
    if (lane == r) {
      s_cv[warp * 4 + r] = bv;
      s_cj[warp * 4 + r] = bj;
    }
  }
  double wb = fmax(lb, t.v1);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) wb = fmax(wb, __shfl_xor_sync(0xffffffffu, wb, o));
  if (lane == 0) s_wb[warp] = wb;
  __syncthreads();
  Top2 out{NEG_INF, NEG_INF, -1, -1};
  if (warp == 0) {
    constexpr int NCAND = NT / 32 * 4;
    double a1 = lane < NCAND ? s_cv[lane] : NEG_INF;
    int b1 = lane < NCAND ? s_cj[lane] : -1;
    if (b1 < 0) a1 = NEG_INF;
    double ev = NEG_INF;
    int ej = -1;
    for (int r = 0; r < kc; ++r) {
      double bv = a1;
      int bj = b1;
      warp_argmax(bv, bj);
      if (bj >= 0 && bj == b1) a1 = NEG_INF, b1 = -1;
      if (lane == r) ev = bv, ej = bj;
    }
    double cb = fmax(a1, lane < NT / 32 ? s_wb[lane] : NEG_INF);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cb = fmax(cb, __shfl_xor_sync(0xffffffffu, cb, o));
    if (lane < kc) {
      s.lj[(int64_t)i * LIST_K + c * kc + lane] = ej >= 0 ? ej : j0 < s.m ? j0 : 0;
      s.lw[(int64_t)i * LIST_K + c * kc + lane] = ej >= 0 ? __ldg(w + ej) : NEG_INF;
    }
    out.v1 = __shfl_sync(0xffffffffu, ev, 0);
    out.j1 = __shfl_sync(0xffffffffu, ej, 0);
    out.v2 = __shfl_sync(0xffffffffu, ev, 1);
    out.j2 = __shfl_sync(0xffffffffu, ej, 1);
    if (lane == 0) {
      s_cv[0] = out.v1, s_cv[1] = out.v2, s_cv[2] = cb;
      s_cj[0] = out.j1, s_cj[1] = out.j2;
    }
  }
  __syncthreads();
  out.v1 = s_cv[0], out.v2 = s_cv[1], out.j1 = s_cj[0], out.j2 = s_cj[1];
  *bound_out = s_cv[2];
  __syncthreads();
  return out;
}

// chunk_scan_select for 16 < kc <= 64 (few chunks per row: the rounds with many list failures), still without a
// sort: every lane keeps its top-2 and the largest value it dropped, every warp hands its best KW = kc / 4 to the
// CTA by KW arg-max rounds (NT/32 * KW = 2 kc candidates), and the chunk's kc are picked by RANK: candidate t counts
// the candidates that beat it (2 kc shared-memory compares per thread, all threads in parallel) and, if fewer than
// kc do, that count is its list slot.  Everything not passed on only raises the bound.  (chunk_scan_build's exact
// top-kc costs a 55-stage bitonic sort of 1024 candidates: ~4 us of the ~10 us rebuild chain of a wide round.)
// The chunk bound is returned in thread 0.
template <int NT>
__device__ void chunk_scan_rank(const LapState& s, int i, int j0, int j1, int c, int kc, double* s_cv, int* s_cj,
                                double* s_wb, double* bound_out) {
  constexpr int NW = NT / 32;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int kw = kc / 4;        // 8 or 16 per warp
  const int ncand = NW * kw;    // 2 * kc <= 128
  const double* w = s.W + (int64_t)i * s.ldw;
  Top2 t{NEG_INF, NEG_INF, -1, -1};
  double lb = NEG_INF;
  auto push = [&](double v, int j) {
    if (v > t.v1) {
      lb = fmax(lb, t.v2);
      t.v2 = t.v1, t.j2 = t.j1, t.v1 = v, t.j1 = j;
    } else if (v > t.v2) {
      lb = fmax(lb, t.v2);
      t.v2 = v, t.j2 = j;
    } else {
      lb = fmax(lb, v);
    }
  };
  if (s.vec) {  // j0 is even
    constexpr int S = 2 * NT;
    for (int j = j0 + 2 * tid; j < j1; j += 8 * S) {
      double2 wv[8], pv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int jj = j + u * S;
        wv[u] = make_double2(NEG_INF, NEG_INF);
        pv[u] = make_double2(0.0, 0.0);
        if (jj + 1 < j1) {
          wv[u] = __ldg(reinterpret_cast<const double2*>(w + jj));
          pv[u] = ldm(reinterpret_cast<const double2*>(s.price + jj));
        } else if (jj < j1) {
          wv[u].x = __ldg(w + jj);
          pv[u].x = ldm(s.price + jj);
        }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int jj = j + u * S;
        if (jj < j1) push(wv[u].x - pv[u].x, jj);
        if (jj + 1 < j1) push(wv[u].y - pv[u].y, jj + 1);
      }
    }
  } else {
    for (int j = j0 + tid; j < j1; j += NT) push(__ldg(w + j) - ldm(s.price + j), j);
  }
  for (int r = 0; r < kw; ++r) {
    double bv = t.v1;
    int bj = t.j1;
    warp_argmax(bv, bj);
    if (bj >= 0 && bj == t.j1) {
      t.v1 = t.v2, t.j1 = t.j2;
      t.v2 = NEG_INF, t.j2 = -1;
    }
    if (lane == (r & 31)) {
      s_cv[warp * kw + r] = bv;
      s_cj[warp * kw + r] = bj;
    }
  }
  double wb = fmax(lb, t.v1);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) wb = fmax(wb, __shfl_xor_sync(0xffffffffu, wb, o));
  if (lane == 0) s_wb[warp] = wb;
  __syncthreads();
  // rank of candidate tid among the ncand: order (value desc, object asc, slot asc) -- a strict total order even
  // among the empty candidates (object -1, value NEG_INF)
  double myv = NEG_INF;
  int myj = -1, rank = 0x7fffffff;
  if (tid < ncand) {
    myv = s_cv[tid];
    myj = s_cj[tid];
    if (myj < 0) myv = NEG_INF;
    rank = 0;
    for (int u = 0; u < ncand; ++u) {
      double uv = s_cv[u];
      const int uj = s_cj[u];
      if (uj < 0) uv = NEG_INF;
      const bool before = (uv > myv) | ((uv == myv) & (((unsigned)uj < (unsigned)myj) | ((uj == myj) & (u < tid))));
      rank += before ? 1 : 0;
    }
    if (rank < kc) {
      s.lj[(int64_t)i * LIST_K + c * kc + rank] = myj >= 0 ? myj : (j0 < s.m ? j0 : 0);
      s.lw[(int64_t)i * LIST_K + c * kc + rank] = myj >= 0 ? __ldg(w + myj) : NEG_INF;
    }
  }
  // chunk bound: the warps' dropped values and the candidates that did not make the list
  double cb = (tid < ncand && rank >= kc) ? myv : NEG_INF;
  if (tid < NW) cb = fmax(cb, s_wb[tid]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cb = fmax(cb, __shfl_xor_sync(0xffffffffu, cb, o));
  __syncthreads();  // every thread has read s_cv / s_cj / s_wb
  if (lane == 0) s_wb[warp] = cb;
  __syncthreads();
  if (tid == 0) {
    double b = NEG_INF;
#pragma unroll
    for (int q = 0; q < NW; ++q) b = fmax(b, s_wb[q]);
    *bound_out = b;
  }
  __syncthreads();  // scratch is free again
}

// One CHUNK [j0, j1) of a row sweep that rebuilds person i's candidate list cooperatively: nch CTAs each sweep
// one chunk and contribute their chunk's top kc = list_k / nch objects to the list slots [c*kc, (c+1)*kc) plus a
// chunk bound (no object of the chunk outside those kc is worth more).  The list is then the union of the chunk
// tops (not the global top-128, but every unlisted object is still below max_c bound_c, which is all the
// certificate needs).  Returns the chunk's exact top-2 in every thread; *bound_out is valid in every thread.
template <int NT>
__device__ Top2 chunk_scan_build(const LapState& s, int i, int j0, int j1, int c, int kc, double* cand_v, int* cand_j,
                                 double* red, double* bound_out) {
  constexpr int NC = NT * CAND_T;
  const int tid = threadIdx.x;
  const double* w = s.W + (int64_t)i * s.ldw;
  double tv[CAND_T];
  int tj[CAND_T];
#pragma unroll
  for (int q = 0; q < CAND_T; ++q) tv[q] = NEG_INF, tj[q] = 0x7fffffff;
  double lb = NEG_INF;
  auto push = [&](double v, int j) {
    if (better(v, j, tv[CAND_T - 1], tj[CAND_T - 1])) {
      lb = fmax(lb, tv[CAND_T - 1]);
      tv[CAND_T - 1] = v;
      tj[CAND_T - 1] = j;
#pragma unroll
      for (int q = CAND_T - 1; q > 0; --q) {
        if (better(tv[q], tj[q], tv[q - 1], tj[q - 1])) {
          const double xv = tv[q];
          tv[q] = tv[q - 1];
          tv[q - 1] = xv;
          const int xj = tj[q];
          tj[q] = tj[q - 1];
          tj[q - 1] = xj;
        }
      }
    } else {
      lb = fmax(lb, v);
    }
  };
  if (s.vec) {  // j0 is even
    constexpr int S = 2 * NT;
    int j = j0 + 2 * tid;
    for (; j + 3 * S + 1 < j1; j += 4 * S) {
      double2 wv[4], pv[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) wv[u] = __ldg(reinterpret_cast<const double2*>(w + j + u * S));
#pragma unroll
      for (int u = 0; u < 4; ++u) pv[u] = ldm(reinterpret_cast<const double2*>(s.price + j + u * S));
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        push(wv[u].x - pv[u].x, j + u * S);
        push(wv[u].y - pv[u].y, j + u * S + 1);
      }
    }
    for (; j < j1; j += S) {
      push(__ldg(w + j) - ldm(s.price + j), j);
      if (j + 1 < j1) push(__ldg(w + j + 1) - ldm(s.price + j + 1), j + 1);
    }
  } else {
    for (int j = j0 + tid; j < j1; j += NT) push(__ldg(w + j) - ldm(s.price + j), j);
  }
#pragma unroll
  for (int q = 0; q < CAND_T; ++q) {
    cand_v[tid * CAND_T + q] = tv[q];
    cand_j[tid * CAND_T + q] = tj[q];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) lb = fmax(lb, __shfl_xor_sync(0xffffffffu, lb, o));
  if ((tid & 31) == 0) red[tid >> 5] = lb;
  __syncthreads();
  for (int k = 2; k <= NC; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int idx = tid; idx < NC; idx += NT) {
        const int ixj = idx ^ j;
        if (ixj > idx) {
          const double va = cand_v[idx], vb = cand_v[ixj];
          const int ja = cand_j[idx], jb = cand_j[ixj];
          const bool a_first = better(va, ja, vb, jb);
          const bool desc = (idx & k) == 0;
          if (desc ? !a_first : a_first) {
            cand_v[idx] = vb;
            cand_v[ixj] = va;
            cand_j[idx] = jb;
            cand_j[ixj] = ja;
          }
        }
      }
      __syncthreads();
    }
  }
  double bound = NEG_INF;
#pragma unroll
  for (int q = 0; q < NT / 32; ++q) bound = fmax(bound, red[q]);
  bound = fmax(bound, cand_v[kc]);  // kc < NC always (kc <= LIST_K < NC)
  for (int q = tid; q < kc; q += NT) {
    const int j = cand_j[q];
    const bool real = j != 0x7fffffff;  // chunks shorter than kc pad their slots with a never-chosen entry
    s.lj[(int64_t)i * LIST_K + c * kc + q] = real ? j : j0;
    s.lw[(int64_t)i * LIST_K + c * kc + q] = real ? __ldg(w + j) : NEG_INF;
  }
  Top2 t;
  t.v1 = cand_v[0];
  t.j1 = cand_j[0] == 0x7fffffff ? -1 : cand_j[0];
  t.v2 = cand_v[1];
  t.j2 = cand_j[1] == 0x7fffffff ? -1 : cand_j[1];
  *bound_out = bound;
  __syncthreads();
  return t;
}

// Plain row sweep (no candidate list): exact top-2 of W[i,:] - price by an NT-thread CTA.  Used for the
// square (eps-scaling) problems, where every price inflates and lists would be rebuilt on every bid.
template <int NT>
__device__ Top2 full_scan_top2(const LapState& s, int i, Top2* wred) {
  const int tid = threadIdx.x;
  const double* w = s.W + (int64_t)i * s.ldw;
  Top2 t{NEG_INF, NEG_INF, -1, -1};
  auto push = [&](double v, int j) {  // candidates arrive in increasing j per thread: strict '>' keeps ties deterministic
    if (v > t.v1) {
      t.v2 = t.v1, t.j2 = t.j1, t.v1 = v, t.j1 = j;
    } else if (v > t.v2) {
      t.v2 = v, t.j2 = j;
    }
  };
  if (s.vec) {
    constexpr int S = 2 * NT;
    int j = 2 * tid;
    for (; j + 3 * S + 1 < s.m; j += 4 * S) {
      double2 wv[4], pv[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) wv[u] = __ldg(reinterpret_cast<const double2*>(w + j + u * S));
#pragma unroll
      for (int u = 0; u < 4; ++u) pv[u] = ldm(reinterpret_cast<const double2*>(s.price + j + u * S));
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        push(wv[u].x - pv[u].x, j + u * S);
        push(wv[u].y - pv[u].y, j + u * S + 1);
      }
    }
    for (; j < s.m; j += S) {
      push(__ldg(w + j) - ldm(s.price + j), j);
      if (j + 1 < s.m) push(__ldg(w + j + 1) - ldm(s.price + j + 1), j + 1);
    }
  } else {
    for (int j = tid; j < s.m; j += NT) push(__ldg(w + j) - ldm(s.price + j), j);
  }
  t = top2_warp_reduce(t);
  if ((tid & 31) == 0) wred[tid >> 5] = t;
  __syncthreads();
  Top2 r = wred[0];
#pragma unroll
  for (int q = 1; q < NT / 32; ++q) top2_merge(r, wred[q]);
  __syncthreads();
  return r;
}

// ------------------------------------------------------------------------------------------------
// Phase A, wide part.  One cooperative launch runs the rounds of ONE eps phase for as long as more
// than `tail_nu` persons are bidding; the narrow remainder of the phase is handed to the single-CTA
// kernel below (the bidder count never grows within a phase: every bidder either wins and evicts at
// most one owner, or re-queues itself).  eps = eps_factor * (cost range); eps_factor == 0 is the
// final, exact, naive phase.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void wide_finalize_bid(const LapState& s, int k, int i, Top2 t, double eps) {
  int j = t.j1;
  if (eps == 0.0 && t.j2 >= 0 && t.v1 == t.v2 && ldm(&s.owner[j]) >= 0 && ldm(&s.owner[t.j2]) < 0) j = t.j2;  // exact tie
  const double gamma = (t.j2 >= 0 ? (t.v1 - t.v2) : 0.0) + eps;
  s.bj[k] = j;
  s.gam[k] = gamma;
  s.bval[k] = (j == t.j1) ? t.v1 : t.v2;
  atomicMax(&s.key[j], pack_bid(gamma, i));
}

__global__ void __launch_bounds__(LAP_THREADS) lap_auction_kernel(LapState s, double eps_factor, int phase_idx,
                                                                  int tail_nu, int use_lists, int list_min_nu,
                                                                  int aug_nu, int rank_select, int only_fallback) {
  LapCtrl* ctrl = s.ctrl;
  if (ctrl->finished || s.flags[0]) return;  // uniform: written only at the very end of earlier launches
  // only_fallback: this launch stands behind the asynchronous kernel and runs only if that one met an exact tie
  // (which optimum it would pick depends on timing: the step is redone here, reproducibly)
  if (only_fallback && !ctrl->a_fallback) return;
  const int first_phase = phase_idx == 0;
  GridBarrier grid{&ctrl->barrier[phase_idx], 0u};
  __shared__ double cand_v[LAP_THREADS * CAND_T];
  __shared__ int cand_j[LAP_THREADS * CAND_T];
  __shared__ double red[LAP_WARPS];
  __shared__ Top2 wred[LAP_WARPS];
  __shared__ int s_last;  // this CTA finished the last chunk of a split row
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const int gtid = blockIdx.x * blockDim.x + tid;
  const int gthreads = gridDim.x * blockDim.x;

  const double range = ctrl->wmax - ctrl->wmin;
  const double eps = (eps_factor > 0.0 && range > 0.0) ? eps_factor * range : 0.0;
  long long rounds = 0, bids = 0, sweeps = 0;
  long long tph[4] = {0, 0, 0, 0};
  bool guard_hit = false;

  // (re)start the phase with everybody unassigned; prices (and candidate lists) are kept from the previous phase
  for (int j = gtid; j < s.m; j += gthreads) {
    if (first_phase) s.price[j] = 0.0;
    s.owner[j] = -1;
    s.key[j] = 0ull;
    if (s.pcls != nullptr) s.ocls[j] = -1;
  }
  for (int i = gtid; i < s.n; i += gthreads) {
    s.col4row[i] = -1;
    s.un[0][i] = i;
    s.done[i] = 0;
    if (first_phase)
      s.lvalid[i] = 0;
    else if (s.lvalid[i] != 0)
      s.lvalid[i] = 1;  // round stamps of the previous launch (see the bidding stage) -> plain "valid"
    if (s.pcls != nullptr) s.clevel[i] = ~0ull;
  }
  if (gtid == 0) {
    ctrl->cnt[0] = s.n;
    ctrl->cnt[1] = 0;
    ctrl->progress[0] = 0;
    ctrl->progress[1] = 0;
    ctrl->nfail[0] = 0;
    ctrl->nfail[1] = 0;
    ctrl->nhold[0] = 0;
    ctrl->nhold[1] = 0;
  }
  grid.sync();
  int cur = 0;
  int parity = 0;
  int nu = s.n;
  bool stalled = false;

  // the exact (eps = 0) phase may hand its last aug_nu persons straight to the augmenting-path kernel
  const int stop_nu = eps == 0.0 ? (aug_nu > tail_nu ? aug_nu : tail_nu) : max(tail_nu, s.scale_cut_nu);
  for (;;) {
    const long long t0 = clock64();
    // (every list that was stamped "being rebuilt" has been rebuilt by the time the loop is left)
    if (nu <= stop_nu || stalled) break;
    if (rounds >= s.max_rounds) {
      guard_hit = true;
      break;
    }
    const int* un = s.un[cur];
    const bool lists_round = use_lists && nu >= list_min_nu;
    const int rnd = (int)rounds;
    int* const failp = s.fail + (size_t)parity * s.n;  // double buffered: the rebuild above reads last round's
    if (lists_round) {
      // ---- bidding from the candidate lists, one warp per bidder.  A bidder whose list cannot certify its top-2
      //      sits out (bj = -1, re-queued by the resolution below) until its list has been rebuilt at the top of the
      //      next round: a Jacobi auction may let any subset of the unassigned persons bid.  lvalid[i] = v means
      //      "usable from round v - 1 on" (1 = always): the failing warp stamps round + 2.
      //      (The rebuild used to be a stage of its own between two barriers, followed by the failed bidders' bids:
      //      ~8 us of every wide round.)
      for (int k = (blockIdx.x * LAP_WARPS + warp); k < nu; k += gridDim.x * LAP_WARPS) {
        const int i = ldm(&un[k]);
        const int lv = ldm(&s.lvalid[i]);
        if (lv > rnd + 1) {  // list being rebuilt: hold
          if (lane == 0) {
            s.bj[k] = -1;
            atomicAdd(&ctrl->nhold[parity], 1);  // a pending rebuild is progress (no false "stalled")
          }
          continue;
        }
        bool ok = false;
        Top2 t;
        ok = list_bid<true>(s, i, lane, t);
        if (lane == 0) {
          if (ok) {
            wide_finalize_bid(s, k, i, t, eps);
          } else {
            s.bj[k] = -1;
            s.lvalid[i] = rnd + 3;
            lb_keys(s)[i] = 0ull;  // below every bound: the chunks of the rebuild fold theirs in by atomic max
            failp[atomicAdd(&ctrl->nfail[parity], 1)] = i;
          }
        }
      }
    } else {
      // ---- bidding without lists: every bidder's row is swept; with few bidders each row is split over
      //      ~grid/nu CTAs and merged by the last CTA to finish, so the round costs one memory latency
      // few bidders: split every row over ~grid/nu CTAs so the round costs one memory latency, not a row sweep
      int nch = 1;
      if (nu < (int)gridDim.x) nch = min(s.max_chunks, (int)gridDim.x / nu);
      const int chunk = (((s.m + nch - 1) / nch) + 1) & ~1;
      const long long items = (long long)nu * nch;
      for (long long item = blockIdx.x; item < items; item += gridDim.x) {
        const int k = (int)(item / nch);
        const int c = (int)(item - (long long)k * nch);
        const int i = ldm(&un[k]);
        const double* w = s.W + (int64_t)i * s.ldw;
        const int j0 = min(s.m, c * chunk);
        const int j1 = min(s.m, j0 + chunk);
        Top2 t{NEG_INF, NEG_INF, -1, -1};
        if (s.vec) {
          constexpr int S = 2 * LAP_THREADS;
          int j = j0 + 2 * tid;
          // 4 independent 128-bit load pairs in flight per thread (latency-bound when few rows are active)
          for (; j + 3 * S + 1 < j1; j += 4 * S) {
            const double2 w0 = __ldg(reinterpret_cast<const double2*>(w + j));
            const double2 w1 = __ldg(reinterpret_cast<const double2*>(w + j + S));
            const double2 w2 = __ldg(reinterpret_cast<const double2*>(w + j + 2 * S));
            const double2 w3 = __ldg(reinterpret_cast<const double2*>(w + j + 3 * S));
            const double2 p0 = ldm(reinterpret_cast<const double2*>(s.price + j));
            const double2 p1 = ldm(reinterpret_cast<const double2*>(s.price + j + S));
            const double2 p2 = ldm(reinterpret_cast<const double2*>(s.price + j + 2 * S));
            const double2 p3 = ldm(reinterpret_cast<const double2*>(s.price + j + 3 * S));
            top2_push_seq(t, w0.x - p0.x, j);
            top2_push_seq(t, w0.y - p0.y, j + 1);
            top2_push_seq(t, w1.x - p1.x, j + S);
            top2_push_seq(t, w1.y - p1.y, j + S + 1);
            top2_push_seq(t, w2.x - p2.x, j + 2 * S);
            top2_push_seq(t, w2.y - p2.y, j + 2 * S + 1);
            top2_push_seq(t, w3.x - p3.x, j + 3 * S);
            top2_push_seq(t, w3.y - p3.y, j + 3 * S + 1);
          }
          for (; j < j1; j += S) {
            if (j + 1 < j1) {
              const double2 wv = __ldg(reinterpret_cast<const double2*>(w + j));
              const double2 pv = ldm(reinterpret_cast<const double2*>(s.price + j));
              top2_push_seq(t, wv.x - pv.x, j);
              top2_push_seq(t, wv.y - pv.y, j + 1);
            } else {
              top2_push_seq(t, __ldg(w + j) - ldm(&s.price[j]), j);
            }
          }
        } else {
          for (int j = j0 + tid; j < j1; j += LAP_THREADS) top2_push_seq(t, __ldg(w + j) - ldm(&s.price[j]), j);
        }
        t = top2_warp_reduce(t);
        if ((tid & 31) == 0) wred[tid >> 5] = t;
        __syncthreads();
        if (tid == 0) {
#pragma unroll
          for (int wi = 1; wi < LAP_THREADS / 32; ++wi) top2_merge(t, wred[wi]);
          if (nch == 1) {
            wide_finalize_bid(s, k, i, t, eps);
          } else {
            const int64_t slot = (int64_t)k * nch + c;
            s.pv1[slot] = t.v1;
            s.pv2[slot] = t.v2;
            s.pj1[slot] = t.j1;
            s.pj2[slot] = t.j2;
            int prev;  // release: the partial above is visible before the count; no L1-invalidating fence
            asm volatile("atom.release.gpu.global.add.u32 %0, [%1], 1;" : "=r"(prev) : "l"(&s.done[k]) : "memory");
            s_last = (prev == nch - 1) ? 1 : 0;
          }
        }
        if (nch > 1) {  // uniform.  Last CTA of the row: lanes of warp 0 fetch the partials in parallel (see above)
          __syncthreads();
          if (s_last && warp == 0) {
            Top2 a{NEG_INF, NEG_INF, -1, -1};
            for (int cc = lane; cc < nch; cc += 32) {
              const int64_t sl = (int64_t)k * nch + cc;
              Top2 b{__ldcg(&s.pv1[sl]), __ldcg(&s.pv2[sl]), __ldcg(&s.pj1[sl]), __ldcg(&s.pj2[sl])};
              top2_merge(a, b);
            }
            a = top2_warp_reduce(a);
            if (lane == 0) {
              s.done[k] = 0;
              wide_finalize_bid(s, k, i, a, eps);
            }
          }
        }
        __syncthreads();
      }
      if (blockIdx.x == 0 && tid == 0) sweeps += nu;
    }
    const long long t1 = clock64();
    grid.sync();
    const long long t2 = clock64();
    // failures of this round's bidding stage (0 in the rounds without lists)
    const int nfail = lists_round ? ldm(&ctrl->nfail[parity]) : 0;
    const int nhold = lists_round ? ldm(&ctrl->nhold[parity]) : 0;
    if (lists_round && gtid == 0) {  // the other parity's counters are next touched behind this round's second barrier
      ctrl->nfail[parity ^ 1] = 0;
      ctrl->nhold[parity ^ 1] = 0;
    }
    // ---- plan the rebuild of the failed lists.  It runs behind this round's SECOND barrier, next to the coming
    //      round's bidding stage (the owners hold): between that barrier and the next first barrier no price changes,
    //      so the rebuilt lists are deterministic, and the sweep shares a barrier interval with the bidding instead of
    //      having one of its own.  With at least a grid-full of failures one CTA sweeps one row; with fewer, every row
    //      is split over nch CTAs (chunk_scan_*: one memory latency instead of one CTA streaming a whole row), dealt
    //      from the END of the grid -- bidder k is handled by CTA k / 8.  What does not depend on the prices is done
    //      between the arrival at and the wait on the second barrier, off the critical path: the person of this
    //      CTA's chunk is fetched and the chunk of its (immutable) cost row is pulled into L2.
    // chunks per failed row: up to 16 (kc = 8), as long as that keeps every CTA at <= ~2 chunks per round, the
    // chunks at >= 1024 objects and the partial slots within their arrays
    int nch = 1;
    if (nfail > 0 && s.list_k == LIST_K) {
      const int item_cap = (int)gridDim.x * s.chunk_waves;
      while (nch < 16 && 2 * nch * nfail <= item_cap && 2 * nch * nfail <= MAX_GRID_SLOTS && s.m / (2 * nch) >= 1024)
        nch *= 2;
    }
    // ---- resolution: one thread per bidder; the winner of each object applies its bid
    int* nxt = s.un[cur ^ 1];
    for (int k = gtid; k < nu; k += gthreads) {
      // two dependent L2 latencies, not three: everything that depends only on k, then everything that depends on j
      const int i = ldm(&un[k]);
      const int j = ldm(&s.bj[k]);
      const double gam = ldm(&s.gam[k]);
      const double bval = ldm(&s.bval[k]);
      if (j < 0) {  // sat the round out (list being rebuilt)
        nxt[atomicAdd(&ctrl->cnt[cur ^ 1], 1)] = i;
        continue;
      }
      const unsigned long long kj = ldm(&s.key[j]);
      const double p_old = ldm(&s.price[j]);
      const int prev = ldm(&s.owner[j]);
      bool requeue = true;
      if ((unsigned)(kj & 0xffffffffull) == (unsigned)(i + 1)) {
        const double p_new = p_old + gam;
        const double defend = class_defends<true>(s, i, prev, gam);
        if (defend > 0.0) {
          // the owner's class has settled lower: the owner raises the price to the class level and keeps the object
          s.price[j] = p_old + defend;
          s.profit[prev] = ldm(s.profit + prev) - defend;
          atomicAdd(&ctrl->progress[parity], 1);
        } else if (prev < 0 || gam > GAMMA_TIE) {
          if (prev >= 0) {
            s.col4row[prev] = -1;
            nxt[atomicAdd(&ctrl->cnt[cur ^ 1], 1)] = prev;
          }
          s.owner[j] = i;
          if (s.pcls != nullptr) s.ocls[j] = __ldg(s.pcls + i);
          s.col4row[i] = j;
          s.price[j] = p_new;
          // profit := value of the owned object at its new price.  bval = fl(W - p_old) from the scan;
          // (bval + p_old) - p_new reproduces W - p_new to rounding, keeping the matched edge tight
          // at the 1-ulp level without re-reading W.
          const double prof = (bval + p_old) - p_new;
          s.profit[i] = prof;
          class_settle(s, i, prof);
          atomicAdd(&ctrl->progress[parity], 1);
          requeue = false;
        }
        s.key[j] = 0ull;
      }
      if (requeue) nxt[atomicAdd(&ctrl->cnt[cur ^ 1], 1)] = i;
    }
    rounds++;
    bids += nu;
    const long long t3 = clock64();
    grid.arrive();
    const int rb = (int)gridDim.x - 1 - (int)blockIdx.x;  // reversed CTA index
    const int rb_chunk = (((s.m + nch - 1) / nch) + 1) & ~1;
    int rb_i = -1;  // person whose chunk (item rb) this CTA sweeps after the second barrier
    if (nch > 1 && rb < nfail * nch) {
      rb_i = ldm(&failp[rb / nch]);
      const int c = rb - (rb / nch) * nch;
      const int j0 = min(s.m, c * rb_chunk), j1 = min(s.m, j0 + rb_chunk);
      const char* row = reinterpret_cast<const char*>(s.W + (int64_t)rb_i * s.ldw);
      for (int64_t off = ((int64_t)j0 * 8 & ~127ll) + (int64_t)tid * 128; off < (int64_t)j1 * 8; off += LAP_THREADS * 128)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(row + off));
    }
    grid.wait();
    // loop control of the coming round, requested before the sweep (their latency hides behind its loads)
    const int nu_next = ldm(&ctrl->cnt[cur ^ 1]);
    const int prog = ldm(&ctrl->progress[parity]);
    if (nfail > 0) {
      // ---- rebuild of the lists that failed in this round's bidding stage (planned above)
      if (nch == 1) {
        for (int f = rb; f < nfail; f += gridDim.x) {
          const int i = ldm(&failp[f]);
          (void)full_scan_build<LAP_THREADS, true>(s, i, cand_v, cand_j, red, false);  // lvalid keeps its stamp
          if (tid == 0) sweeps++;
        }
      } else {
        // nch * nfail <= grid * chunk_waves items: one chunk per CTA with the default chunk_waves = 1 (the first
        // item's person was fetched before the barrier)
        const int kc = LIST_K / nch;
        const int items = nfail * nch;
        for (int item = rb; item < items; item += gridDim.x) {
          const int f = item / nch, c = item - f * nch;
          const int i = item == rb ? rb_i : ldm(&failp[f]);
          const int j0 = min(s.m, c * rb_chunk), j1 = min(s.m, j0 + rb_chunk);
          double cb = NEG_INF;  // needed in thread 0
          if (kc <= 16)
            (void)chunk_scan_select<LAP_THREADS>(s, i, j0, j1, c, kc, cand_v, cand_j, red, &cb);
          else if (rank_select)
            chunk_scan_rank<LAP_THREADS>(s, i, j0, j1, c, kc, cand_v, cand_j, red, &cb);
          else
            (void)chunk_scan_build<LAP_THREADS>(s, i, j0, j1, c, kc, cand_v, cand_j, red, &cb);
          // the chunk's bound goes into the person's bound by one atomic max (no counter, no publisher: the list
          // is complete when every chunk CTA has passed the next barrier, which precedes the round it is stamped for)
          if (tid == 0) {
            atomicMax(lb_keys(s) + i, f64_sortable(cb));
            if (c == 0) sweeps++;
          }
        }
      }
    }
    const long long t4 = clock64();
    tph[0] += t1 - t0;
    tph[1] += t2 - t1;
    tph[2] += t3 - t2;
    tph[3] += t4 - t3;
    if (gtid == 0) {
      ctrl->cnt[cur] = 0;  // becomes the "next" list of the coming round
      ctrl->progress[parity ^ 1] = 0;
    }
    cur ^= 1;
    parity ^= 1;
    nu = nu_next;
    if (prog == 0 && nfail == 0 && nhold == 0 && nu > 0) stalled = true;  // (a requested / pending rebuild is progress)
  }
  if (gtid == 0) {
    ctrl->cur = cur;
    ctrl->eps = eps;
    const bool aborted = stalled || guard_hit;
    if (eps == 0.0) {
      // final phase: either done, or the narrow kernel finishes it, or the augmentation kernel must
      const bool to_aug = !aborted && nu > 0 && nu <= aug_nu;
      ctrl->in_tail = (!aborted && nu > 0 && !to_aug) ? 1 : 0;
      ctrl->stalled = ((aborted || to_aug) && nu > 0) ? 1 : 0;
      ctrl->finished = (aborted || nu == 0 || to_aug) ? 1 : 0;
    } else {
      // scaling phase: its only product is the price vector; a guard hit just ends it early
      ctrl->in_tail = (!aborted && nu > s.scale_cut_nu && s.scale_tail_rounds > 0) ? 1 : 0;
    }
    atomicAdd(reinterpret_cast<unsigned long long*>(&s.counters->rounds), (unsigned long long)rounds);
    atomicAdd(reinterpret_cast<unsigned long long*>(&s.counters->bids), (unsigned long long)bids);
    for (int q = 0; q < 4; ++q) s.counters->t_phase[q] += tph[q];
  }
  // row sweeps are counted per CTA (thread 0 of each)
  if (tid == 0 && sweeps > 0)
    atomicAdd(reinterpret_cast<unsigned long long*>(&s.counters->bytes), (unsigned long long)sweeps * s.m * 8ull);
}

// ------------------------------------------------------------------------------------------------
// Phase A, wide part, ASYNCHRONOUS form (n < m, eps = 0, candidate lists, no classes).
//
// The round-synchronous kernel above spends ~15 us per round on two grid barriers and the slowest list rebuild
// whatever the bidder count; the wide rounds of a 10k x 50k step are ~1 500 such rounds.  An auction does not need
// rounds (Bertsekas' asynchronous auction): a bid computed from prices that may already be out of date is still a
// valid bid as long as (a) the prices it saw were not HIGHER than the true ones -- prices only rise, so every value it
// computed is an upper bound of the true value -- and (b) it is applied only if it still raises the object's price.
// Here every CTA is a worker that owns one unassigned person at a time and FOLLOWS THE CHAIN:
//   take the next person that has never bid (atomic counter) -> warp 0 bids from the candidate list (prices + owners
//   gathered from `pw`, one 16-byte {price, owner} word per object) -> if the list cannot certify its top-2 the whole
//   CTA sweeps the row and rebuilds it -> the bid is applied with ONE 128-bit compare-and-swap on pw[j] (expected = the
//   {price, owner} the bid was computed from; on a mismatch the bid is re-checked against the returned state and
//   either retried or recomputed) -> the worker carries on with the evicted owner.  The number of unassigned persons
//   never grows, so nobody is ever queued.
// Exactness: a person that wins j at level b = W_ij - v2 values j at v2 afterwards, and v2 bounds every other object's
// current value from above (listed objects: prices read <= current; unlisted: the list bound); prices only rise, an
// object once owned stays owned, unassigned objects keep price 0: the same invariants as the synchronous kernel, so the
// master/helper tail, the augmenting-path kernel and the certificate continue from its state unchanged.
// Reproducibility: a tie-free instance has ONE optimum, whatever the order of the bids.  With exact ties the optimum
// that comes out would depend on timing, so the first exact tie a worker meets (two equal best values, or a bid that
// cannot raise a price) stops the kernel and the step is redone by the synchronous kernel, whose trajectory is fixed.
// The kernel stops when at most stop_nu persons are still unassigned (or a bid budget is spent) and leaves
// price / owner / col4row / profit and the ascending list of unassigned persons behind.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool cas128(ulonglong2* addr, unsigned long long& e0, unsigned long long& e1,
                                       unsigned long long n0, unsigned long long n1) {
  unsigned long long r0, r1;
  asm volatile(
      "{\n"
      ".reg .b128 cmp, swp, res;\n"
      "mov.b128 cmp, {%2, %3};\n"
      "mov.b128 swp, {%4, %5};\n"
      "atom.relaxed.gpu.global.cas.b128 res, [%6], cmp, swp;\n"
      "mov.b128 {%0, %1}, res;\n"
      "}\n"
      : "=l"(r0), "=l"(r1)
      : "l"(e0), "l"(e1), "l"(n0), "l"(n1), "l"(addr)
      : "memory");
  const bool ok = (r0 == e0) && (r1 == e1);
  e0 = r0;
  e1 = r1;
  return ok;
}
__device__ __forceinline__ int ld_relaxed_s32(const int* p) {
  int v;
  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// A person's candidate list in registers (lane l holds entries l, l + 32, l + 64, l + 96).
struct ListRegs {
  int valid;
  double bound;
  int js[LIST_K / 32];
  double ws[LIST_K / 32];
};
__device__ __forceinline__ void load_list(const LapState& s, int i, int lane, ListRegs& L) {
  const int* lj = s.lj + (int64_t)i * LIST_K;
  const double* lw = s.lw + (int64_t)i * LIST_K;
  L.valid = ldm(&s.lvalid[i]);
  L.bound = sortable_f64(ldm(lb_keys(s) + i));
#pragma unroll
  for (int q = 0; q < LIST_K / 32; ++q) {
    L.js[q] = ldm(lj + lane + 32 * q);
    L.ws[q] = ldm(lw + lane + 32 * q);
  }
}
// Bid from a list against the packed {price, owner} words.  Returns false when the list is missing or cannot certify
// its top-2.  p1/o1, p2/o2: price and owner of t.j1 / t.j2 as read.
__device__ __forceinline__ bool list_bid_pw(const LapState& s, const ListRegs& L, int lane, Top2& out, double& p1, int& o1,
                                            double& p2, int& o2) {
  Top2 t{NEG_INF, NEG_INF, -1, -1};
  out = t;
  p1 = p2 = 0.0;
  o1 = o2 = -1;
  if (!L.valid) return false;  // never built: the slots hold garbage
  double ps[LIST_K / 32];
  int ow[LIST_K / 32];
#pragma unroll
  for (int q = 0; q < LIST_K / 32; ++q) {
    ps[q] = 0.0;
    ow[q] = -1;
    if (L.js[q] >= 0) {
      const ulonglong2 e = __ldcg(s.pw + L.js[q]);
      ps[q] = __longlong_as_double((long long)e.x);
      ow[q] = (int)(unsigned)e.y;
    }
  }
#pragma unroll
  for (int q = 0; q < LIST_K / 32; ++q)
    if (L.js[q] >= 0) top2_push(t, L.ws[q] - ps[q], L.js[q]);
  t = top2_warp_reduce(t);
  out = t;
  // price / owner of the two winners, from the lanes that hold them
  double mp1 = 0.0, mp2 = 0.0;
  int mo1 = -1, mo2 = -1;
  bool h1 = false, h2 = false;
#pragma unroll
  for (int q = 0; q < LIST_K / 32; ++q) {
    if (L.js[q] >= 0 && L.js[q] == t.j1) h1 = true, mp1 = ps[q], mo1 = ow[q];
    if (L.js[q] >= 0 && L.js[q] == t.j2) h2 = true, mp2 = ps[q], mo2 = ow[q];
  }
  const unsigned b1 = __ballot_sync(0xffffffffu, h1), b2 = __ballot_sync(0xffffffffu, h2);
  if (b1 != 0u) {
    const int src = __ffs(b1) - 1;
    p1 = __shfl_sync(0xffffffffu, mp1, src);
    o1 = __shfl_sync(0xffffffffu, mo1, src);
  }
  if (b2 != 0u) {
    const int src = __ffs(b2) - 1;
    p2 = __shfl_sync(0xffffffffu, mp2, src);
    o2 = __shfl_sync(0xffffffffu, mo2, src);
  }
  return t.j1 >= 0 && t.j2 >= 0 && t.v2 >= L.bound;
}

template <int NT>
__global__ void __launch_bounds__(NT) lap_async_kernel(LapState s, int stop_nu, int max_nu, int cont, int fallback_ok) {
  LapCtrl* ctrl = s.ctrl;
  if (ctrl->finished || s.flags[0]) return;  // uniform
  GridBarrier grid{&ctrl->barrier[MAX_PHASES - 1 - cont], 0u};  // (slot 0: the synchronous kernel's launch; a launch
                                                                    // that continues another one has a counter of its own)
  __shared__ double cand_v[NT * CAND_T];
  __shared__ int cand_j[NT * CAND_T];
  __shared__ double red[(NT / 32)];
  __shared__ int s_person, s_res;
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const int gtid = blockIdx.x * blockDim.x + tid;
  const int gthreads = gridDim.x * blockDim.x;
  const unsigned long long FREE = 0xffffffffull;  // owner word of a free object (-1 as u32)

  // cont = 0: the kernel starts the step (everybody unassigned, prices 0).  cont = 1: it takes over from the
  // round-synchronous kernel, which ran the rounds with thousands of bidders (there the work per round, not the two
  // barriers, is what a round costs): prices / owners are packed, the persons to place are its bidder list.
  if (cont && !ctrl->in_tail) return;  // uniform (written at the end of the previous launch)
  const int* worklist = cont ? s.un[ctrl->cur] : nullptr;
  const int nwork = cont ? ctrl->cnt[ctrl->cur] : s.n;
  if (cont) {
    for (int j = gtid; j < s.m; j += gthreads)
      s.pw[j] = make_ulonglong2((unsigned long long)__double_as_longlong(s.price[j]), (unsigned long long)(unsigned)s.owner[j]);
  } else {
    for (int j = gtid; j < s.m; j += gthreads) {
      s.pw[j] = make_ulonglong2(0ull, FREE);  // price +0.0, nobody
      s.price[j] = 0.0;
      s.owner[j] = -1;
      s.key[j] = 0ull;
    }
    for (int i = gtid; i < s.n; i += gthreads) {
      s.col4row[i] = -1;
      s.lvalid[i] = 0;
      s.done[i] = 0;
    }
  }
  if (gtid == 0) {
    ctrl->aq_head = 0u;
    ctrl->a_active = nwork;
    ctrl->a_stop = nwork <= stop_nu ? 1 : 0;
    ctrl->a_parked = 0;
    ctrl->a_bids = 0ull;
    ctrl->a_guard = 0;
    ctrl->a_tie = 0;
    ctrl->a_fallback = 0;
    ctrl->a_hops = 0ull;
    unsigned long long now;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
    ctrl->a_t0 = now;
  }
  grid.sync();
  unsigned long long T0 = 0;
  if (gtid == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(T0));

  // One CTA = one worker.  It takes the next person that has never bid (an atomic counter over 0 .. n-1) and FOLLOWS
  // THE CHAIN: when its bid evicts an owner, the worker carries on with the evicted person itself -- the number of
  // unassigned persons never grows, so nobody ever has to be queued, and a hop of a chain costs one list bid + one
  // compare-and-swap (a hand-over through a queue cost as much again: measured 23-30 ms -> see DESIGN for the C5 step).
  // Warp 0 bids from the list; a list that cannot certify its top-2 is rebuilt by the whole CTA (a single warp needs
  // ~200 dependent load batches for a 400 KB row: measured, the kernel was then no faster than the synchronous one).
  long long bids = 0, scans = 0;
  const long long max_bids = 1000000ll + 1000ll * s.n;
  for (;;) {
    if (tid == 0) {
      int i = -1;
      if (ld_relaxed_s32(&ctrl->a_stop) == 0) {
        const unsigned h = atomicAdd(&ctrl->aq_head, 1u);
        if (h < (unsigned)nwork) i = cont ? ldm(worklist + h) : (int)h;
      }
      s_person = i;
    }
    __syncthreads();
    int i = s_person;
    if (i < 0) break;
    // ---- bid until the chain ends on a free object, the person is parked on an exact tie, or the kernel stops.
    //      Warp 0 runs the hops of the chain by itself; the CTA only meets when a list has to be rebuilt.
    int fails = 0, last_scanned = -1;
    for (;;) {
      if (warp == 0) {
        int res;  // -1 = chain ended; -3 = rebuild the list of s_person
        int tie_tries = 0;
        ListRegs L, N;
        bool have = false;  // L already holds person i's list (fetched speculatively, see below)
        for (;;) {
          Top2 t;
          double p1, p2;
          int o1, o2;
          res = -1;  // (>= 0: placed, carry on with this evicted person; -2 = bid again)
          if (!have) load_list(s, i, lane, L);
          have = false;
          const bool ok = list_bid_pw(s, L, lane, t, p1, o1, p2, o2);
          // The person this bid will evict, if it is applied, is the owner just read: request ITS list now, so that
          // the loads travel while the compare-and-swap does (a hop of a chain is then two memory latencies, not
          // three).  Nobody can be rebuilding that list: its person is assigned until this very bid evicts it.
          const int spec = ok ? ((t.v1 == t.v2 && o1 >= 0 && o2 < 0) ? -1 : o1) : -1;
          if (spec >= 0) load_list(s, spec, lane, N);
          // ... and only a compare-and-swap that succeeds at the first attempt proves it: the word of the object was
          // unchanged from the gather to the swap, so that person held it all the time (taking an owned object back
          // raises its price).  After a retry the person may have been evicted, had its list rebuilt under these very
          // loads, and come back: the speculative copy is then dropped.
          int spec_ok = 0;
          if (!ok) {
            res = -3;
          } else if (lane == 0) {
            int j = t.j1, own_read = o1;
            double p_read = p1;
            if (t.v1 == t.v2 && o1 >= 0 && o2 < 0) {
              // two equal best values, one of the objects free: which of several optima comes out would depend on
              // timing from here on.  Stop; the round-synchronous kernel redoes the step reproducibly.
              atomicExch(&ctrl->a_tie, 1);
              atomicExch(&ctrl->a_stop, 1);
              j = t.j2, own_read = o2, p_read = p2;  // exact tie: take the free one
            }
            const double level = p_read + (t.v1 - t.v2);  // the price up to which i prefers j to everything else
            unsigned long long e0 = (unsigned long long)__double_as_longlong(p_read), e1 = (unsigned long long)(unsigned)own_read;
            bool first = true, parked = false, placed = false;
            int prev = -1;
            for (;;) {
              const double p_cur = __longlong_as_double((long long)e0);
              const int own_cur = (int)(unsigned)e1;
              if (own_cur >= 0 && !(level - p_cur > GAMMA_TIE)) {
                parked = first;  // the state the bid was computed from: an exact tie; a newer state: bid again
                break;
              }
              const double p_new = level > p_cur ? level : p_cur;  // (a free object keeps its price on a tie)
              if (cas128(s.pw + j, e0, e1, (unsigned long long)__double_as_longlong(p_new), (unsigned long long)(unsigned)i)) {
                prev = own_cur;
                placed = true;
                spec_ok = first ? 1 : 0;
                // the sweeps' copy of the price: prices are >= 0, so their bit patterns order like the values and an
                // atomic max keeps the copy monotone even when two winners' updates arrive out of order
                atomicMax(reinterpret_cast<unsigned long long*>(s.price + j), (unsigned long long)__double_as_longlong(p_new));
                break;
              }
              first = false;
            }
            bids++;
            atomicAdd(&ctrl->a_hops, 1ull);  // (fire and forget; read by the debug time line only)
            if (placed) {
              res = prev;  // -1: the chain ended on a free object
              if (prev < 0) {
                const int left = atomicSub(&ctrl->a_active, 1) - 1;
                if (left <= stop_nu) atomicExch(&ctrl->a_stop, 1);
                if (left == stop_nu || (left >= 64 && left <= 4096 && (left & (left - 1)) == 0)) {
                  unsigned long long now;
                  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                  const int slot = left == stop_nu ? 7 : 12 - (31 - __clz(left));  // 4096 -> 0 ... 64 -> 6
                  s.counters->a_ts[slot] = (long long)(now - ctrl->a_t0);
                  s.counters->a_hops[slot] = (long long)ctrl->a_hops;
                }
              }
            } else if (parked && ++tie_tries <= 32) {
              // the bid cannot raise the price (exact or near tie on an owned object).  Mostly transient: the prices
              // around it are moving.  Bid again a little later (the synchronous kernel re-queues such a bidder too).
              res = -2;
              __nanosleep(400);
            } else if (parked) {
              // a standing tie.  One or two of them occur in tie-free instances too (two values that are equal to the
              // last bit while nothing around them moves any more): the person is left to the tail, which ends in the
              // augmenting-path kernel if the tie is still there.  Many of them mean duplicated cells: redo the step
              // reproducibly.
              res = -1;
              if (atomicAdd(&ctrl->a_parked, 1) + 1 > 4) atomicExch(&ctrl->a_tie, 1), atomicExch(&ctrl->a_stop, 1);
              if (atomicSub(&ctrl->a_active, 1) - 1 <= stop_nu) atomicExch(&ctrl->a_stop, 1);
            } else {
              res = -2;
            }
            if ((bids & 63) == 0) {
              const unsigned long long tot = atomicAdd(&ctrl->a_bids, 64ull) + 64ull;
              if ((long long)tot > max_bids) atomicExch(&ctrl->a_guard, 1), atomicExch(&ctrl->a_stop, 1);
            }
            // (a worker in the middle of a chain leaves its person unassigned when the kernel stops: the epilogue finds it)
            if (res != -1 && ld_relaxed_s32(&ctrl->a_stop) != 0) res = -1;
          }
          res = __shfl_sync(0xffffffffu, res, 0);
          spec_ok = __shfl_sync(0xffffffffu, spec_ok, 0);
          if (res >= 0) {
            if (res == spec && spec_ok) L = N, have = true;
            i = res, tie_tries = 0;
          }
          if (res == -1 || res == -3) break;
        }
        if (lane == 0) s_res = res, s_person = i;
      }
      __syncthreads();
      const int res = s_res;
      i = s_person;
      __syncthreads();  // (s_res / s_person are rewritten by the next attempt)
      if (res != -3) break;
      fails = (i == last_scanned) ? fails + 1 : 1;
      last_scanned = i;
      if (fails > 8 || ld_relaxed_s32(&ctrl->a_stop) != 0) {
        // prices of its candidates keep moving under the sweeps (or the kernel has stopped): leave it to the tail
        if (tid == 0 && fails > 8) {
          atomicAdd(&ctrl->a_parked, 1);
          if (atomicSub(&ctrl->a_active, 1) - 1 <= stop_nu) atomicExch(&ctrl->a_stop, 1);
        }
        break;
      }
      (void)full_scan_build<NT, true>(s, i, cand_v, cand_j, red);
      __threadfence();  // the list is read by whichever CTA handles this person next
      scans++;
    }
  }
  unsigned long long T1 = 0, T2 = 0;
  if (gtid == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(T1));
  __syncthreads();
  grid.sync();
  if (gtid == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(T2));
  // ---- epilogue: unpack the object state, derive the person state from it
  if (cont) {
    for (int i = gtid; i < s.n; i += gthreads) s.col4row[i] = -1;
    grid.sync();
  }
  for (int j = gtid; j < s.m; j += gthreads) {
    const ulonglong2 e = __ldcg(s.pw + j);
    const double p = __longlong_as_double((long long)e.x);
    const int own = (int)(unsigned)e.y;
    s.price[j] = p;
    s.owner[j] = own;
    if (own >= 0) {
      s.col4row[own] = j;
      s.profit[own] = __ldg(s.W + (int64_t)own * s.ldw + j) - p;
    }
  }
  if (tid == 0 && (bids | scans) != 0) {
    atomicAdd(reinterpret_cast<unsigned long long*>(&s.counters->bids), (unsigned long long)bids);
    atomicAdd(reinterpret_cast<unsigned long long*>(&s.counters->bytes), (unsigned long long)scans * s.m * 8ull);
  }
  grid.sync();
  if (blockIdx.x == 0) {  // ascending list of the unassigned persons
    __shared__ int s_wsum[(NT / 32)];
    __shared__ int s_base;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int i0 = 0; i0 < s.n; i0 += NT) {
      const int i = i0 + tid;
      const bool un = i < s.n && ldm(&s.col4row[i]) < 0;
      const unsigned bal = __ballot_sync(0xffffffffu, un);
      if (lane == 0) s_wsum[warp] = __popc(bal);
      __syncthreads();
      int off = s_base;
      for (int wq = 0; wq < warp; ++wq) off += s_wsum[wq];
      if (un) s.un[0][off + __popc(bal & ((1u << lane) - 1u))] = i;
      __syncthreads();
      if (tid == 0) {
        int tot = 0;
        for (int wq = 0; wq < (NT / 32); ++wq) tot += s_wsum[wq];
        s_base += tot;
      }
      __syncthreads();
    }
    if (tid == 0) {
      const int nu = s_base;
      // exact ties, or the bid budget is spent (no instance measured comes near it): the synchronous kernel redoes the
      // step (no such fallback behind a hand-over from the synchronous kernel)
      const bool tie = fallback_ok && (ctrl->a_tie != 0 || ctrl->a_guard != 0) && nu > 0;
      ctrl->a_fallback = tie ? 1 : 0;
      const bool aborted = (ctrl->a_guard != 0 || nu > max_nu) && !tie;
      ctrl->cnt[0] = nu;
      ctrl->cnt[1] = 0;
      ctrl->cur = 0;
      ctrl->eps = 0.0;
      ctrl->in_tail = (!aborted && !tie && nu > 0) ? 1 : 0;
      ctrl->stalled = (aborted && nu > 0) ? 1 : 0;
      ctrl->finished = (aborted || nu == 0) ? 1 : 0;
      atomicAdd(reinterpret_cast<unsigned long long*>(&s.counters->rounds), 1ull);
      unsigned long long T3;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(T3));
      // (ns) bidding until CTA 0 saw the stop flag, drain of the other workers, epilogue; persons parked
      s.counters->t_phase[0] += (long long)(T1 - T0);
      s.counters->t_phase[1] += (long long)(T2 - T1);
      s.counters->t_phase[2] += (long long)(T3 - T2);
      s.counters->t_phase[3] += ctrl->a_parked;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Phase A, narrow part: ONE CTA runs the rounds with <= TAIL_NU bidders.  A round is: 16 warps bid
// from candidate lists (price gathers served by this SM's L1/L2), the few whose list fails get a
// CTA-wide row sweep, the first TAIL_NU threads resolve winners in shared memory and apply them to
// the global state -- which only this CTA touches for the rest of the phase, so plain loads/stores
// ordered by __syncthreads are enough.  No grid barrier, no fence: ~1 us per round.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(TAIL_THREADS, 1) lap_tail_list_kernel(LapState s) {
  LapCtrl* ctrl = s.ctrl;
  if (ctrl->finished || !ctrl->in_tail || s.flags[0]) return;
  __shared__ double cand_v[TAIL_THREADS * CAND_T];
  __shared__ int cand_j[TAIL_THREADS * CAND_T];
  __shared__ double red[TAIL_WARPS];
  __shared__ int s_list[2][TAIL_NU];
  __shared__ int s_bj[TAIL_NU];
  __shared__ double s_gam[TAIL_NU], s_bval[TAIL_NU];
  __shared__ unsigned long long s_key[TAIL_NU];
  __shared__ int s_fail[TAIL_NU];
  __shared__ int s_cnt[8];  // [0] failures, [1..4] per-warp next counts, [5] accepted
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const int cur_list = ctrl->cur;
  int nu = ctrl->cnt[cur_list];
  const double eps = ctrl->eps;
  if (tid < TAIL_NU) s_list[0][tid] = tid < nu ? s.un[cur_list][tid] : -1;
  __syncthreads();
  long long rounds = 0, bids = 0, sweeps = 0;
  long long tq[4] = {0, 0, 0, 0};
  int cur = 0, stalled = 0;

  auto finalize = [&](int b, Top2 t) {  // one thread records bidder b's bid in shared memory
    int j = t.j1;
    if (eps == 0.0 && t.j2 >= 0 && t.v1 == t.v2 && s.owner[j] >= 0 && s.owner[t.j2] < 0) j = t.j2;  // exact tie
    const double gamma = (t.j2 >= 0 ? (t.v1 - t.v2) : 0.0) + eps;
    s_bj[b] = j;
    s_gam[b] = gamma;
    s_bval[b] = (j == t.j1) ? t.v1 : t.v2;
    s_key[b] = pack_bid(gamma, s_list[cur][b]);
  };

  while (nu > 0) {
    if (rounds >= s.max_rounds) {
      stalled = 1;
      break;
    }
    const long long c0 = clock64();
    if (tid == 0) s_cnt[0] = 0, s_cnt[5] = 0;
    __syncthreads();
    // ---- 1. bids from the candidate lists, one warp per bidder
    for (int b = warp; b < nu; b += TAIL_WARPS) {
      const int i = s_list[cur][b];
      bool ok = false;
      Top2 t;
      ok = list_bid<false>(s, i, lane, t);
      if (lane == 0) {
        if (ok)
          finalize(b, t);
        else
          s_fail[atomicAdd(&s_cnt[0], 1)] = b;
      }
    }
    __syncthreads();
    const long long c1 = clock64();
    // ---- 2. row sweeps for the bidders whose list could not certify its top-2
    const int nfail = s_cnt[0];
    for (int f = 0; f < nfail; ++f) {
      const int b = s_fail[f];
      Top2 t = full_scan_build<TAIL_THREADS, false>(s, s_list[cur][b], cand_v, cand_j, red);
      if (s.pcls != nullptr) {  // the scan does not know the classes of similar persons: bid from the fresh list
        __syncthreads();
        if (warp == 0) list_bid<false>(s, s_list[cur][b], lane, t);
      }
      if (tid == 0) finalize(b, t);
    }
    sweeps += nfail;
    __syncthreads();
    const long long c2 = clock64();
    // ---- 3. resolution
    int person_out = -1;
    bool applied = false;
    if (tid < nu) {
      const int i = s_list[cur][tid];
      const int j = s_bj[tid];
      const unsigned long long key = s_key[tid];
      bool win = true;
      for (int q = 0; q < nu; ++q)
        if (s_bj[q] == j && s_key[q] > key) win = false;
      person_out = i;  // re-queue unless the bid is applied
      if (win) {
        const double p_old = s.price[j];
        const double p_new = p_old + s_gam[tid];
        const int prev = s.owner[j];
        const double defend = class_defends<false>(s, i, prev, s_gam[tid]);
        if (defend > 0.0) {  // the owner's class has settled lower: the owner raises the price and keeps the object
          s.price[j] = p_old + defend;
          s.profit[prev] -= defend;
          applied = true;  // (progress; the bidder is re-queued: person_out stays i)
        } else if (prev < 0 || s_gam[tid] > GAMMA_TIE) {
          applied = true;
          person_out = prev;  // the evicted owner (or -1) bids next round
          s.owner[j] = i;
          if (s.pcls != nullptr) s.ocls[j] = s.pcls[i];
          s.price[j] = p_new;
          s.col4row[i] = j;
          const double prof = (s_bval[tid] + p_old) - p_new;
          s.profit[i] = prof;
          class_settle(s, i, prof);
          if (prev >= 0) s.col4row[prev] = -1;
        }
      }
    }
    // ordered compaction of the next bidder list (threads 0..TAIL_NU-1 = warps 0..3)
    if (warp < TAIL_NU / 32) {
      const unsigned has = __ballot_sync(0xffffffffu, person_out >= 0);
      const unsigned acc = __ballot_sync(0xffffffffu, applied);
      if (lane == 0) {
        s_cnt[1 + warp] = __popc(has);
        atomicAdd(&s_cnt[5], __popc(acc));
      }
    }
    __syncthreads();
    int nu_next = 0;
    for (int w = 0; w < TAIL_NU / 32; ++w) nu_next += s_cnt[1 + w];
    if (warp < TAIL_NU / 32) {
      int off = 0;
      for (int w = 0; w < warp; ++w) off += s_cnt[1 + w];
      const unsigned has = __ballot_sync(0xffffffffu, person_out >= 0);
      if (person_out >= 0) s_list[cur ^ 1][off + __popc(has & ((1u << lane) - 1u))] = person_out;
    }
    const int accepted = s_cnt[5];
    rounds++;
    bids += nu;
    __syncthreads();
    const long long c3 = clock64();
    tq[0] += c1 - c0;
    tq[1] += c2 - c1;
    tq[2] += c3 - c2;
    cur ^= 1;
    nu = nu_next;
    if (accepted == 0 && nu > 0) {  // nobody could raise a price: exact ties -> augmentation kernel
      stalled = 1;
      break;
    }
  }
  if (tid < nu) s.un[cur_list][tid] = s_list[cur][tid];
  if (tid == 0) {
    ctrl->cnt[cur_list] = nu;
    ctrl->in_tail = 0;
    if (eps == 0.0) {
      ctrl->finished = 1;
      ctrl->stalled = (stalled && nu > 0) ? 1 : 0;
    }
    s.counters->rounds += rounds;
    s.counters->bids += bids;
    s.counters->bytes += sweeps * (long long)s.m * 8;
    for (int q = 0; q < 4; ++q) s.counters->t_phase[4 + q] += tq[q];
  }
}


__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// ------------------------------------------------------------------------------------------------
// Phase A, narrow part: one thread-block cluster runs the rounds with <= CL_NU bidders.
//
// ~93 % of all rounds have a handful of bidders and are pure latency; on the whole grid a round costs
// ~35 dependent L2 round trips + two grid barriers (~10 us).  Here the object side of the state lives in
// DISTRIBUTED SHARED MEMORY: CTA c of the cluster owns a contiguous slice of the objects (prices +
// owners in its smem), every CTA scans its slice of each bidder's cost row (the only global-memory
// round trip of the round), per-CTA (best, second) partials travel to CTA 0 with st.async
// (DSMEM store + mbarrier complete_tx: no fence, no L1 invalidate), CTA 0's first warp merges them,
// resolves the winners and multicasts a fixed-size packet (next bidder list + price/owner updates)
// back to every CTA the same way.  Global memory is only written behind the critical path, so the
// wide kernel / augmentation kernel find a consistent state afterwards.
// ------------------------------------------------------------------------------------------------
constexpr int CL_NU = 32;          // max bidders per round in the cluster kernel (one warp resolves them)
constexpr int CL_MAX_CS = 16;    // largest (non-portable) cluster

struct __align__(16) TailPart {  // 32 bytes: one CTA's best / second-best object for one bidder
  double v1, v2;                 // values (W - price)
  int j1, j2, pad0, pad1;        // objects
};
struct __align__(16) TailPacket {  // lives in CTA 0; every CTA pulls it over DSMEM once per round
  int4 ent[CL_NU];             // x: next-round bidder (or -1), y: updated object (or -1), z: its new owner
  double price[CL_NU];         // new price of ent[t].y
};
constexpr uint32_t TAIL_SIGNAL_BYTES = 8;  // per round CTA 0 pushes one 8-byte header (next count, accepted bids)

__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_smem_addr, uint32_t cta) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(cta));
  return r;
}
__device__ __forceinline__ void st_async_v2(uint32_t raddr, uint64_t a, uint64_t b, uint32_t rbar) {
  asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.v2.b64 [%0], {%1, %2}, [%3];" ::"r"(raddr),
               "l"(a), "l"(b), "r"(rbar)
               : "memory");
}
__device__ __forceinline__ void st_async_b64(uint32_t raddr, uint64_t a, uint32_t rbar) {
  asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.b64 [%0], %1, [%2];" ::"r"(raddr), "l"(a),
               "r"(rbar)
               : "memory");
}
__device__ __forceinline__ void st_async_v4i(uint32_t raddr, int4 v, uint32_t rbar) {
  asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(raddr),
               "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(rbar)
               : "memory");
}
__device__ __forceinline__ void tail_mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void tail_mbar_expect(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tail_mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "TW_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra TW_DONE;\n"
      "bra TW_LOOP;\n"
      "TW_DONE:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}

__device__ __forceinline__ double ld_cluster_f64(uint32_t raddr) {
  double v;
  asm volatile("ld.shared::cluster.f64 %0, [%1];" : "=d"(v) : "r"(raddr) : "memory");
  return v;
}
__device__ __forceinline__ int ld_cluster_s32(uint32_t raddr) {
  int v;
  asm volatile("ld.shared::cluster.s32 %0, [%1];" : "=r"(v) : "r"(raddr) : "memory");
  return v;
}
__device__ __forceinline__ int4 ld_cluster_v4(uint32_t raddr) {
  int4 v;
  asm volatile("ld.shared::cluster.v4.s32 {%0, %1, %2, %3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
               : "r"(raddr)
               : "memory");
  return v;
}

__global__ void __launch_bounds__(TAIL_THREADS, 1) lap_tail_cluster_kernel(LapState s, int mc /* objects per CTA, even */) {
  LapCtrl* ctrl = s.ctrl;
  if (ctrl->finished || !ctrl->in_tail || s.flags[0]) return;  // uniform over the cluster
  extern __shared__ __align__(16) unsigned char tsm[];
  uint32_t cta, ncta;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(cta));
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(ncta));
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;

  // ---- shared-memory carve-up (identical in every CTA, so mapa addresses line up)
  TailPart* cpart = reinterpret_cast<TailPart*>(tsm);                               // [CL_NU][CL_MAX_CS] (used in CTA 0)
  TailPacket* packet = reinterpret_cast<TailPacket*>(cpart + CL_NU * CL_MAX_CS);
  Top2* wpart = reinterpret_cast<Top2*>(packet + 1);                                // [CL_NU][TAIL_WARPS]
  int* s_list = reinterpret_cast<int*>(wpart + CL_NU * TAIL_WARPS);               // [CL_NU]
  int* s_tmp = s_list + CL_NU;                                                     // [CL_NU]
  uint32_t* s_rpkt = reinterpret_cast<uint32_t*>(s_tmp + CL_NU);                   // [CL_MAX_CS] remote header slot
  uint32_t* s_rbar = s_rpkt + CL_MAX_CS;                                           // [CL_MAX_CS] remote barB
  int* s_bj = reinterpret_cast<int*>(s_rbar + CL_MAX_CS);                          // [CL_NU] bid objects (CTA 0)
  unsigned long long* s_bkey = reinterpret_cast<unsigned long long*>(s_bj + CL_NU);  // [CL_NU] bid keys (CTA 0)
  unsigned long long* bars = s_bkey + CL_NU;                                       // barA, barB, header slot, pad
  unsigned long long* s_hdr = bars + 2;                                              // (next count) | (accepted bids) << 32
  double* sprice = reinterpret_cast<double*>(bars + 4);                              // [mc]
  int* sowner = reinterpret_cast<int*>(sprice + mc);                                 // [mc]
  const uint32_t barA = smem_addr(bars), barB = smem_addr(bars + 1);

  const int o0 = min(s.m, (int)cta * mc), o1 = min(s.m, o0 + mc);
  for (int j = o0 + tid; j < o1; j += TAIL_THREADS) {
    sprice[j - o0] = s.price[j];
    sowner[j - o0] = s.owner[j];
  }
  const int cur_list = ctrl->cur;
  int nu = ctrl->cnt[cur_list];
  if (tid < CL_NU) s_list[tid] = tid < nu ? s.un[cur_list][tid] : -1;
  const double eps = ctrl->eps;
  if (tid == 0) {
    tail_mbar_init(barA, 1);
    tail_mbar_init(barB, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid < (int)ncta) {
    s_rpkt[tid] = map_to_cta(smem_addr(s_hdr), tid);
    s_rbar[tid] = map_to_cta(barB, tid);
  }
  __syncthreads();
  if (tid == 0) {
    if (cta == 0) tail_mbar_expect(barA, ncta * (uint32_t)nu * (uint32_t)sizeof(TailPart));
    tail_mbar_expect(barB, TAIL_SIGNAL_BYTES);
  }
  const uint32_t pkt0 = map_to_cta(smem_addr(packet), 0);          // the packet, as seen from this CTA
  const uint32_t price0 = map_to_cta(smem_addr(sprice), 0) - 0u;   // CTA 0's slice base; other CTAs: + stride
  const uint32_t cta_stride = map_to_cta(smem_addr(sprice), 1 % ncta) - price0;  // shared::cluster window stride
  const uint32_t owner0 = map_to_cta(smem_addr(sowner), 0);
  // all barriers of the cluster are initialised and armed before anybody stores remotely
  asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");

  long long rounds = 0, bids = 0;
  uint32_t parity = 0;
  int stalled = 0;
  const int span = o1 - o0;

  long long tq[4] = {0, 0, 0, 0};
  while (nu > 0) {
    if (eps > 0.0 && (nu <= s.scale_cut_nu || rounds >= s.scale_tail_rounds)) break;  // (uniform over the cluster)
    const long long c0 = clock64();
    // ---- 1. scan.  G warps share one bidder's slice (G = 16, 8, 4, 2, 1 for nu = 1, 2, <=4, <=8, more), so a
    //         round costs one row-latency plus ONE warp reduction per warp whatever the bidder count.
    int G = TAIL_WARPS;
    while (G > 1 && G * nu > TAIL_WARPS) G >>= 1;
    const int per_pass = TAIL_WARPS / G;
    const int sub = (((span + G - 1) / G) + 1) & ~1;  // even sub-slice length
    const int g = warp % G;
    const int ws = min(o1, o0 + g * sub), we = min(o1, ws + sub);
    for (int b = warp / G; b < nu; b += per_pass) {
      const double* wrow = s.W + (int64_t)s_list[b] * s.ldw;
      Top2 t{NEG_INF, NEG_INF, -1, -1};
      if (s.vec) {
        // every load of a batch is issued before the first use (guards instead of a scalar tail loop: a short
        // sub-slice -- 78 objects per warp on the 10k x 10k square step -- must cost ONE memory latency, not two)
        auto batch = [&](auto depth_tag) {
          constexpr int D = decltype(depth_tag)::value;
          for (int j = ws + 2 * lane; j < we; j += D * 64) {
            double2 wv[D];
#pragma unroll
            for (int u = 0; u < D; ++u) {
              const int jj = j + u * 64;
              wv[u] = make_double2(NEG_INF, NEG_INF);
              if (jj + 1 < we)
                wv[u] = __ldg(reinterpret_cast<const double2*>(wrow + jj));
              else if (jj < we)
                wv[u].x = __ldg(wrow + jj);
            }
#pragma unroll
            for (int u = 0; u < D; ++u) {
              const int jj = j + u * 64;
              if (jj + 1 < we) {
                const double2 pv = *reinterpret_cast<const double2*>(sprice + (jj - o0));
                top2_push_seq(t, wv[u].x - pv.x, jj);
                top2_push_seq(t, wv[u].y - pv.y, jj + 1);
              } else if (jj < we) {
                top2_push_seq(t, wv[u].x - sprice[jj - o0], jj);
              }
            }
          }
        };
        if (we - ws <= 128)
          batch(std::integral_constant<int, 2>{});
        else
          batch(std::integral_constant<int, 8>{});
      } else {
        for (int j = ws + lane; j < we; j += 32) top2_push_seq(t, __ldg(wrow + j) - sprice[j - o0], j);
      }
      t = top2_warp_reduce(t);
      if (lane == 0) wpart[b * TAIL_WARPS + g] = t;
    }
    __syncthreads();
    const long long c1 = clock64();
    // ---- 2. thread b merges the 16 warp partials of bidder b and ships the CTA partial to CTA 0
    //         (G > 1: warp b reduces bidder b's G partials with the redux arg-max; G == 1: nothing to merge)
    if (G > 1 ? warp < nu : tid < nu) {
      Top2 a;
      int b;
      if (G > 1) {
        b = warp;
        a = lane < G ? wpart[b * TAIL_WARPS + lane] : Top2{NEG_INF, NEG_INF, -1, -1};
        a = top2_warp_reduce(a);
      } else {
        b = tid;
        a = wpart[b * TAIL_WARPS];
      }
      if (G == 1 || lane == 0) {
        const uint32_t dst = map_to_cta(smem_addr(&cpart[b * CL_MAX_CS + cta]), 0);
        const uint32_t rbar = map_to_cta(barA, 0);
        st_async_v2(dst, __double_as_longlong(a.v1), __double_as_longlong(a.v2), rbar);
        st_async_v2(dst + 16, ((uint64_t)(uint32_t)a.j2 << 32) | (uint32_t)a.j1, 0ull, rbar);
      }
    }
    // ---- 3. CTA 0, warp 0: merge over CTAs, resolve, multicast the round packet
    if (cta == 0 && warp == 0) {
      tail_mbar_wait(barA, parity);
      const long long c2 = clock64();
      tq[1] += c2 - c1;
      const bool live = lane < nu;
      Top2 a{NEG_INF, NEG_INF, -1, -1};
      if (nu <= 4) {  // few bidders (the usual case): one redux reduction per bidder over the CTAs' partials
        for (int bb = 0; bb < nu; ++bb) {
          Top2 q{NEG_INF, NEG_INF, -1, -1};
          if (lane < (int)ncta) {
            const TailPart& pq = cpart[bb * CL_MAX_CS + lane];
            q = Top2{pq.v1, pq.v2, pq.j1, pq.j2};
          }
          q = top2_warp_reduce(q);
          if (lane == bb) a = q;
        }
      } else if (live) {
        for (uint32_t c = 0; c < ncta; ++c) {
          const TailPart& q = cpart[lane * CL_MAX_CS + c];
          top2_merge(a, Top2{q.v1, q.v2, q.j1, q.j2});
        }
      }
      // price / owner of the two candidates live in the owning CTA's shared memory
      double p1 = 0.0, p2 = 0.0;
      int own1 = -1, own2 = -1;
      if (a.j1 >= 0) {
        const uint32_t c = (uint32_t)(a.j1 / mc), off = (uint32_t)(a.j1 - (int)c * mc);
        p1 = ld_cluster_f64(price0 + c * cta_stride + off * 8);
        own1 = ld_cluster_s32(owner0 + c * cta_stride + off * 4);
      }
      if (a.j2 >= 0 && eps == 0.0 && a.v1 == a.v2) {
        const uint32_t c = (uint32_t)(a.j2 / mc), off = (uint32_t)(a.j2 - (int)c * mc);
        p2 = ld_cluster_f64(price0 + c * cta_stride + off * 8);
        own2 = ld_cluster_s32(owner0 + c * cta_stride + off * 4);
      }
      const int i = live ? s_list[lane] : -1;
      int j = a.j1;
      double p_old = p1, bval = a.v1;
      int prev = own1;
      if (live && eps == 0.0 && a.j2 >= 0 && a.v1 == a.v2 && own1 >= 0 && own2 < 0) {  // exact tie: take the free one
        j = a.j2, p_old = p2, bval = a.v2, prev = own2;
      }
      const double gamma = (a.j2 >= 0 ? (a.v1 - a.v2) : 0.0) + eps;
      const unsigned long long key = live ? pack_bid(gamma, i) : 0ull;
      s_bj[lane] = j;
      s_bkey[lane] = key;
      __syncwarp();
      bool win = live;
      for (int q = 0; q < nu; ++q)
        if (s_bj[q] == j && s_bkey[q] > key) win = false;
      const double p_new = p_old + gamma;
      const bool applied = win && (prev < 0 || gamma > GAMMA_TIE);
      const bool has = live && (applied ? prev >= 0 : true);
      const int person_out = applied ? prev : i;
      const unsigned hmask = __ballot_sync(0xffffffffu, has);
      const int nu_next = __popc(hmask);
      const int nacc = __popc(__ballot_sync(0xffffffffu, applied));
      if (has) s_tmp[__popc(hmask & ((1u << lane) - 1u))] = person_out;
      __syncwarp();
      int4 ent;
      ent.x = lane < nu_next ? s_tmp[lane] : -1;
      ent.y = applied ? j : -1;
      ent.z = i;
      ent.w = 0;
      if (lane == 0 && nu_next > 0 && nacc > 0)
        tail_mbar_expect(barA, ncta * (uint32_t)nu_next * (uint32_t)sizeof(TailPart));  // arm the next round first
      __syncwarp();
      packet->ent[lane] = ent;
      packet->price[lane] = p_new;
      __syncwarp();
      // one 8-byte push per CTA completes its barB; the packet itself is pulled by the receivers
      if (lane < (int)ncta)
        st_async_b64(s_rpkt[lane], ((uint64_t)(uint32_t)nacc << 32) | (uint32_t)nu_next, s_rbar[lane]);
      // global state, off the critical path (read again only by later kernels)
      if (applied) {
        s.owner[j] = i;
        s.price[j] = p_new;
        s.col4row[i] = j;
        s.profit[i] = (bval + p_old) - p_new;
        if (prev >= 0) s.col4row[prev] = -1;
      }
      __syncwarp();  // orders this round's col4row stores before the next round's (different lanes, same warp)
      tq[2] += clock64() - c2;
    }
    const long long c3 = clock64();
    // ---- 4. everybody: take the packet, apply the updates that fall into the own slice
    tail_mbar_wait(barB, parity);
    tq[3] += clock64() - c3;
    tq[0] += c1 - c0;
    const unsigned long long hw = *s_hdr;
    const int4 hdr = make_int4((int)(uint32_t)hw, (int)(uint32_t)(hw >> 32), 0, 0);
    int4 ent = make_int4(-1, -1, -1, 0);
    double pnew = 0.0;
    if (tid < nu || tid < hdr.x) {  // entries beyond max(bidders, next bidders) carry nothing
      ent = ld_cluster_v4(pkt0 + (uint32_t)(tid * sizeof(int4)));
      pnew = ld_cluster_f64(pkt0 + (uint32_t)(sizeof(int4) * CL_NU + tid * sizeof(double)));
    }
    __syncthreads();  // everyone is past the wait and has its entry before the barrier is re-armed
    if (tid == 0 && hdr.x > 0 && hdr.y > 0) tail_mbar_expect(barB, TAIL_SIGNAL_BYTES);
    if (tid < CL_NU) {
      s_list[tid] = tid < hdr.x ? ent.x : -1;
      if (ent.y >= o0 && ent.y < o1) {
        sprice[ent.y - o0] = pnew;
        sowner[ent.y - o0] = ent.z;
      }
    }
    rounds++;
    bids += nu;
    parity ^= 1;
    nu = hdr.x;
    __syncthreads();
    if (hdr.y == 0 && nu > 0) {  // nobody could raise a price: exact ties -> augmentation kernel
      stalled = 1;
      break;
    }
  }
  // no CTA may leave while peers can still address its shared memory
  asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");
  if (cta == 0) {
    if (tid < nu) s.un[cur_list][tid] = s_list[tid];
    if (tid == 0) {
      ctrl->cnt[cur_list] = nu;
      ctrl->in_tail = 0;
      if (eps == 0.0) {
        ctrl->finished = 1;
        ctrl->stalled = (stalled && nu > 0) ? 1 : 0;
      }
      s.counters->rounds += rounds;
      s.counters->bids += bids;
      s.counters->bytes += bids * (long long)s.m * 8;
      for (int q = 0; q < 4; ++q) s.counters->t_phase[4 + q] += tq[q];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Phase A, narrow part, SYMMETRIC cluster form (round 2; replaces the kernel above for the square phases).
//
// The kernel above runs a round as  scan -> partials to CTA 0 -> CTA 0 resolves (two DSMEM reads of the winner's
// price / owner) -> 8-byte signal to every CTA -> every CTA pulls the packet over DSMEM  : three dependent DSMEM
// latencies behind the row scan, and seven CTAs idle while CTA 0 resolves.  Here every CTA sends its partial --
// extended by the price and owner of its two candidates, which it holds anyway -- to EVERY CTA (st.async into a
// parity-double-buffered inbox, one mbarrier per parity), and every CTA resolves the round by itself: same inputs,
// same deterministic arithmetic, same result everywhere, so there is nothing to send back.  One DSMEM latency per
// round; the next scan starts as soon as the local resolution is done.  CTA 0 alone writes the global state.
// The resolution is the one of the kernel above instruction for instruction: identical trajectories and results.
// Barrier arming without a race: a peer may be one resolution ahead and send its next partial before this CTA has
// finished the current round, so the barrier of round r + 1 is armed at the TOP of round r (no peer can send for
// r + 1 before it has this CTA's round-r partial) for nu_r slots; the bidder count never grows inside a phase, and
// the warps of the slots that have gone send filler.
// ------------------------------------------------------------------------------------------------
struct __align__(16) SymPart {  // 48 bytes: one CTA's best / second-best object for one bidder, with price and owner
  double v1, v2;
  double p1, p2;
  int j1, j2, own1, own2;
};

__global__ void __launch_bounds__(TAIL_THREADS, 1) lap_tail_sym_kernel(LapState s, int mc /* objects per CTA, even */) {
  LapCtrl* ctrl = s.ctrl;
  if (ctrl->finished || !ctrl->in_tail || s.flags[0]) return;  // uniform over the cluster
  extern __shared__ __align__(16) unsigned char tsm[];
  uint32_t cta, ncta;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(cta));
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(ncta));
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;

  // ---- shared-memory carve-up (identical in every CTA, so mapa addresses line up)
  SymPart* inbox = reinterpret_cast<SymPart*>(tsm);                                   // [2][CL_NU][CL_MAX_CS]
  Top2* wpart = reinterpret_cast<Top2*>(inbox + 2 * CL_NU * CL_MAX_CS);               // [CL_NU][TAIL_WARPS]
  int* s_list = reinterpret_cast<int*>(wpart + CL_NU * TAIL_WARPS);                   // [CL_NU]
  int* s_tmp = s_list + CL_NU;                                                         // [CL_NU]
  int* s_bj = s_tmp + CL_NU;                                                           // [CL_NU]
  int* s_ctl = s_bj + CL_NU;                                                           // [4]: next count, accepted bids
  unsigned long long* s_bkey = reinterpret_cast<unsigned long long*>(s_ctl + 4);      // [CL_NU]
  unsigned long long* bars = s_bkey + CL_NU;                                           // [2]
  double* sprice = reinterpret_cast<double*>(bars + 2);                                // [mc]
  int* sowner = reinterpret_cast<int*>(sprice + mc);                                   // [mc]
  const uint32_t bar0 = smem_addr(bars);

  const int o0 = min(s.m, (int)cta * mc), o1 = min(s.m, o0 + mc);
  for (int j = o0 + tid; j < o1; j += TAIL_THREADS) {
    sprice[j - o0] = s.price[j];
    sowner[j - o0] = s.owner[j];
  }
  const int cur_list = ctrl->cur;
  int nu = ctrl->cnt[cur_list];
  if (tid < CL_NU) s_list[tid] = tid < nu ? s.un[cur_list][tid] : -1;
  const double eps = ctrl->eps;
  if (tid == 0) {
    tail_mbar_init(bar0, 1);
    tail_mbar_init(bar0 + 8, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    tail_mbar_expect(bar0, ncta * (uint32_t)nu * (uint32_t)sizeof(SymPart));  // round 0
  }
  // this lane's destination (lanes < ncta): the inbox and the two barriers of CTA `lane`
  const uint32_t dst_inbox = map_to_cta(smem_addr(inbox), lane < (int)ncta ? lane : 0);
  const uint32_t dst_bar = map_to_cta(bar0, lane < (int)ncta ? lane : 0);
  __syncthreads();
  // all barriers of the cluster are initialised and armed before anybody stores remotely
  asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");

  long long rounds = 0, bids = 0;
  int stalled = 0;
  int slots = nu;  // slots the current round's barrier was armed for (>= nu)
  const uint32_t pf_slice = (s.vec && s.prefetch_rows) ? ((uint32_t)(o1 - o0) * 8u) & ~15u : 0u;
  const uint32_t pf_bytes = (s.vec && s.prefetch_rows) ? (uint32_t)s.m * 8u : 0u;  // rows are 16-byte aligned multiples of 16
  const int span = o1 - o0;
  long long tq[4] = {0, 0, 0, 0};
  while (nu > 0) {
    if (eps > 0.0 && (nu <= s.scale_cut_nu || rounds >= s.scale_tail_rounds)) break;  // (uniform over the cluster)
    const long long c0 = clock64();
    const uint32_t par = (uint32_t)rounds & 1u;
    // arm the NEXT round's barrier (see the header comment) for this round's bidder count
    if (tid == 0) tail_mbar_expect(bar0 + 8 * (par ^ 1u), ncta * (uint32_t)nu * (uint32_t)sizeof(SymPart));
    // ---- 1. scan: as in lap_tail_cluster_kernel
    int G = TAIL_WARPS;
    while (G > 1 && G * nu > TAIL_WARPS) G >>= 1;
    const int per_pass = TAIL_WARPS / G;
    const int sub = (((span + G - 1) / G) + 1) & ~1;  // even sub-slice length
    const int g = warp % G;
    const int ws = min(o1, o0 + g * sub), we = min(o1, ws + sub);
    for (int b = warp / G; b < nu; b += per_pass) {
      const double* wrow = s.W + (int64_t)s_list[b] * s.ldw;
      Top2 t{NEG_INF, NEG_INF, -1, -1};
      if (s.vec) {
        auto batch = [&](auto depth_tag) {
          constexpr int D = decltype(depth_tag)::value;
          for (int j = ws + 2 * lane; j < we; j += D * 64) {
            double2 wv[D];
#pragma unroll
            for (int u = 0; u < D; ++u) {
              const int jj = j + u * 64;
              wv[u] = make_double2(NEG_INF, NEG_INF);
              if (jj + 1 < we)
                wv[u] = __ldg(reinterpret_cast<const double2*>(wrow + jj));
              else if (jj < we)
                wv[u].x = __ldg(wrow + jj);
            }
#pragma unroll
            for (int u = 0; u < D; ++u) {
              const int jj = j + u * 64;
              if (jj + 1 < we) {
                const double2 pv = *reinterpret_cast<const double2*>(sprice + (jj - o0));
                top2_push_seq(t, wv[u].x - pv.x, jj);
                top2_push_seq(t, wv[u].y - pv.y, jj + 1);
              } else if (jj < we) {
                top2_push_seq(t, wv[u].x - sprice[jj - o0], jj);
              }
            }
          }
        };
        if (we - ws <= 128)
          batch(std::integral_constant<int, 2>{});
        else
          batch(std::integral_constant<int, 8>{});
      } else {
        for (int j = ws + lane; j < we; j += 32) top2_push_seq(t, __ldg(wrow + j) - sprice[j - o0], j);
      }
      t = top2_warp_reduce(t);
      if (lane == 0) wpart[b * TAIL_WARPS + g] = t;
    }
    __syncthreads();
    const long long c1 = clock64();
    // ---- 2. warp b merges the G warp partials of bidder b; lane c ships the CTA partial to CTA c.  Slots
    //         nu .. slots-1 (bidders that have gone since the barrier was armed) get filler.
    for (int b = warp; b < slots; b += TAIL_WARPS) {
      Top2 a{NEG_INF, NEG_INF, -1, -1};
      if (b < nu) {
        if (lane < G) a = wpart[b * TAIL_WARPS + lane];
        a = top2_warp_reduce(a);
      }
      if (lane < (int)ncta) {
        double p1 = 0.0, p2 = 0.0;
        int own1 = -1, own2 = -1;
        if (a.j1 >= 0) p1 = sprice[a.j1 - o0], own1 = sowner[a.j1 - o0];
        if (a.j2 >= 0) p2 = sprice[a.j2 - o0], own2 = sowner[a.j2 - o0];
        // If this CTA's candidate wins, its owner is evicted and bids next round: pull that person's cost row into
        // L2 now, one exchange + one resolution ahead of the scan that needs it (a cold row is a TLB miss + a DRAM
        // page miss: ~2 us per scan measured, against ~0.7 us for the exchange and ~0.9 us for the resolution).
        // Every CTA does this for its own candidate: ncta rows per bidder, one of them the right one.
        if (lane == 0 && pf_bytes != 0u && own1 >= 0 && nu <= 4)
          asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(s.W + (int64_t)own1 * s.ldw), "r"(pf_bytes)
                       : "memory");
        const uint32_t dst = dst_inbox + (uint32_t)(((par * CL_NU + b) * CL_MAX_CS + cta) * sizeof(SymPart));
        const uint32_t rbar = dst_bar + 8 * par;
        st_async_v2(dst, __double_as_longlong(a.v1), __double_as_longlong(a.v2), rbar);
        st_async_v2(dst + 16, __double_as_longlong(p1), __double_as_longlong(p2), rbar);
        st_async_v2(dst + 32, ((uint64_t)(uint32_t)a.j2 << 32) | (uint32_t)a.j1,
                    ((uint64_t)(uint32_t)own2 << 32) | (uint32_t)own1, rbar);
      }
    }
    // ---- 3. warp 0 of EVERY CTA: merge over the CTAs, resolve, apply to the own slice
    if (warp == 0) {
      tail_mbar_wait(bar0 + 8 * par, (uint32_t)(rounds >> 1) & 1u);
      const long long c2 = clock64();
      tq[1] += c2 - c1;
      const SymPart* in = inbox + (size_t)par * CL_NU * CL_MAX_CS;
      const bool live = lane < nu;
      Top2 a{NEG_INF, NEG_INF, -1, -1};
      if (nu <= 4) {  // few bidders (the usual case): one redux reduction per bidder over the CTAs' partials
        for (int bb = 0; bb < nu; ++bb) {
          Top2 q{NEG_INF, NEG_INF, -1, -1};
          if (lane < (int)ncta) {
            const SymPart& pq = in[bb * CL_MAX_CS + lane];
            q = Top2{pq.v1, pq.v2, pq.j1, pq.j2};
          }
          q = top2_warp_reduce(q);
          if (lane == bb) a = q;
        }
      } else if (live) {
        for (uint32_t c = 0; c < ncta; ++c) {
          const SymPart& q = in[lane * CL_MAX_CS + c];
          top2_merge(a, Top2{q.v1, q.v2, q.j1, q.j2});
        }
      }
      // price / owner of the two candidates travelled with the partial of the CTA that owns them
      double p1 = 0.0, p2 = 0.0;
      int own1 = -1, own2 = -1;
      if (live && a.j1 >= 0) {
        const SymPart& q = in[lane * CL_MAX_CS + a.j1 / mc];
        const bool first = q.j1 == a.j1;
        p1 = first ? q.p1 : q.p2;
        own1 = first ? q.own1 : q.own2;
      }
      if (live && a.j2 >= 0 && eps == 0.0 && a.v1 == a.v2) {
        const SymPart& q = in[lane * CL_MAX_CS + a.j2 / mc];
        const bool first = q.j1 == a.j2;
        p2 = first ? q.p1 : q.p2;
        own2 = first ? q.own1 : q.own2;
      }
      const int i = live ? s_list[lane] : -1;
      int j = a.j1;
      double p_old = p1, bval = a.v1;
      int prev = own1;
      if (live && eps == 0.0 && a.j2 >= 0 && a.v1 == a.v2 && own1 >= 0 && own2 < 0) {  // exact tie: take the free one
        j = a.j2, p_old = p2, bval = a.v2, prev = own2;
      }
      const double gamma = (a.j2 >= 0 ? (a.v1 - a.v2) : 0.0) + eps;
      const unsigned long long key = live ? pack_bid(gamma, i) : 0ull;
      s_bj[lane] = j;
      s_bkey[lane] = key;
      __syncwarp();
      bool win = live;
      // (a __match_any_sync here instead of the loop was measured slower: 54.0 vs 45.0 Mcycles over the C5 square step)
      for (int q = 0; q < nu; ++q)
        if (s_bj[q] == j && s_bkey[q] > key) win = false;
      const double p_new = p_old + gamma;
      const bool applied = win && (prev < 0 || gamma > GAMMA_TIE);
      const bool has = live && (applied ? prev >= 0 : true);
      const int person_out = applied ? prev : i;
      const unsigned hmask = __ballot_sync(0xffffffffu, has);
      const int nu_next = __popc(hmask);
      const int nacc = __popc(__ballot_sync(0xffffffffu, applied));
      if (has) s_tmp[__popc(hmask & ((1u << lane) - 1u))] = person_out;
      __syncwarp();
      s_list[lane] = lane < nu_next ? s_tmp[lane] : -1;
      // several bidders next round: their rows' slices are swept in up to six dependent batches per warp -- pull this
      // CTA's slice of each row into L2 now (one next bidder: its row was requested a round ago, see above)
      if (pf_slice != 0u && nu_next > 1 && lane < nu_next)
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(s.W + (int64_t)s_tmp[lane] * s.ldw + o0),
                     "r"(pf_slice)
                     : "memory");
      if (lane == 0) s_ctl[0] = nu_next, s_ctl[1] = nacc;
      if (applied) {
        if (j >= o0 && j < o1) {
          sprice[j - o0] = p_new;
          sowner[j - o0] = i;
        }
        if (cta == 0) {  // global state, read again only by later kernels
          s.owner[j] = i;
          s.price[j] = p_new;
          s.col4row[i] = j;
          s.profit[i] = (bval + p_old) - p_new;
          if (prev >= 0) s.col4row[prev] = -1;
        }
      }
      __syncwarp();  // orders this round's col4row stores before the next round's (different lanes, same warp)
      tq[2] += clock64() - c2;
    }
    tq[0] += c1 - c0;
    if (nu == 1) tq[3] += c1 - c0;  // (t_phase[7] of this kernel: scan cycles of the single-bidder rounds)
    __syncthreads();
    rounds++;
    bids += nu;
    slots = nu;
    nu = s_ctl[0];
    const int nacc = s_ctl[1];
    if (nacc == 0 && nu > 0) {  // nobody could raise a price: exact ties -> augmentation kernel
      stalled = 1;
      break;
    }
  }
  // no CTA may leave while peers can still address its shared memory
  asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");
  if (cta == 0) {
    if (tid < nu) s.un[cur_list][tid] = s_list[tid];
    if (tid == 0) {
      ctrl->cnt[cur_list] = nu;
      ctrl->in_tail = 0;
      if (eps == 0.0) {
        ctrl->finished = 1;
        ctrl->stalled = (stalled && nu > 0) ? 1 : 0;
      }
      s.counters->rounds += rounds;
      s.counters->bids += bids;
      s.counters->bytes += bids * (long long)s.m * 8;
      for (int q = 0; q < 4; ++q) s.counters->t_phase[4 + q] += tq[q];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Phase A, narrow part, MASTER / HELPER form (long rows and the square phases).
//
// Measured on the 10k x 50k steps: a person's top-128 candidate list certifies ~90 % of its bids, and the ~25k
// narrow rounds of a step are one dependent chain -- what matters is the latency of ONE round.  So CTA 0 of a
// cluster (the master) runs the rounds by itself: one warp per bidder reads the bidder's list (L1/L2 resident:
// the same few persons bid over and over), gathers the prices of its 128 candidates, reduces to the top-2 and
// checks the certificate; the winners are resolved in shared memory and applied to the global state, which only
// the master writes while this kernel runs.  No cluster traffic at all in such a round (~0.5 us instead of ~7 us
// for the scan-every-row cluster kernel above).
// Only when a list FAILS does the cluster work: the master fences its price updates, posts the row to every CTA
// (st.async + mbarrier complete_tx), each CTA sweeps its slice of the row (W from HBM, prices from L2), keeps its
// slice's top KC = 128 / #CTAs objects plus a slice bound, and ships them back into the master's shared memory
// the same way.  The union of the slice tops IS the person's new list (every unlisted object lies below
// max_c bound_c, which is all the certificate needs, and the row's true top-2 are always in it).
// ------------------------------------------------------------------------------------------------
constexpr int MH_NU = 128;          // bidders per round the master can take (threads 0..MH_NU-1 resolve them)
constexpr int MH_KW = 4;            // candidates every warp hands to its CTA's selection
constexpr uint32_t MH_CMD_BYTES = 16;
// A narrow-round phase that is still running after this many rounds with a handful of bidders is a price war over a
// starved group (e.g. a clone with more DNA than remaining RNA cells): the last few persons would need 10^5 more rounds
// of ~2 us, while an augmenting path costs one Dijkstra tree each.  The phase is cut and the augmenting-path kernel
// -- exact from any dual-feasible state -- places them.  (Resampled replicates: 150k-270k-round phases.)
// The budget grows with the row length (a Dijkstra step of the augmenting-path kernel scans one row of m costs).
constexpr int MH_BUDGET_NU = 16;

struct __align__(16) MhEntry {  // one list entry travelling from a helper to the master
  double w;                     // cost W[i, j]
  int j, pad;
};

__global__ void __launch_bounds__(TAIL_THREADS, 1) lap_tail_mh_kernel(LapState s, int mc /* objects per CTA, even */) {
  LapCtrl* ctrl = s.ctrl;
  if (ctrl->finished || !ctrl->in_tail || s.flags[0]) return;  // uniform over the cluster
  uint32_t cta, ncta;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(cta));
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(ncta));
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const int kc = LIST_K / (int)ncta;  // list slots every CTA fills (8 for 16 CTAs, 16 for 8)

  __shared__ __align__(16) MhEntry s_reply[LIST_K];      // master: [cta][kc] entries of the rebuilt list
  __shared__ __align__(16) double s_rbound[2 * CL_MAX_CS];  // master: slice bounds (16-byte slots)
  __shared__ __align__(16) int s_cmd[4];                  // every CTA: {row, type, -, -} posted by the master
  __shared__ __align__(8) unsigned long long s_bars[2];   // [0] command arrived (every CTA), [1] replies in (master)
  __shared__ double s_cv[TAIL_WARPS * MH_KW];
  __shared__ int s_cj[TAIL_WARPS * MH_KW];
  __shared__ double s_wb[TAIL_WARPS];
  __shared__ int s_list[2][MH_NU];
  __shared__ int s_bj[MH_NU];
  __shared__ double s_gam[MH_NU], s_bval[MH_NU];
  __shared__ unsigned long long s_key[MH_NU];
  __shared__ int s_fail[MH_NU];
  __shared__ int s_cnt[4];  // [0] failures, [1] next count, [2] accepted
  __shared__ int s_wcnt[MH_NU / 32], s_wacc[MH_NU / 32];  // per resolving warp: persons for the next round, applied bids
  const uint32_t bar_cmd = smem_addr(&s_bars[0]), bar_reply = smem_addr(&s_bars[1]);

  const int o0 = min(s.m, (int)cta * mc), o1 = min(s.m, o0 + mc);
  const int cur_list = ctrl->cur;
  int nu = ctrl->cnt[cur_list];
  const double eps = ctrl->eps;
  if (tid < MH_NU) s_list[0][tid] = tid < nu ? s.un[cur_list][tid] : -1;
  if (tid == 0) {
    tail_mbar_init(bar_cmd, 1);
    tail_mbar_init(bar_reply, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    tail_mbar_expect(bar_cmd, MH_CMD_BYTES);
  }
  __syncthreads();
  asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");
  const uint32_t reply0 = map_to_cta(smem_addr(s_reply), 0);
  const uint32_t rbound0 = map_to_cta(smem_addr(s_rbound), 0);
  const uint32_t bar_reply0 = map_to_cta(bar_reply, 0);

  // Sweep this CTA's slice of row i: slice top-kc (+ bound) to the master.  Called by all threads of every CTA.
  auto sweep_slice = [&](int i) {
    const double* wrow = s.W + (int64_t)i * s.ldw;
    Top2 t{NEG_INF, NEG_INF, -1, -1};
    double lb = NEG_INF;  // largest value this lane dropped
    auto push = [&](double v, int j) {
      if (v > t.v1) {
        lb = fmax(lb, t.v2);
        t.v2 = t.v1, t.j2 = t.j1, t.v1 = v, t.j1 = j;
      } else if (v > t.v2) {
        lb = fmax(lb, t.v2);
        t.v2 = v, t.j2 = j;
      } else {
        lb = fmax(lb, v);
      }
    };
    int j = o0 + 2 * tid;
    if (s.vec) {
      constexpr int S = 2 * TAIL_THREADS;
      for (; j + 3 * S + 1 < o1; j += 4 * S) {
        double2 wv[4], pv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) wv[u] = __ldg(reinterpret_cast<const double2*>(wrow + j + u * S));
#pragma unroll
        for (int u = 0; u < 4; ++u) pv[u] = ldm(reinterpret_cast<const double2*>(s.price + j + u * S));
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          push(wv[u].x - pv[u].x, j + u * S);
          push(wv[u].y - pv[u].y, j + u * S + 1);
        }
      }
      // remainder: up to 4 more pairs per lane, all loads issued before the first use
      double2 wv[4], pv[4];
      bool full[4], half[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int jj = j + u * S;
        full[u] = jj + 1 < o1;
        half[u] = !full[u] && jj < o1;
        wv[u] = make_double2(0.0, 0.0);
        pv[u] = make_double2(0.0, 0.0);
        if (full[u]) {
          wv[u] = __ldg(reinterpret_cast<const double2*>(wrow + jj));
          pv[u] = ldm(reinterpret_cast<const double2*>(s.price + jj));
        } else if (half[u]) {
          wv[u].x = __ldg(wrow + jj);
          pv[u].x = ldm(s.price + jj);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int jj = j + u * S;
        if (full[u] || half[u]) push(wv[u].x - pv[u].x, jj);
        if (full[u]) push(wv[u].y - pv[u].y, jj + 1);
      }
    } else {
      for (int jj = o0 + tid; jj < o1; jj += TAIL_THREADS) push(__ldg(wrow + jj) - ldm(s.price + jj), jj);
    }
    // warp: hand the warp's best MH_KW candidates to the CTA, everything else goes into the warp bound
#pragma unroll
    for (int r = 0; r < MH_KW; ++r) {
      double bv = t.v1;
      int bj = t.j1;
      warp_argmax(bv, bj);
      if (bj >= 0 && bj == t.j1) {  // this lane held the winner: pop it
        t.v1 = t.v2, t.j1 = t.j2;
        t.v2 = NEG_INF, t.j2 = -1;
      }
      if (lane == r) {
        s_cv[warp * MH_KW + r] = bv;
        s_cj[warp * MH_KW + r] = bj;
      }
    }
    double wb = fmax(lb, t.v1);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) wb = fmax(wb, __shfl_xor_sync(0xffffffffu, wb, o));
    if (lane == 0) s_wb[warp] = wb;
    __syncthreads();
    // warp 0: the CTA's best kc of the TAIL_WARPS * MH_KW = 64 candidates (two per lane)
    if (warp == 0) {
      double a1 = s_cv[lane], a2 = s_cv[lane + 32];
      int b1 = s_cj[lane], b2 = s_cj[lane + 32];
      if (b1 < 0) a1 = NEG_INF;
      if (b2 < 0) a2 = NEG_INF;
      if (a2 > a1 || (a2 == a1 && (unsigned)b2 < (unsigned)b1)) {
        const double xa = a1;
        a1 = a2, a2 = xa;
        const int xb = b1;
        b1 = b2, b2 = xb;
      }
      double ev = NEG_INF;
      int ej = -1;
      for (int r = 0; r < kc; ++r) {
        double bv = a1;
        int bj = b1;
        warp_argmax(bv, bj);
        if (bj >= 0 && bj == b1) {
          a1 = a2, b1 = b2;
          a2 = NEG_INF, b2 = -1;
        }
        if (lane == r) ev = bv, ej = bj;
      }
      double cb = fmax(a1, lane < TAIL_WARPS ? s_wb[lane] : NEG_INF);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) cb = fmax(cb, __shfl_xor_sync(0xffffffffu, cb, o));
      if (lane < kc) {
        // empty slots (slice shorter than kc) become never-chosen entries on a valid object index
        const double wv = ej >= 0 ? __ldg(wrow + ej) : NEG_INF;
        const int jv = ej >= 0 ? ej : 0;
        st_async_v2(reply0 + (uint32_t)((cta * kc + lane) * sizeof(MhEntry)), (uint64_t)__double_as_longlong(wv),
                    (uint64_t)(uint32_t)jv, bar_reply0);
      }
      if (lane == 0) st_async_v2(rbound0 + cta * 16, (uint64_t)__double_as_longlong(cb), 0ull, bar_reply0);
    }
    __syncthreads();  // s_cv / s_cj / s_wb are free again
  };

  if (cta != 0) {
    // ===================== helpers: sleep on the command barrier =====================
    uint32_t par = 0;
    for (;;) {
      tail_mbar_wait(bar_cmd, par);
      par ^= 1;
      const int row = s_cmd[0], type = s_cmd[1];
      __syncthreads();  // everybody has the command before the barrier is re-armed
      if (tid == 0) tail_mbar_expect(bar_cmd, MH_CMD_BYTES);
      if (type != 0) break;
      sweep_slice(row);
    }
  } else {
    // ===================== master =====================
    long long rounds = 0, bids = 0, sweeps = 0;
    long long tq[4] = {0, 0, 0, 0};
    int cur = 0, stalled = 0;
    uint32_t rpar = 0;
    if (tid == 0) s_cnt[0] = 0;
    __syncthreads();
    const uint32_t reply_bytes = ncta * (uint32_t)(kc * sizeof(MhEntry) + 16);

    auto finalize = [&](int b, Top2 t) {  // one thread records bidder b's bid in shared memory
      int j = t.j1;
      if (eps == 0.0 && t.j2 >= 0 && t.v1 == t.v2 && s.owner[j] >= 0 && s.owner[t.j2] < 0) j = t.j2;  // exact tie
      const double gamma = (t.j2 >= 0 ? (t.v1 - t.v2) : 0.0) + eps;
      s_bj[b] = j;
      s_gam[b] = gamma;
      s_bval[b] = (j == t.j1) ? t.v1 : t.v2;
      s_key[b] = pack_bid(gamma, s_list[cur][b]);
    };

    while (nu > 0) {
      if (rounds >= s.max_rounds || (eps == 0.0 && rounds >= s.tail_budget && nu <= MH_BUDGET_NU)) {
        stalled = 1;
        break;
      }
      if (eps > 0.0 && (nu <= s.scale_cut_nu || rounds >= s.scale_tail_rounds)) break;
      // (two CTA barriers per certified round: the failure counter is reset by the resolving warp behind the previous
      //  round's last barrier, and the barrier behind the failure loop only exists when a list failed)
      const long long c0 = clock64();
      // ---- 1. bids from the candidate lists, one warp per bidder (at most two bidders per warp)
      for (int b = warp; b < nu; b += TAIL_WARPS) {
        const int i = s_list[cur][b];
        bool ok = false;
        Top2 t;
        ok = list_bid<false>(s, i, lane, t);
        if (lane == 0) {
          if (ok)
            finalize(b, t);
          else
            s_fail[atomicAdd(&s_cnt[0], 1)] = b;
        }
      }
      __syncthreads();
      const long long c1 = clock64();
      // ---- 2. failed lists: the whole cluster sweeps the row, the master takes the new list
      const int nfail = s_cnt[0];
      for (int f = 0; f < nfail; ++f) {
        const int b = s_fail[f];
        const int i = s_list[cur][b];
        if (s.list_k == s.m) {  // short rows: the list is simply every object
          for (int e = tid; e < s.m; e += TAIL_THREADS) {
            s.lj[(int64_t)i * LIST_K + e] = e;
            s.lw[(int64_t)i * LIST_K + e] = s.W[(int64_t)i * s.ldw + e];
          }
          if (tid == 0) lb_store(s, i, NEG_INF), s.lvalid[i] = 1;
          __syncthreads();
        } else {
          if (tid == 0) {
            __threadfence();  // the helpers read prices from L2: every update of the earlier rounds is there first
            tail_mbar_expect(bar_reply, reply_bytes);
          }
          __syncthreads();
          if (tid >= 1 && tid < (int)ncta)
            st_async_v2(map_to_cta(smem_addr(s_cmd), tid), (uint64_t)(uint32_t)i, 0ull, map_to_cta(bar_cmd, tid));
          sweep_slice(i);
          tail_mbar_wait(bar_reply, rpar);
          rpar ^= 1;
          if (tid < LIST_K) {
            s.lj[(int64_t)i * LIST_K + tid] = s_reply[tid].j;
            s.lw[(int64_t)i * LIST_K + tid] = s_reply[tid].w;
          }
          if (tid == 0) {
            double bound = NEG_INF;
            for (uint32_t c = 0; c < ncta; ++c) bound = fmax(bound, s_rbound[2 * c]);
            lb_store(s, i, bound);
            s.lvalid[i] = 1;
          }
          __syncthreads();  // list + bound visible to warp 0 below; s_reply may be overwritten by the next sweep
        }
        if (warp == 0) {
          Top2 t;
          list_bid<false>(s, i, lane, t);  // the fresh list holds the row's true top-2
          if (lane == 0) finalize(b, t);
        }
      }
      sweeps += nfail;
      if (nfail > 0) __syncthreads();  // (uniform) the bids recorded by the failure loop above
      const long long c2 = clock64();
      // ---- 3. resolution, one bidder per thread
      auto resolve = [&](bool live, bool win, int& person_out, bool& applied) {
        person_out = -1;
        applied = false;
        if (!live) return;
        const int j = s_bj[tid];
        const int i = s_list[cur][tid];
        person_out = i;  // re-queue unless the bid is applied
        if (!win) return;
        const double p_old = s.price[j];
        const double p_new = p_old + s_gam[tid];
        const int prev = s.owner[j];
        const double defend = class_defends<false>(s, i, prev, s_gam[tid]);
        if (defend > 0.0) {  // the owner's class has settled lower: the owner raises the price and keeps the object
          s.price[j] = p_old + defend;
          s.profit[prev] -= defend;
          applied = true;  // (progress; the bidder is re-queued: person_out stays i)
        } else if (prev < 0 || s_gam[tid] > GAMMA_TIE) {
          applied = true;
          person_out = prev;  // the evicted owner (or -1) bids next round
          s.owner[j] = i;
          if (s.pcls != nullptr) s.ocls[j] = s.pcls[i];
          s.price[j] = p_new;
          s.col4row[i] = j;
          const double prof = (s_bval[tid] + p_old) - p_new;
          s.profit[i] = prof;
          class_settle(s, i, prof);
          if (prev >= 0) s.col4row[prev] = -1;
        }
      };
      if (nu <= 32) {
        // the usual case: warp 0 resolves, compacts the next bidder list and publishes the counts by itself (one
        // CTA barrier per resolution instead of two)
        if (warp == 0) {
          const bool live = lane < nu;
          const int j = live ? s_bj[lane] : -1 - lane;
          const unsigned long long key = live ? s_key[lane] : 0ull;
          bool win = live;
          if (nu <= 4) {
            for (int q = 0; q < nu; ++q)
              if (s_bj[q] == j && s_key[q] > key) win = false;  // (keys carry the person: never equal)
          } else {
            // the lanes bidding on the same object find each other with one match instruction
            for (unsigned g = __match_any_sync(0xffffffffu, j) & ~(1u << lane); g != 0u; g &= g - 1u)
              if (s_key[__ffs(g) - 1] > key) win = false;
          }
          int person_out;
          bool applied;
          resolve(live, win, person_out, applied);
          const unsigned has = __ballot_sync(0xffffffffu, person_out >= 0);
          const unsigned acc = __ballot_sync(0xffffffffu, applied);
          if (person_out >= 0) s_list[cur ^ 1][__popc(has & ((1u << lane) - 1u))] = person_out;
          if (lane == 0) s_cnt[1] = __popc(has), s_cnt[2] = __popc(acc), s_cnt[0] = 0;
        }
        __syncthreads();
      } else {
        int person_out = -1;
        bool applied = false;
        if (tid < MH_NU) {
          const bool live = tid < nu;
          const int j = live ? s_bj[tid] : -1;
          const unsigned long long key = live ? s_key[tid] : 0ull;
          bool win = live;
          if (live)
            for (int q = 0; q < nu; ++q)  // broadcast reads
              if (s_bj[q] == j && s_key[q] > key) win = false;
          resolve(live, win, person_out, applied);
          // ordered compaction of the next bidder list over the resolving warps
          const unsigned has = __ballot_sync(0xffffffffu, person_out >= 0);
          const unsigned acc = __ballot_sync(0xffffffffu, applied);
          if (lane == 0) s_wcnt[warp] = __popc(has), s_wacc[warp] = __popc(acc);
        }
        __syncthreads();
        if (tid < MH_NU) {
          int off = 0;
          for (int w = 0; w < warp; ++w) off += s_wcnt[w];
          const unsigned has = __ballot_sync(0xffffffffu, person_out >= 0);
          if (person_out >= 0) s_list[cur ^ 1][off + __popc(has & ((1u << lane) - 1u))] = person_out;
          if (tid == 0) {
            int tn = 0, ta = 0;
            for (int w = 0; w < MH_NU / 32; ++w) tn += s_wcnt[w], ta += s_wacc[w];
            s_cnt[1] = tn, s_cnt[2] = ta, s_cnt[0] = 0;
          }
        }
        __syncthreads();
      }
      const int nu_next = s_cnt[1], accepted = s_cnt[2];
      rounds++;
      bids += nu;
      const long long c3 = clock64();
      tq[0] += c1 - c0;
      tq[1] += c2 - c1;
      tq[2] += c3 - c2;
      cur ^= 1;
      nu = nu_next;
      if (accepted == 0 && nu > 0) {  // nobody could raise a price: exact ties -> augmentation kernel
        stalled = 1;
        break;
      }
    }
    // release the helpers
    __syncthreads();
    if (tid >= 1 && tid < (int)ncta)
      st_async_v2(map_to_cta(smem_addr(s_cmd), tid), (uint64_t)1 << 32, 0ull, map_to_cta(bar_cmd, tid));
    if (tid < nu) s.un[cur_list][tid] = s_list[cur][tid];
    if (tid == 0) {
      ctrl->cnt[cur_list] = nu;
      ctrl->in_tail = 0;
      if (eps == 0.0) {
        ctrl->finished = 1;
        ctrl->stalled = (stalled && nu > 0) ? 1 : 0;
      }
      s.counters->rounds += rounds;
      s.counters->bids += bids;
      s.counters->bytes += sweeps * (long long)s.m * 8;
      for (int q = 0; q < 4; ++q) s.counters->t_phase[4 + q] += tq[q];
    }
  }
  // no CTA may leave while peers can still address its shared memory
  asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ------------------------------------------------------------------------------------------------
// Phase B: shortest augmenting paths for the persons phase A left unassigned.  One CTA; the
// per-step work is one cost row (m objects) spread over 1024 threads.  min-form duals:
// u_i = -profit_i, v_j = -price_j, cost' = -W.
// ------------------------------------------------------------------------------------------------
struct MinItem {
  double v;
  int j;
  int free_;  // 1 if the column is unowned
};
__device__ __forceinline__ bool min_better(const MinItem& a, const MinItem& b) {
  if (a.v != b.v) return a.v < b.v;
  if (a.free_ != b.free_) return a.free_ > b.free_;
  return a.j < b.j;
}

__global__ void __launch_bounds__(JV_THREADS) lap_augment_kernel(LapState s) {
  LapCtrl* ctrl = s.ctrl;
  if (!ctrl->stalled || s.flags[0]) return;
  __shared__ MinItem red[JV_THREADS / 32];
  __shared__ MinItem best;
  const int tid = threadIdx.x;
  const int cur_list = ctrl->cur;
  const int nfree = ctrl->cnt[cur_list];
  int* freelist = s.un[cur_list];
  long long steps = 0, bytes = 0;

  // The wide kernel appends to the bidder list with atomics, so its ORDER depends on scheduling; the augmentations
  // below run in list order and on exact-tie instances the order decides which optimum comes out.  Sort it ascending
  // (rank sort: the list is short): same input -> same assignment, on every run and every rank.
  {
    int* sorted = s.un[cur_list ^ 1];
    for (int a = tid; a < nfree; a += JV_THREADS) {
      const int v = freelist[a];
      int rank = 0;
      for (int b = 0; b < nfree; ++b) rank += (freelist[b] < v) ? 1 : 0;  // persons are distinct
      sorted[rank] = v;
    }
    __syncthreads();
    for (int a = tid; a < nfree; a += JV_THREADS) freelist[a] = sorted[a];
    __syncthreads();
  }

  for (int f = 0; f < nfree; ++f) {
    const int cur_row = freelist[f];
    for (int j = tid; j < s.m; j += JV_THREADS) s.sp[j] = 1.0e300;
    __syncthreads();
    double minval = 0.0;
    int i = cur_row;
    double ui = 0.0;  // dual of the row being scanned (min-form); the free row starts at 0
    int nsc = 0;
    int sink = -1;
    while (sink < 0) {
      const double* w = s.W + (int64_t)i * s.ldw;
      MinItem loc{1.0e300, 0x7fffffff, 0};
      for (int j = tid; j < s.m; j += JV_THREADS) {
        double spj = s.sp[j];
        if (spj == NEG_INF) continue;  // already scanned
        const double r = minval - w[j] - ui + s.price[j];
        if (r < spj) {
          spj = r;
          s.sp[j] = r;
          s.pred[j] = i;
        }
        MinItem it{spj, j, s.owner[j] < 0 ? 1 : 0};
        if (min_better(it, loc)) loc = it;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        MinItem ot{__shfl_xor_sync(0xffffffffu, loc.v, o), __shfl_xor_sync(0xffffffffu, loc.j, o),
                   __shfl_xor_sync(0xffffffffu, loc.free_, o)};
        if (min_better(ot, loc)) loc = ot;
      }
      if ((tid & 31) == 0) red[tid >> 5] = loc;
      __syncthreads();
      if (tid < 32) {
        MinItem x = red[tid];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          MinItem ot{__shfl_xor_sync(0xffffffffu, x.v, o), __shfl_xor_sync(0xffffffffu, x.j, o),
                     __shfl_xor_sync(0xffffffffu, x.free_, o)};
          if (min_better(ot, x)) x = ot;
        }
        if (tid == 0) {
          best = x;
          s.sc_col[nsc] = x.j;
          s.sc_val[nsc] = x.v;
          s.sp[x.j] = NEG_INF;
        }
      }
      __syncthreads();
      const MinItem b = best;
      minval = b.v;
      nsc++;
      steps++;
      bytes += (long long)s.m * 8;
      if (nsc > s.n + 1 || !(b.v < 1.0e299)) {
        // more scans than persons, or nothing reachable: only possible on corrupt (non-finite) costs
        if (tid == 0) s.counters->status |= 1;
        return;
      }
      if (b.free_) {
        sink = b.j;
      } else {
        i = s.owner[b.j];
        ui = -s.profit[i];
      }
      __syncthreads();
    }
    // dual update (every scanned column but the sink is owned; its owner is the row it led to)
    for (int q = tid; q < nsc; q += JV_THREADS) {
      const int j = s.sc_col[q];
      const double d = minval - s.sc_val[q];
      s.price[j] += d;  // v_j -= d
      const int r = s.owner[j];
      if (r >= 0) s.profit[r] -= d;  // u_r += d
    }
    __syncthreads();
    // augment along the predecessor chain (sequential, short)
    if (tid == 0) {
      s.profit[cur_row] = -minval;  // u_cur = 0 + minval
      int j = sink;
      for (;;) {
        const int r = s.pred[j];
        s.owner[j] = r;
        const int jn = s.col4row[r];
        s.col4row[r] = j;
        if (r == cur_row) break;
        j = jn;
      }
    }
    __syncthreads();
  }
  if (tid == 0) {
    s.counters->aug_rows += nfree;
    s.counters->aug_steps += steps;
    s.counters->bytes += bytes;
    ctrl->stalled = 0;
  }
}

// ------------------------------------------------------------------------------------------------
// Phase B on the whole grid (lap.sap): the last lap.sap_nu persons of a rectangular step, handed over by the
// asynchronous wide kernel.  Dijkstra above pops one column at a time, so a person costs as many dependent row scans
// as columns it settles (170-290 at 10k x 50k, ~20 us each).  Label-correcting search with pruning needs as many
// dependent ROUNDS as the shortest-path tree is deep, and a round relaxes all its rows at once:
//   init   d[j] = -W[f, j] + price[j] (min-form, u_f = 0), pred[j] = f;  best = min over free columns of d
//   round  the owned columns whose d improved in the last round and is still below best form the frontier; every
//          column j takes  min over frontier entries (k, r = owner[k]) of ((d[k] - W[r, j]) + profit[r]) + price[j]
//          (same arithmetic as Dijkstra's relaxation; ties to the smaller row), and keeps it when it is lower than
//          d[j] by more than GAMMA_TIE -- after the naive auction many persons are exactly indifferent between two
//          objects, and a cycle of such zero reduced costs that rounds to a few ulps below zero must not be walked
//          around forever (Dijkstra is protected by its settled set)
//   stop   when the frontier is empty.  The sink is the free column at best (smaller index on ties: Dijkstra's order),
//          the JV dual update touches the owned columns below the sink's distance, the path is flipped along pred.
// Exact from any dual-feasible state, like lap_augment_kernel; the result does not depend on the order of updates.
// Layout: every CTA owns a fixed slice of the columns and PULLS the frontier rows into it -- each column has one
// writer, so no atomics on {d, pred}.  One grid barrier per round: a round appends the columns that improved below
// the previous best, and the next round drops the entries that the fresh best prunes.  scripts/research/sim_lcsap.py
// is the NumPy restatement (rounds, rows relaxed).
// ------------------------------------------------------------------------------------------------
constexpr int SAP_THREADS = 256;
constexpr int SAP_WARPS = SAP_THREADS / 32;
constexpr int SAP_UNROLL = 16;  // frontier rows whose W loads one thread has in flight (8 measured the same at C5)

__device__ __forceinline__ bool sap_less(double va, int ja, double vb, int jb) {  // smaller value, then smaller index
  return (va < vb) | ((va == vb) & (ja < jb));
}
// block-wide arg-min of (v, j), returned in every thread
__device__ __forceinline__ void sap_block_min(double& v, int& j, double* sv, int* sj) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, v, o);
    const int oj = __shfl_xor_sync(0xffffffffu, j, o);
    if (sap_less(ov, oj, v, j)) v = ov, j = oj;
  }
  __syncthreads();  // earlier readers of sv / sj are done
  if (lane == 0) sv[warp] = v, sj[warp] = j;
  __syncthreads();
  v = lane < SAP_WARPS ? sv[lane] : 1.0e300;
  j = lane < SAP_WARPS ? sj[lane] : 0x7fffffff;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, v, o);
    const int oj = __shfl_xor_sync(0xffffffffu, j, o);
    if (sap_less(ov, oj, v, j)) v = ov, j = oj;
  }
}
// best free column over the grid: arg-min of the CTAs' partials in slot `slot`; the length of the next frontier is
// read in the same batch of L2 loads
__device__ __forceinline__ void sap_grid_min(const LapState& s, int slot, double& v, int& j, double* sv, int* sj,
                                             const int* cntp, int& cnt) {
  cnt = cntp != nullptr ? ldm(cntp) : 0;
  v = 1.0e300;
  j = 0x7fffffff;
  for (int q = threadIdx.x; q < (int)gridDim.x; q += SAP_THREADS) {
    const double qv = ldm(s.pv1 + slot * gridDim.x + q);
    const int qj = ldm(s.pj1 + slot * gridDim.x + q);
    if (sap_less(qv, qj, v, j)) v = qv, j = qj;
  }
  sap_block_min(v, j, sv, sj);
}

__global__ void __launch_bounds__(SAP_THREADS) lap_sap_kernel(LapState s) {
  LapCtrl* ctrl = s.ctrl;
  // only behind the asynchronous kernel (ascending list of the unassigned persons, exact-CS prices); after an exact
  // tie the step was redone round-synchronously and its own tail / lap_augment_kernel finish it
  if (ctrl->finished || !ctrl->in_tail || ctrl->a_fallback || s.flags[0]) return;  // uniform
  GridBarrier grid{&ctrl->barrier[MAX_PHASES - 3], 0u};  // slots 0 / MAX_PHASES - 1, - 2: the auction kernels
  __shared__ double sv[SAP_WARPS];
  __shared__ int sj[SAP_WARPS];
  __shared__ double e_d[SAP_THREADS], e_p[SAP_THREADS];
  __shared__ int e_r[SAP_THREADS];
  __shared__ int e_n;
  const int tid = threadIdx.x;
  const int G = gridDim.x;
  const int m = s.m;
  const int slice = (m + G - 1) / G;
  const int j0 = min(m, (int)blockIdx.x * slice), j1 = min(m, j0 + slice);
  const int waves = (j1 - j0 + SAP_THREADS - 1) / SAP_THREADS;  // uniform over the CTA
  const int cur_list = ctrl->cur;
  int* freelist = s.un[cur_list];
  const int nfree = ctrl->cnt[cur_list];
  const bool lead = blockIdx.x == 0 && tid == 0;
  long long rounds = 0, rows = 0;
  unsigned long long t_init = 0, t_rounds = 0, t_aug = 0, T0, T1, T2, T3;  // (ns, CTA 0)
  int q = 0, err = 0;  // persons placed; 1 = nothing reachable, 2 = round guard
  for (; q < nfree; ++q) {
    if (lead) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(T0));
    const int f = ldm(freelist + q);
    if (blockIdx.x == 0 && tid < 3) ctrl->sap_cnt[tid] = 0;
    // ---- init: distances from f's row, best free column
    const double* wf = s.W + (int64_t)f * s.ldw;
    double lv = 1.0e300;
    int lj = 0x7fffffff;
    for (int j = j0 + tid; j < j1; j += SAP_THREADS) {
      const double d = -__ldg(wf + j) + ldm(s.price + j);
      s.sp[j] = d;
      s.pred[j] = f;
      if (ldm(s.owner + j) < 0 && sap_less(d, j, lv, lj)) lv = d, lj = j;
    }
    sap_block_min(lv, lj, sv, sj);
    if (tid == 0) s.pv1[blockIdx.x] = lv, s.pj1[blockIdx.x] = lj;  // slot 0
    grid.sync();
    double best;
    int sink, cnt;
    sap_grid_min(s, 0, best, sink, sv, sj, nullptr, cnt);
    if (!(best < 1.0e299)) {  // no free column reachable: only possible on corrupt (non-finite) costs
      err = 1;
      break;
    }
    for (int j = j0 + tid; j < j1; j += SAP_THREADS) {  // round 0's frontier: every owned column below best
      const double d = ldm(s.sp + j);
      const int o = ldm(s.owner + j);
      if (o >= 0 && d < best) {
        const int k = atomicAdd(&ctrl->sap_cnt[0], 1);
        s.sap_r[k] = o;
        s.sap_d[k] = d;
        s.sap_p[k] = ldm(s.profit + o);
      }
    }
    grid.sync();
    cnt = ldm(&ctrl->sap_cnt[0]);
    if (lead) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(T1));
    // ---- rounds: round t relaxes list t (buffer t & 1, length sap_cnt[t % 3]) against the best of slot t & 1
    for (int t = 0;; ++t) {
      if (cnt == 0) break;
      if (t > s.n + 1) {  // more rounds than a shortest-path tree can be deep: Dijkstra takes over (exact anyway)
        err = 2;
        break;
      }
      const int* fr = s.sap_r + (t & 1) * s.n;
      const double* fd = s.sap_d + (t & 1) * s.n;
      const double* fp = s.sap_p + (t & 1) * s.n;
      const int nb = ((t + 1) & 1) * s.n;
      lv = 1.0e300;
      lj = 0x7fffffff;
      for (int wv = 0; wv < waves; ++wv) {
        const int j = j0 + wv * SAP_THREADS + tid;
        const bool has = j < j1;
        // the column's own state is requested up front: nothing in this round changes it before the relaxation ends
        const double pj = has ? ldm(s.price + j) : 0.0;
        double d = has ? ldm(s.sp + j) : 0.0;
        const int o = has ? ldm(s.owner + j) : -1;
        double bv = 1.0e300;
        int br = 0x7fffffff;
        for (int e0 = 0; e0 < cnt; e0 += SAP_THREADS) {
          __syncthreads();
          if (tid == 0) e_n = 0;
          __syncthreads();
          if (e0 + tid < cnt) {
            const double dk = ldm(fd + e0 + tid);
            const double pk = ldm(fp + e0 + tid);
            const int rk = ldm(fr + e0 + tid);
            if (dk < best) {  // the fresh best prunes entries appended against the previous one
              const int k = atomicAdd(&e_n, 1);
              e_d[k] = dk;
              e_p[k] = pk;
              e_r[k] = rk;
            }
          }
          __syncthreads();
          const int ne = e_n;
          if (wv == 0) rows += ne;  // (every CTA sees the same frontier: CTA 0 reports it)
          if (has) {
            for (int e = 0; e < ne; e += SAP_UNROLL) {
              double w[SAP_UNROLL];
#pragma unroll
              for (int u = 0; u < SAP_UNROLL; ++u)
                w[u] = e + u < ne ? __ldg(s.W + (int64_t)e_r[e + u] * s.ldw + j) : 0.0;
#pragma unroll
              for (int u = 0; u < SAP_UNROLL; ++u) {
                if (e + u < ne) {
                  const double v = ((e_d[e + u] - w[u]) + e_p[e + u]) + pj;
                  if (sap_less(v, e_r[e + u], bv, br)) bv = v, br = e_r[e + u];
                }
              }
            }
          }
        }
        if (has) {
          if (bv < d - GAMMA_TIE) {
            d = bv;
            s.sp[j] = bv;
            s.pred[j] = br;
            if (o >= 0 && bv < best) {
              const int k = atomicAdd(&ctrl->sap_cnt[(t + 1) % 3], 1);
              s.sap_r[nb + k] = o;
              s.sap_d[nb + k] = bv;
              s.sap_p[nb + k] = ldm(s.profit + o);
            }
          }
          if (o < 0 && sap_less(d, j, lv, lj)) lv = d, lj = j;
        }
      }
      sap_block_min(lv, lj, sv, sj);
      if (tid == 0) s.pv1[((t + 1) & 1) * G + blockIdx.x] = lv, s.pj1[((t + 1) & 1) * G + blockIdx.x] = lj;
      if (lead) ctrl->sap_cnt[(t + 2) % 3] = 0;  // list t - 1: read before the last barrier
      grid.sync();
      sap_grid_min(s, (t + 1) & 1, best, sink, sv, sj, &ctrl->sap_cnt[(t + 1) % 3], cnt);
      rounds++;
    }
    if (err) break;
    if (lead) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(T2));
    // ---- JV dual update of the owned columns below the sink's distance, then the augmentation (as lap_augment_kernel)
    for (int j = j0 + tid; j < j1; j += SAP_THREADS) {
      const int o = ldm(s.owner + j);
      const double d = ldm(s.sp + j);
      if (o >= 0 && d < best) {  // (a person's profit is written by whichever CTA holds its column: through L2)
        const double dd = best - d;
        s.price[j] = ldm(s.price + j) + dd;
        s.profit[o] = ldm(s.profit + o) - dd;
      }
    }
    grid.sync();
    if (lead) {
      s.profit[f] = -best;
      int j = sink;
      for (int hop = 0;; ++hop) {
        const int r = ldm(s.pred + j);
        s.owner[j] = r;
        const int jn = ldm(s.col4row + r);
        s.col4row[r] = j;
        if (r == f || hop > s.n) break;
        j = jn;
      }
    }
    grid.sync();
    if (lead) {
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(T3));
      t_init += T1 - T0, t_rounds += T2 - T1, t_aug += T3 - T2;
    }
  }
  if (lead) {
    // (ns) distances from the free row, label-correcting rounds, dual update + augmentation; persons placed.  The
    // master/helper tail's slots: it has nothing to do after this kernel.
    s.counters->t_phase[4] += (long long)t_init;
    s.counters->t_phase[5] += (long long)t_rounds;
    s.counters->t_phase[6] += (long long)t_aug;
    s.counters->t_phase[7] += q;
    s.counters->aug_rows += q;
    s.counters->aug_steps += rounds;
    s.counters->rounds += rounds;  // dependent grid-wide rounds, like the tail rounds they replace
    s.counters->bytes += (rows + q) * (long long)m * 8;
    if (err == 1) s.counters->status |= 1;
    // round guard: the persons not yet placed go to lap_augment_kernel (the list stays ascending)
    const int left = err == 2 ? nfree - q : 0;
    for (int a = 0; a < left; ++a) freelist[a] = freelist[q + a];
    ctrl->cnt[cur_list] = left;
    ctrl->stalled = left > 0 ? 1 : 0;
    ctrl->in_tail = 0;
    ctrl->finished = 1;
  }
}

__global__ void __launch_bounds__(1024) lap_minmax_kernel(const double* __restrict__ W, int n, int m, int64_t ldw,
                                                          LapCtrl* ctrl, int* flags) {
  __shared__ double smin[32], smax[32];
  double lo = 1.0e300, hi = -1.0e300;
  const int64_t total = (int64_t)n * m;
  bool bad = false;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const double v = W[(e / m) * ldw + (e % m)];
    bad |= !isfinite(v);
    lo = fmin(lo, v);
    hi = fmax(hi, v);
  }
  if (bad) atomicOr(flags, 1);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if ((threadIdx.x & 31) == 0) {
    smin[threadIdx.x >> 5] = lo;
    smax[threadIdx.x >> 5] = hi;
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    lo = smin[threadIdx.x];
    hi = smax[threadIdx.x];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
      hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if (threadIdx.x == 0) {
      unsigned long long* pmin = reinterpret_cast<unsigned long long*>(&ctrl->wmin);
      unsigned long long old = *pmin;
      while (__longlong_as_double((long long)old) > lo) {
        const unsigned long long seen = atomicCAS(pmin, old, (unsigned long long)__double_as_longlong(lo));
        if (seen == old) break;
        old = seen;
      }
      unsigned long long* pmax = reinterpret_cast<unsigned long long*>(&ctrl->wmax);
      old = *pmax;
      while (__longlong_as_double((long long)old) < hi) {
        const unsigned long long seen = atomicCAS(pmax, old, (unsigned long long)__double_as_longlong(hi));
        if (seen == old) break;
        old = seen;
      }
    }
  }
}

__global__ void lap_ctrl_init_kernel(LapCtrl* ctrl, mcd_lap_counters* counters, int zero_counters) {
  ctrl->cnt[0] = ctrl->cnt[1] = 0;
  ctrl->progress[0] = ctrl->progress[1] = 0;
  ctrl->cur = 0;
  ctrl->stalled = 0;
  ctrl->wmin = 1.0e300;
  ctrl->wmax = -1.0e300;
  for (int q = 0; q < MAX_PHASES; ++q) ctrl->barrier[q] = 0u;
  ctrl->finished = 0;
  ctrl->in_tail = 0;
  ctrl->eps = 0.0;
  ctrl->nfail[0] = ctrl->nfail[1] = 0;
  ctrl->a_tie = ctrl->a_fallback = 0;
  if (zero_counters) {
    counters->rounds = counters->bids = counters->bytes = counters->aug_rows = counters->aug_steps = 0;
    counters->status = 0;
    for (int q = 0; q < 8; ++q) counters->t_phase[q] = 0, counters->a_ts[q] = 0, counters->a_hops[q] = 0;
  }
}

// objective = sum_i W[i, col4row[i]], fixed summation order (deterministic bits)
__global__ void __launch_bounds__(1024) lap_objective_kernel(const double* __restrict__ W, int n, int64_t ldw,
                                                             const int* __restrict__ col4row, double* out,
                                                             mcd_lap_counters* counters) {
  __shared__ double red[32];
  double acc = 0.0;
  int bad = 0;
  for (int i = threadIdx.x; i < n; i += 1024) {
    const int j = col4row[i];
    if (j < 0)
      bad = 1;
    else
      acc += W[(int64_t)i * ldw + j];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  bad = __syncthreads_or(bad);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    acc = red[threadIdx.x];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (threadIdx.x == 0) {
      if (out != nullptr) *out = acc;
      if (bad) counters->status = 1;
    }
  }
}


// ------------------------------------------------------------------------------------------------
// Classes of similar persons, closing step.  During the auction a person ignores the objects its own copies hold,
// so copies may sit at different profit levels: pi_A > pi_B for two copies A, B of one cell means B would prefer A's
// object -- harmless for the ASSIGNMENT (A and B are interchangeable) but not a dual-feasible point.  Raising the
// price of every copy's object until its profit equals the lowest profit of the class,
//     p[c(i)] <- W[i, c(i)] - min_{k in class(i)} (W[k, c(k)] - p[c(k)]),
// restores exact complementary slackness for everybody: the copy at the lowest level was at its best response
// against every object outside the class; the class's objects are now tight at that level; other persons only see
// prices rise on objects they do not hold; unassigned objects keep price 0.  (This is the bid of a similarity class
// in the auction for transportation problems, Bertsekas & Castanon 1989, applied once at the end.)  One CTA.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) lap_class_equalize_kernel(LapState s) {
  if (s.pcls == nullptr || s.flags[0]) return;
  unsigned long long* level = reinterpret_cast<unsigned long long*>(s.bval);  // [n] scratch: class id < n
  const int tid = threadIdx.x;
  for (int i = tid; i < s.n; i += 1024) level[i] = ~0ull;
  __syncthreads();
  for (int i = tid; i < s.n; i += 1024) {
    const int c = s.col4row[i];
    if (c >= 0) atomicMin(level + s.pcls[i], f64_sortable(s.W[(int64_t)i * s.ldw + c] - s.price[c]));
  }
  __syncthreads();
  for (int i = tid; i < s.n; i += 1024) {
    const int c = s.col4row[i];
    if (c < 0) continue;
    const double w = s.W[(int64_t)i * s.ldw + c];
    const double lvl = sortable_f64(level[s.pcls[i]]);
    const double pnew = w - lvl;
    if (pnew > s.price[c]) s.price[c] = pnew;
    s.profit[i] = w - s.price[c];
  }
}

// ------------------------------------------------------------------------------------------------
// Dual certificate of one solve (SURVEY.md appendix C, K3c) -- independent of HOW the assignment was found.
// Inputs: the cost block W, the assignment col4row and the object prices the solver ended with.  With
//   lambda = min price over the assigned objects,  q_j = max(price_j - lambda, 0) >= 0,  u_i = max_j (W_ij - q_j),
// (u, q) is feasible for the dual of the reference's ILP (macrodna.py:27-84: row sums <= 1, column sums <= 1,
// all n rows matched), so  D = sum_i u_i + sum_j q_j  bounds EVERY feasible objective from above, whatever the
// prices are.  The assignment's own objective is  P = sum_i W[i, c(i)], and
//   D - P = sum_i [u_i - (W[i, c(i)] - q_c(i))]  +  sum_{j unassigned} q_j  =: gap >= 0.
// gap == 0 (to rounding) proves optimality; gap / |P| is the certified relative distance from the optimum.
// Also checked: every person assigned, no object used twice.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) lap_cert_prepare_kernel(LapState s, mcd_lap_cert* cert) {
  __shared__ double red[32];
  __shared__ int bad_s;
  const int tid = threadIdx.x;
  if (tid == 0) bad_s = 0;
  for (int j = tid; j < s.m; j += 1024) s.pred[j] = 0;  // pred doubles as the "object used" marks
  __syncthreads();
  double lam = 1.0e300;
  int bad = 0;
  for (int i = tid; i < s.n; i += 1024) {
    const int c = s.col4row[i];
    if (c < 0 || c >= s.m) {
      bad++;
    } else {
      if (atomicExch(&s.pred[c], 1) != 0) bad++;
      lam = fmin(lam, s.price[c]);
    }
  }
  if (bad) atomicAdd(&bad_s, bad);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) lam = fmin(lam, __shfl_xor_sync(0xffffffffu, lam, o));
  if ((tid & 31) == 0) red[tid >> 5] = lam;
  __syncthreads();
  if (tid == 0) {
    for (int q = 1; q < 32; ++q) lam = fmin(lam, red[q]);
    cert->lambda = lam;
    cert->n_bad = bad_s;
    cert->max_violation = 0.0;
    cert->gap = 0.0;
    cert->rel_gap = 0.0;
  }
}

// one CTA per person (grid-stride): u_i over the whole row, violation against the matched edge -> s.gam[i]
__global__ void __launch_bounds__(256) lap_cert_rows_kernel(LapState s, const mcd_lap_cert* cert) {
  __shared__ double red[8];
  const int tid = threadIdx.x;
  const double lam = cert->lambda;
  for (int i = blockIdx.x; i < s.n; i += gridDim.x) {
    const double* w = s.W + (int64_t)i * s.ldw;
    double best = -1.0e300;
    if (s.vec) {
      int j = 2 * tid;
      for (; j + 3 * 512 + 1 < s.m; j += 4 * 512) {
        double2 wv[4], pv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) wv[u] = __ldg(reinterpret_cast<const double2*>(w + j + u * 512));
#pragma unroll
        for (int u = 0; u < 4; ++u) pv[u] = *reinterpret_cast<const double2*>(s.price + j + u * 512);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          best = fmax(best, wv[u].x - fmax(pv[u].x - lam, 0.0));
          best = fmax(best, wv[u].y - fmax(pv[u].y - lam, 0.0));
        }
      }
      for (; j < s.m; j += 512) {
        best = fmax(best, __ldg(w + j) - fmax(s.price[j] - lam, 0.0));
        if (j + 1 < s.m) best = fmax(best, __ldg(w + j + 1) - fmax(s.price[j + 1] - lam, 0.0));
      }
    } else {
      for (int j = tid; j < s.m; j += 256) best = fmax(best, __ldg(w + j) - fmax(s.price[j] - lam, 0.0));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = fmax(best, __shfl_xor_sync(0xffffffffu, best, o));
    if ((tid & 31) == 0) red[tid >> 5] = best;
    __syncthreads();
    if (tid == 0) {
#pragma unroll
      for (int q = 1; q < 8; ++q) best = fmax(best, red[q]);
      const int c = s.col4row[i];
      double viol = 0.0;
      if (c >= 0 && c < s.m) viol = best - (w[c] - fmax(s.price[c] - lam, 0.0));  // >= 0: c is one of the j
      s.gam[i] = viol;
    }
    __syncthreads();
  }
}

// fixed-order sums (deterministic bits): gap = sum of the row violations + the surplus price of unassigned objects
__global__ void __launch_bounds__(1024) lap_cert_finish_kernel(LapState s, mcd_lap_cert* cert, const double* objective,
                                                               double tol_rel, mcd_lap_counters* counters) {
  __shared__ double rs[32], rm[32];
  const int tid = threadIdx.x;
  const double lam = cert->lambda;
  double sum = 0.0, mx = 0.0;
  for (int i = tid; i < s.n; i += 1024) {
    const double v = s.gam[i];
    sum += v;
    mx = fmax(mx, v);
  }
  double surplus = 0.0;
  for (int j = tid; j < s.m; j += 1024)
    if (s.pred[j] == 0) surplus += fmax(s.price[j] - lam, 0.0);
  mx = fmax(mx, surplus);
  sum += surplus;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sum += __shfl_xor_sync(0xffffffffu, sum, o);
    mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((tid & 31) == 0) rs[tid >> 5] = sum, rm[tid >> 5] = mx;
  __syncthreads();
  if (tid == 0) {
    for (int q = 1; q < 32; ++q) sum += rs[q], mx = fmax(mx, rm[q]);
    const double P = objective != nullptr ? *objective : 0.0;
    // scale of the problem for the relative gap: |P|, or the summed |matched values| when P cancels
    const double scale = fmax(fabs(P), 1.0e-300);
    cert->gap = sum;
    cert->max_violation = mx;
    cert->rel_gap = sum / scale;
    cert->primal = P;
    if (cert->n_bad != 0 || !(sum <= tol_rel * scale + 1.0e-290)) counters->status |= 2;
  }
}

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

}  // namespace

size_t mcd_lap_workspace_bytes(int64_t n, int64_t m) {
  size_t b = 0;
  b += align_up(sizeof(LapCtrl), 256);
  b += align_up(m * 8, 256);            // price
  b += align_up(m * 4, 256);            // owner
  b += align_up(m * 8, 256);            // key
  b += align_up(n * 8, 256);            // profit
  b += align_up(n * 4, 256);            // bj
  b += 2 * align_up(n * 8, 256);        // gam, bval
  b += 2 * align_up(n * 4, 256);        // un lists
  b += align_up(n * LIST_K * 4, 256);   // lj
  b += align_up(n * LIST_K * 8, 256);   // lw
  b += align_up(n * 8, 256);            // lbound
  b += 2 * align_up(n * 4, 256) + align_up(2 * n * 4, 256);  // lvalid, done, fail (x2)
  b += 3 * align_up(MAX_GRID_SLOTS * 8, 256) + 2 * align_up(MAX_GRID_SLOTS * 4, 256);  // split-row partials
  b += align_up(m * 8, 256);            // sp
  b += align_up(m * 4, 256);            // pred
  b += align_up((n + 1) * 4, 256);      // sc_col
  b += align_up((n + 1) * 8, 256);      // sc_val
  b += align_up(m * 4, 256);            // ocls
  b += align_up(n * 8, 256);            // clevel
  b += align_up(m * 16, 256);           // pw
  b += align_up(2 * n * 4, 256) + 2 * align_up(2 * n * 8, 256);  // sap_r, sap_d, sap_p
  return b;
}

int mcd_launch_lap(mcd_context* h, const double* W, int64_t n, int64_t m, int64_t ldw, int32_t* col4row,
                   double* objective, void* work, mcd_lap_counters* d_counters, bool check_finite,
                   mcd_lap_cert* d_cert, double* prices_out, const int* person_class) {
  if (n <= 0) return MCD_OK;
  if (n > m) return mcd_fail(h, MCD_ERR_INVALID, "lap: rows must be the smaller side");
  if (m > 0x3fffffff) return mcd_fail(h, MCD_ERR_UNSUPPORTED, "lap: too many objects");
  LapState s;
  s.W = W;
  s.n = (int)n;
  s.m = (int)m;
  s.ldw = ldw;
  s.vec = ((reinterpret_cast<uintptr_t>(W) & 15) == 0) && ((ldw & 1) == 0);
  s.list_k = (int)(m < LIST_K ? m : LIST_K);
  char* p = static_cast<char*>(work);
  auto take = [&](size_t bytes) {
    char* r = p;
    p += align_up(bytes, 256);
    return r;
  };
  s.ctrl = reinterpret_cast<LapCtrl*>(take(sizeof(LapCtrl)));
  s.price = reinterpret_cast<double*>(take(m * 8));
  s.owner = reinterpret_cast<int*>(take(m * 4));
  s.key = reinterpret_cast<unsigned long long*>(take(m * 8));
  s.profit = reinterpret_cast<double*>(take(n * 8));
  s.bj = reinterpret_cast<int*>(take(n * 4));
  s.gam = reinterpret_cast<double*>(take(n * 8));
  s.bval = reinterpret_cast<double*>(take(n * 8));
  s.un[0] = reinterpret_cast<int*>(take(n * 4));
  s.un[1] = reinterpret_cast<int*>(take(n * 4));
  s.lj = reinterpret_cast<int*>(take(n * LIST_K * 4));
  s.lw = reinterpret_cast<double*>(take(n * LIST_K * 8));
  s.lbound = reinterpret_cast<double*>(take(n * 8));
  s.lvalid = reinterpret_cast<int*>(take(n * 4));
  s.fail = reinterpret_cast<int*>(take(2 * n * 4));  // double buffered by round parity
  s.done = reinterpret_cast<int*>(take(n * 4));
  s.pv1 = reinterpret_cast<double*>(take(MAX_GRID_SLOTS * 8));
  s.pv2 = reinterpret_cast<double*>(take(MAX_GRID_SLOTS * 8));
  s.pj1 = reinterpret_cast<int*>(take(MAX_GRID_SLOTS * 4));
  s.pj2 = reinterpret_cast<int*>(take(MAX_GRID_SLOTS * 4));
  s.pbound = reinterpret_cast<double*>(take(MAX_GRID_SLOTS * 8));
  const mcd_options& opt = h->opt;
  {
    int min_chunk = opt.lap_min_chunk < 2 ? 2 : opt.lap_min_chunk;
    int64_t mc2 = m / min_chunk;
    s.max_chunks = (int)(mc2 < 1 ? 1 : (mc2 > 256 ? 256 : mc2));
    s.chunk_waves = opt.lap_chunk_waves < 1 ? 1 : opt.lap_chunk_waves;  // swept at 10k x 50k: 1 -> 554 ms, 2 -> 570, 4 -> 577
  }
  s.sp = reinterpret_cast<double*>(take(m * 8));
  s.pred = reinterpret_cast<int*>(take(m * 4));
  s.sc_col = reinterpret_cast<int*>(take((n + 1) * 4));
  s.sc_val = reinterpret_cast<double*>(take((n + 1) * 8));
  s.ocls = reinterpret_cast<int*>(take(m * 4));
  s.clevel = reinterpret_cast<unsigned long long*>(take(n * 8));
  s.pw = reinterpret_cast<ulonglong2*>(take(m * 16));
  s.sap_r = reinterpret_cast<int*>(take(2 * n * 4));
  s.sap_d = reinterpret_cast<double*>(take(2 * n * 8));
  s.sap_p = reinterpret_cast<double*>(take(2 * n * 8));
  s.pcls = (n < m) ? person_class : nullptr;  // classes ride on the candidate-list bids, which only n < m uses
  s.col4row = col4row;
  s.counters = d_counters;
  s.flags = h->d_flags;
  double theta = opt.lap_theta;  // swept on 10k x 10k: 2 -> 55k rounds, 3 -> 34k, 4 -> 38k, 8 -> 51k
  if (!(theta > 1.0)) theta = 3.0;
  double eps0 = opt.lap_eps0;
  if (eps0 <= 0.0 && opt.lap_theta == 3.0 && n >= 4096) {
    // Large square steps, knobs untouched: start at range/27 and divide by 6.  Round counts of the eps schedules are
    // erratic (chains of single bidders whose length depends on where the previous phase left the prices); measured on
    // the square step of ten instances (round 2, scripts/research/gpu_sched.py): 10k x 10k 149 -> 113 ms and
    // 165 -> 145 ms (34.3k -> 23.6k, 41.9k -> 36.3k rounds), 1k x 1k 15.0 / 17.2 / 10.3 / 18.3 -> 12.2 / 12.6 / 15.2 /
    // 8.8 ms, 200 x 200 four instances 4-25 % slower (hence the size threshold).
    eps0 = 1.0 / 27.0;
    theta = 6.0;
  }
  const double eps_min_rel = opt.lap_eps_min > 0.0 ? opt.lap_eps_min : 1e-7;
  const bool square_scaling = (n == m && n > 1) && opt.lap_scaling != 0;
  s.max_rounds = opt.lap_max_rounds >= 1.0 ? (long long)opt.lap_max_rounds : 200000 + 64 * (long long)n;
  // measured (round 2): budget 2048 vs none: C3 31.7 -> 19.5 ms, C4 55.0 -> 39.7 ms, replicate sweep 20.4 -> 25.2 /s; at
  // m = 50 000 a Dijkstra step scans a 400 KB row (~20 us) and a budget of 2048 costs 512 vs 334 ms: hence m / 2
  // (budgets 2048 / 1024 / 512 / 256 at 200 x 400: 19.4 / 17.9 / 16.6 / 15.9 ms; at 1000 x 2000: 40.6 / 37.2 / 38.0 / 40.9 ms)
  s.prefetch_rows = opt.lap_prefetch_rows;
  s.scale_cut_nu = opt.lap_scale_cut < 0 ? 0 : opt.lap_scale_cut;
  s.scale_tail_rounds = opt.lap_scale_tail_rounds >= 0.0 ? (long long)opt.lap_scale_tail_rounds : (1ll << 60);
  s.tail_budget = opt.lap_tail_budget >= 1.0 ? (long long)opt.lap_tail_budget : (m / 2 > 1024 ? (long long)m / 2 : 1024);

  // eps phases: range/theta, range/theta^2, ... >= eps_min_rel * range, then the exact eps = 0 phase
  double factors[MAX_PHASES];
  int nphases = 0;
  if (square_scaling)
    for (double f = (eps0 > 0.0 ? eps0 : 1.0 / theta); f >= eps_min_rel && nphases < MAX_PHASES - 1; f /= theta)
      factors[nphases++] = f;
  factors[nphases++] = 0.0;

  // a solve that no-ops (non-finite input flag) must still leave a well-defined "nobody assigned" result behind:
  // the record / objective / certificate kernels index with col4row
  MCD_CUDA(h, cudaMemsetAsync(col4row, 0xFF, (size_t)n * 4, h->stream));
  lap_ctrl_init_kernel<<<1, 1, 0, h->stream>>>(s.ctrl, d_counters, 0);
  MCD_LAUNCH_CHECK(h, "lap_ctrl_init_kernel");
  if (square_scaling || check_finite) {
    lap_minmax_kernel<<<h->sm_count * 2, 1024, 0, h->stream>>>(W, s.n, s.m, ldw, s.ctrl, h->d_flags);
    MCD_LAUNCH_CHECK(h, "lap_minmax_kernel");
  }
  int per_sm = 0;
  MCD_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, lap_auction_kernel, LAP_THREADS, 0));
  if (per_sm < 1) return mcd_fail(h, MCD_ERR_CUDA, "lap_auction_kernel cannot be resident");
  int want = opt.lap_blocks_per_sm < 1 ? 1 : opt.lap_blocks_per_sm;
  int blocks = h->sm_count * (per_sm < want ? per_sm : want);
  if (opt.lap_grid_blocks > 0 && opt.lap_grid_blocks < blocks) blocks = opt.lap_grid_blocks;  // concurrent solves share the chip
  if (blocks > MAX_GRID_SLOTS) blocks = MAX_GRID_SLOTS;
  // Mode selection.
  //   n < m, short rows (m <= 16384)  : candidate lists everywhere + single-CTA narrow kernel (one SM sweeps a
  //                                     short row cheaply, and list failures are rare)
  //   n < m, long rows                : candidate lists in the rounds with >= a grid-full of bidders, split row
  //                                     sweeps below that, DSMEM cluster kernel for the narrow rounds
  //   n == m                          : no lists (eps-scaling inflates every price, a list would be rebuilt on
  //                                     almost every bid): split row sweeps + cluster kernel
  // single-CTA list tail only on request: the master/helper kernel is as fast or faster at every size measured
  // (C3 43.4 vs 44.3 ms, C4 82.8 vs 88.7 ms)
  const int list_max_m = opt.lap_list_max_m;
  int use_lists = (n < m) ? 1 : 0;
  if (opt.lap_lists >= 0) use_lists = opt.lap_lists ? 1 : 0;
  const bool list_tail = use_lists != 0 && m <= list_max_m;
  // long rows: lists only pay in the rounds with at least a grid-full of bidders (failed lists are then swept by
  // whole CTAs in parallel); below that every row is split over the grid instead
  int list_min_nu = opt.lap_list_min_nu;
  int cs = opt.lap_tail_cluster > 0 ? opt.lap_tail_cluster : (m >= 32768 ? CL_MAX_CS : 8);
  if (cs > CL_MAX_CS) cs = CL_MAX_CS;
  size_t tail_smem = 0;
  int mc = 0;
  bool cluster_tail = !list_tail && cs >= 1;
  if (cluster_tail) {
    mc = (int)((((m + cs - 1) / cs) + 1) & ~1LL);
    tail_smem = sizeof(TailPart) * CL_NU * CL_MAX_CS + sizeof(TailPacket) + sizeof(Top2) * CL_NU * TAIL_WARPS +
                2 * CL_NU * sizeof(int) + 2 * CL_MAX_CS * 4 + CL_NU * 12 + 32 + (size_t)mc * 12 + 64;
    if (tail_smem > 220 * 1024) cluster_tail = false;  // object slice does not fit: the wide kernel runs every round
  }
  // symmetric form of the scan-every-row cluster tail (every CTA resolves the round itself): default
  bool sym_tail = cluster_tail && opt.lap_tail_sym != 0 && !(n < m && opt.lap_tail_mh != 0);
  if (sym_tail && opt.lap_tail_cluster <= 0 && m >= 8192) {
    // measured (C5 square step, 10k objects): 16 CTAs 118.7 ms, 8 CTAs 124.3 ms, 4 CTAs 146.4 ms; at 1000 objects
    // 8 CTAs 15.6 ms, 16 CTAs 16.1 ms
    cs = CL_MAX_CS;
    mc = (int)((((m + cs - 1) / cs) + 1) & ~1LL);
  }
  if (sym_tail) {
    const size_t sym_smem = sizeof(SymPart) * 2 * CL_NU * CL_MAX_CS + sizeof(Top2) * CL_NU * TAIL_WARPS +
                            3 * CL_NU * sizeof(int) + 16 + CL_NU * 8 + 16 + (size_t)mc * 12 + 64;
    if (sym_smem > 220 * 1024)
      sym_tail = false;
    else
      tail_smem = sym_smem;
  }
  if (cluster_tail) {
    const void* tail_fn = sym_tail ? (const void*)lap_tail_sym_kernel : (const void*)lap_tail_cluster_kernel;
    MCD_CUDA(h, cudaFuncSetAttribute(tail_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tail_smem));
    if (cs > 8) MCD_CUDA(h, cudaFuncSetAttribute(tail_fn, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  }
  // n < m: master/helper tail (candidate lists certify ~90 % of the bids).  n == m: eps-scaling flattens every
  // person's values, ~90 % of the lists fail (measured), so the scan-every-row cluster kernel stays.
  bool mh_tail = cluster_tail && n < m;
  if (opt.lap_tail_mh >= 0) mh_tail = cluster_tail && opt.lap_tail_mh != 0;
  if (mh_tail && cs != 4 && cs != 8 && cs != 16) cs = 16;  // list slots per CTA = 128 / cs must be <= 32
  if (mh_tail) {
    mc = (int)((((m + cs - 1) / cs) + 1) & ~1LL);
    if (cs > 8)
      MCD_CUDA(h, cudaFuncSetAttribute(lap_tail_mh_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  }
  int tail_nu = list_tail ? TAIL_NU : (cluster_tail ? (mh_tail ? opt.lap_mh_nu : CL_NU) : 0);
  if (mh_tail && (tail_nu < 1 || tail_nu > MH_NU)) tail_nu = MH_NU;
  if (opt.lap_tail_nu >= 0 && opt.lap_tail_nu < tail_nu) tail_nu = opt.lap_tail_nu;

  int aug_nu = opt.lap_aug_nu;
  if (n == m && opt.lap_aug_nu_square >= 0) aug_nu = opt.lap_aug_nu_square;
  // asynchronous wide kernel: the exact phase of a rectangular step with candidate lists and the master/helper tail
  bool use_async = opt.lap_async != 0 && opt.deterministic == 0 && n < m && use_lists != 0 && mh_tail && tail_nu > 0 && s.pcls == nullptr &&
                   m >= 256 && nphases == 1 && s.list_k == LIST_K;
  int async_blocks = 0;
  const int async_threads = opt.lap_async_threads == 64 ? 64 : (opt.lap_async_threads == 256 ? 256 : 128);
  const void* async_fn = async_threads == 64    ? (const void*)lap_async_kernel<64>
                         : async_threads == 128 ? (const void*)lap_async_kernel<128>
                                                : (const void*)lap_async_kernel<256>;
  if (use_async) {
    int aper = 0;
    MCD_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&aper, async_fn, async_threads, 0));
    const int awant = opt.lap_async_blocks_per_sm > 0 ? opt.lap_async_blocks_per_sm : 16;
    if (aper < 1) {
      use_async = false;
    } else {
      async_blocks = h->sm_count * (aper < awant ? aper : awant);
      if (opt.lap_grid_blocks > 0 && opt.lap_grid_blocks < async_blocks) async_blocks = opt.lap_grid_blocks;
    }
  }
  // the asynchronous kernel stops at lap.sap_nu unassigned persons and lap_sap_kernel places them (instead of the
  // master/helper tail): a grid of one column slice per CTA (at most one 256-column wave each where the chip allows)
  bool use_sap = use_async && opt.lap_sap != 0;
  int sap_blocks = 0;
  if (use_sap) {
    int sper = 0;
    MCD_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&sper, lap_sap_kernel, SAP_THREADS, 0));
    sap_blocks = (int)((m + SAP_THREADS - 1) / SAP_THREADS);
    // more slices than SMs: the same number of CTAs on every SM (a round waits for the most loaded SM)
    if (sap_blocks > h->sm_count) sap_blocks = (sap_blocks + h->sm_count - 1) / h->sm_count * h->sm_count;
    if (sap_blocks > h->sm_count * sper) sap_blocks = h->sm_count * sper;
    if (sap_blocks > MAX_GRID_SLOTS / 2) sap_blocks = MAX_GRID_SLOTS / 2;  // two slots of best-free partials per CTA
    if (opt.lap_grid_blocks > 0 && opt.lap_grid_blocks < sap_blocks) sap_blocks = opt.lap_grid_blocks;
    if (sap_blocks < 1) use_sap = false;
  }
  const int scale_cut_nu = s.scale_cut_nu;
  const long long scale_tail_rounds = s.scale_tail_rounds;
  for (int ph = 0; ph < nphases; ++ph) {
    double factor = factors[ph];
    // the last lap.scale_full_phases scaling phases always run to completion: the exact phase needs their prices
    const bool may_cut = ph < nphases - 1 - opt.lap_scale_full_phases;
    s.scale_cut_nu = may_cut ? scale_cut_nu : 0;
    s.scale_tail_rounds = may_cut ? scale_tail_rounds : (1ll << 60);
    int rank_select = opt.lap_rank_select;
    if (use_async) {
      int stop_nu = opt.lap_async_stop > 0 && opt.lap_async_stop < tail_nu ? opt.lap_async_stop : tail_nu;
      int max_nu = MH_NU, cont = 0;
      if (use_sap) {
        stop_nu = opt.lap_sap_nu > 0 ? opt.lap_sap_nu : 1;
        if (stop_nu > max_nu) max_nu = stop_nu;
      }
      if (opt.lap_async_nu > tail_nu) {  // the rounds with more than lap.async_nu bidders stay round-synchronous
        int wide_stop = opt.lap_async_nu, no = 0;
        void* args[] = {&s, &factor, &ph, &wide_stop, &use_lists, &list_min_nu, &aug_nu, &rank_select, &no};
        MCD_CUDA(h, cudaLaunchCooperativeKernel((const void*)lap_auction_kernel, dim3(blocks), dim3(LAP_THREADS), args,
                                                0, h->stream));
        h->launches++;
        cont = 1;
      }
      int fallback_ok = cont == 0 ? 1 : 0;
      void* aargs[] = {&s, &stop_nu, &max_nu, &cont, &fallback_ok};
      MCD_CUDA(h, cudaLaunchCooperativeKernel(async_fn, dim3(async_blocks), dim3(async_threads), aargs, 0, h->stream));
      if (fallback_ok) {  // exact ties: the step is redone round-synchronously (a no-op launch otherwise)
        int yes = 1;
        void* args[] = {&s, &factor, &ph, &tail_nu, &use_lists, &list_min_nu, &aug_nu, &rank_select, &yes};
        MCD_CUDA(h, cudaLaunchCooperativeKernel((const void*)lap_auction_kernel, dim3(blocks), dim3(LAP_THREADS), args,
                                                0, h->stream));
        h->launches++;
      }
      if (use_sap) {  // a no-op after the fallback: that step ends in the tail kernels below, as without lap.sap
        void* sargs[] = {&s};
        MCD_CUDA(h, cudaLaunchCooperativeKernel((const void*)lap_sap_kernel, dim3(sap_blocks), dim3(SAP_THREADS), sargs,
                                                0, h->stream));
        h->launches++;
      }
    } else {
      int no = 0;
      void* args[] = {&s, &factor, &ph, &tail_nu, &use_lists, &list_min_nu, &aug_nu, &rank_select, &no};
      MCD_CUDA(h, cudaLaunchCooperativeKernel((const void*)lap_auction_kernel, dim3(blocks), dim3(LAP_THREADS), args, 0,
                                              h->stream));
    }
    h->launches++;
    if (tail_nu > 0 && list_tail) {
      lap_tail_list_kernel<<<1, TAIL_THREADS, 0, h->stream>>>(s);
      MCD_LAUNCH_CHECK(h, "lap_tail_list_kernel");
    } else if (tail_nu > 0 && cluster_tail) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(cs);
      cfg.blockDim = dim3(TAIL_THREADS);
      cfg.dynamicSmemBytes = mh_tail ? 0 : tail_smem;
      cfg.stream = h->stream;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = cs;
      attr[0].val.clusterDim.y = 1;
      attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
      if (mh_tail)
        MCD_CUDA(h, cudaLaunchKernelEx(&cfg, lap_tail_mh_kernel, s, mc));
      else if (sym_tail)
        MCD_CUDA(h, cudaLaunchKernelEx(&cfg, lap_tail_sym_kernel, s, mc));
      else
        MCD_CUDA(h, cudaLaunchKernelEx(&cfg, lap_tail_cluster_kernel, s, mc));
      h->launches++;
    }
  }
  if (s.pcls != nullptr) {
    lap_class_equalize_kernel<<<1, 1024, 0, h->stream>>>(s);
    MCD_LAUNCH_CHECK(h, "lap_class_equalize_kernel");
  }
  lap_augment_kernel<<<1, JV_THREADS, 0, h->stream>>>(s);
  MCD_LAUNCH_CHECK(h, "lap_augment_kernel");
  double* obj_dev = objective != nullptr ? objective : reinterpret_cast<double*>(s.sc_val);  // scratch when unwanted
  lap_objective_kernel<<<1, 1024, 0, h->stream>>>(W, s.n, ldw, col4row, obj_dev, d_counters);
  MCD_LAUNCH_CHECK(h, "lap_objective_kernel");
  if (d_cert != nullptr && h->opt.certify) {
    lap_cert_prepare_kernel<<<1, 1024, 0, h->stream>>>(s, d_cert);
    MCD_LAUNCH_CHECK(h, "lap_cert_prepare_kernel");
    int cert_blocks = h->sm_count * 8;
    if ((int64_t)cert_blocks > n) cert_blocks = (int)n;
    lap_cert_rows_kernel<<<cert_blocks, 256, 0, h->stream>>>(s, d_cert);
    MCD_LAUNCH_CHECK(h, "lap_cert_rows_kernel");
    lap_cert_finish_kernel<<<1, 1024, 0, h->stream>>>(s, d_cert, obj_dev, MCD_CERT_TOL_REL, d_counters);
    MCD_LAUNCH_CHECK(h, "lap_cert_finish_kernel");
  }
  if (prices_out != nullptr)
    MCD_CUDA(h, cudaMemcpyAsync(prices_out, s.price, (size_t)m * 8, cudaMemcpyDeviceToDevice, h->stream));
  return MCD_OK;
}

// Stand-alone certificate of ANY (assignment, prices) pair for the problem W -- the checker is usable on results
// that did not come from this solver (tests feed it SciPy's assignment with and without deliberate damage).
int mcd_launch_lap_certify(mcd_context* h, const double* W, int64_t n, int64_t m, int64_t ldw, const int32_t* col4row,
                           const double* prices, void* work, mcd_lap_cert* d_cert, mcd_lap_counters* d_counters) {
  if (n <= 0) return MCD_OK;
  LapState s = {};
  s.W = W;
  s.n = (int)n;
  s.m = (int)m;
  s.ldw = ldw;
  s.vec = ((reinterpret_cast<uintptr_t>(W) & 15) == 0) && ((ldw & 1) == 0) && ((reinterpret_cast<uintptr_t>(prices) & 15) == 0);
  s.price = const_cast<double*>(prices);
  s.col4row = const_cast<int*>(col4row);
  char* p = static_cast<char*>(work);
  s.pred = reinterpret_cast<int*>(p);
  p += align_up(m * 4, 256);
  s.gam = reinterpret_cast<double*>(p);
  p += align_up(n * 8, 256);
  double* obj = reinterpret_cast<double*>(p);
  lap_objective_kernel<<<1, 1024, 0, h->stream>>>(W, s.n, ldw, col4row, obj, d_counters);
  MCD_LAUNCH_CHECK(h, "lap_objective_kernel");
  lap_cert_prepare_kernel<<<1, 1024, 0, h->stream>>>(s, d_cert);
  MCD_LAUNCH_CHECK(h, "lap_cert_prepare_kernel");
  int cert_blocks = h->sm_count * 8;
  if ((int64_t)cert_blocks > n) cert_blocks = (int)n;
  lap_cert_rows_kernel<<<cert_blocks, 256, 0, h->stream>>>(s, d_cert);
  MCD_LAUNCH_CHECK(h, "lap_cert_rows_kernel");
  lap_cert_finish_kernel<<<1, 1024, 0, h->stream>>>(s, d_cert, obj, MCD_CERT_TOL_REL, d_counters);
  MCD_LAUNCH_CHECK(h, "lap_cert_finish_kernel");
  return MCD_OK;
}
