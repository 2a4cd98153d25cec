"""Research: finish an auction's last unassigned persons with label-correcting shortest augmenting paths.

NumPy restatement of lap_sap_kernel (csrc/lap.cu), and the go / no-go count for it.  From the naive (eps = 0)
Jacobi auction stopped at `stop` unassigned persons, every free person f (ascending) gets one augmenting path:

  d[j] = -W[f, j] + p[j]                                        (min-form: reduced cost of the free row, u_f = 0)
  best = min over free columns of d                             (ties: smaller column)
  round: frontier = owned columns whose d improved last round and is still below best; every column j takes
         min over frontier entries (k, r = owner[k]) of ((d[k] - W[r, j]) + profit[r]) + p[j]  (ties: smaller r),
         and keeps it if it is below d[j] by more than GAMMA_TIE; then best is recomputed
  stop when the frontier is empty: the sink is the free column at best (smaller index on ties), the JV dual update
  touches the columns below the sink's distance, and the path is flipped along pred.

The rounds are Jacobi (a round reads the distances of the previous one), as on the GPU, where every CTA owns a
slice of the columns and pulls the frontier rows into it.  Reported per step: label-correcting rounds, rows
relaxed, the largest frontier, the Dijkstra pops of the present single-CTA kernel (= its dependent row scans), and
the auction rounds the present tail needs from the same state.

    python scripts/research/sim_lcsap.py C4 64            # synth instance, hand-over at 64 persons
    python scripts/research/sim_lcsap.py C5 64 0.2        # C5 shapes scaled by 0.2
    python scripts/research/sim_lcsap.py dump.npy 64      # a correlation matrix from dump_corr.py
"""
import sys
import time

import numpy as np

GAMMA_TIE = 1.4210854715202004e-14  # lap.cu: an improvement must be larger than this


def top2(V):
    j1 = V.argmax(axis=1)
    r = np.arange(V.shape[0])
    v1 = V[r, j1]
    V[r, j1] = -np.inf
    j2 = V.argmax(axis=1)
    v2 = V[r, j2]
    V[r, j1] = v1
    return v1, j1, v2, j2


def auction_until(W, stop_nu, max_rounds=10**7):
    """Naive Jacobi forward auction (eps = 0) for n <= m, until at most stop_nu persons are unassigned."""
    n, m = W.shape
    p = np.zeros(m)
    owner = -np.ones(m, int)
    col = -np.ones(n, int)
    profit = np.zeros(n)
    un = np.arange(n)
    rounds = 0
    while un.size > stop_nu and rounds < max_rounds:
        if m == 1:
            v1, j1 = W[un, 0] - p[0], np.zeros(un.size, int)
            v2 = np.full(un.size, -np.inf)
        else:
            v1, j1, v2, j2 = top2(W[un] - p)
        gam = np.where(np.isfinite(v2), v1 - v2, 0.0)
        win = {}
        for k in np.lexsort((un, gam.astype(np.float32))):
            win[j1[k]] = k
        won = np.zeros(un.size, bool)
        nxt = []
        for j, k in win.items():
            if owner[j] < 0 or gam[k] > 0:
                if owner[j] >= 0:
                    col[owner[j]] = -1
                    nxt.append(owner[j])
                owner[j] = un[k]
                col[un[k]] = j
                p[j] += gam[k]
                profit[un[k]] = v1[k] - gam[k]
                won[k] = True
        nxt.extend(un[~won].tolist())
        rounds += 1
        un = np.array(sorted(nxt), int)
    return p, owner, col, profit, un, rounds


def dijkstra_pops(W, p, owner, profit, f):
    """Pops of the present kernel's Dijkstra for free person f (read only)."""
    d = -W[f] + p
    settled = np.zeros(W.shape[1], bool)
    pops = 0
    while True:
        key = np.where(settled, np.inf, d)
        v = key.min()
        cand = np.flatnonzero(key == v)
        free = cand[owner[cand] < 0]
        j = free[0] if free.size else cand[0]
        pops += 1
        settled[j] = True
        if owner[j] < 0:
            return pops
        r = owner[j]
        nd = ((v - W[r]) + profit[r]) + p
        upd = (nd < d) & ~settled
        d[upd] = nd[upd]


def lcsap_person(W, p, owner, col, profit, f):
    """One augmenting path for free person f by label-correcting rounds; updates the duals and the matching in
    place.  Returns (rounds, rows relaxed, largest frontier)."""
    n, m = W.shape
    d = -W[f] + p
    pred = np.full(m, f)
    changed = np.ones(m, bool)
    freecol = owner < 0
    if not freecol.any():
        raise ValueError("no free column")
    best = d[freecol].min()
    rounds = rows = maxf = 0
    while True:
        front = np.flatnonzero(changed & ~freecol & (d < best))
        if front.size == 0:
            break
        rounds += 1
        rows += front.size
        maxf = max(maxf, front.size)
        dk = d[front].copy()  # Jacobi: the round reads last round's distances
        rr = owner[front]
        cand = ((dk[:, None] - W[rr]) + profit[rr][:, None]) + p[None, :]
        # min over entries, ties to the smaller row
        order = np.lexsort((rr,))
        cand, rr = cand[order], rr[order]
        a = cand.argmin(axis=0)
        v = cand[a, np.arange(m)]
        upd = v < d - GAMMA_TIE
        d[upd] = v[upd]
        pred[upd] = rr[a[upd]]
        changed = upd
        best = d[freecol].min()
    sink = int(np.flatnonzero(freecol & (d == best))[0])
    sc = ~freecol & (d < best)
    delta = best - d[sc]
    p[sc] += delta
    profit[owner[sc]] -= delta
    profit[f] = -best
    j = sink
    while True:
        r = pred[j]
        jn = col[r]
        owner[j] = r
        col[r] = j
        if r == f:
            break
        j = jn
    return rounds, rows, maxf


def solve(W, stop):
    """Auction to `stop` unassigned persons, then label-correcting augmenting paths: col4row, prices."""
    p, owner, col, profit, un, _ = auction_until(W, stop)
    for f in sorted(un.tolist()):
        lcsap_person(W, p, owner, col, profit, f)
    return col, p


def step_report(W, stop):
    n, m = W.shape
    t0 = time.time()
    p, owner, col, profit, un, r_stop = auction_until(W, stop)
    *_, r_full = auction_until(W, 0)
    pops = rounds = rows = maxf = 0
    for f in sorted(un.tolist()):
        pops += dijkstra_pops(W, p, owner, profit, f)
        a, b, c = lcsap_person(W, p, owner, col, profit, f)
        rounds, rows, maxf = rounds + a, rows + b, max(maxf, c)
    from scipy.optimize import linear_sum_assignment

    r_, c_ = linear_sum_assignment(W, maximize=True)
    ok = bool((col[r_] == c_).all())
    nf = max(len(un), 1)
    print("%dx%d free=%d auction_tail_rounds=%d dijkstra_pops=%d lc_rounds=%d (%.1f/person) rows=%d max_frontier=%d "
          "opt=%s (%.0f s)" % (n, m, len(un), r_full - r_stop, pops, rounds, rounds / nf, rows, maxf, ok,
                               time.time() - t0), flush=True)
    return col


def main():
    src, stop = sys.argv[1], int(sys.argv[2])
    scale = float(sys.argv[3]) if len(sys.argv) > 3 else 1.0
    sys.path.insert(0, __file__.rsplit("/scripts/", 1)[0])
    if src.endswith(".npy"):
        C = np.load(src)
    else:
        from macrodna_b200 import synth
        from oracle import restatement as R

        m0, n0, g, k = synth.CONFIG_SHAPES[src]
        inst = synth.make_arrays(int(m0 * scale), int(n0 * scale), g, k, seed=1234 + int(src[1:]))
        C = R.correlation_matrix(inst.rna, inst.dna)
    act = np.arange(C.shape[0])
    N = C.shape[1]
    while act.size > N:  # rectangular steps (persons = DNA cells)
        W = np.ascontiguousarray(C[act].T)
        col = step_report(W, stop)
        keep = np.ones(act.size, bool)
        keep[col] = False
        act = act[keep]


if __name__ == "__main__":
    main()
