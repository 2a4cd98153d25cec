"""Multi-GPU driver: one process per GPU, NCCL over NVLink via torch.distributed (plumbing only).

Partitioning (SURVEY.md section 8e):

* K1 + K2 shard naturally -- RNA cells are independent rows of the contraction.  Rank r owns
  rows ``row_shard(M, P, r)``; the DNA operand (<= 1.6 GB) is standardised redundantly on
  every rank (cheaper than broadcasting it), so the contraction needs NO collective.
* The correlation shards are all-gathered once (``all_gather_into_tensor``, rows padded to
  ceil(M/P) per rank so shard r lands at row r*ceil(M/P)), C^T is rebuilt locally by a
  transpose kernel, and the assignment step loop runs replicated on every rank: the solver is
  deterministic, so all ranks hold bit-identical results and no further exchange is needed.
  (Why the solver is not sharded: DESIGN.md section 5.)
* Replicate sweeps (config 4) are "replicas only": ``replicate_owner`` maps replicate -> rank,
  no collective.
"""
from __future__ import annotations

import numpy as np

from . import _lib


def row_shard(M: int, world: int, rank: int):
    """Contiguous shard [lo, hi) of rank ``rank``; every shard but the last has ceil(M/world) rows."""
    per = -(-M // world)
    lo = min(M, rank * per)
    hi = min(M, lo + per)
    return lo, hi


def padded_rows(M: int, world: int) -> int:
    return -(-M // world) * world


def replicate_owner(replicate: int, world: int) -> int:
    """Replicate r of a resampling sweep runs on rank r mod P (no collective)."""
    return replicate % world


def gather_rows(local, M: int, world: int):
    """All-gather row shards laid out by ``row_shard`` into the full [M, cols] matrix.

    ``local`` is this rank's [ceil(M/world), cols] buffer (rows beyond the shard are padding).
    Works with any torch.distributed backend (NCCL on the GPU box, gloo in the CPU tests).
    """
    import torch
    import torch.distributed as dist

    per = -(-M // world)
    assert local.shape[0] == per
    full = torch.empty((per * world,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    if world == 1:
        full.copy_(local)
    else:
        dist.all_gather_into_tensor(full, local.contiguous())
    return full[:M]


class ShardedCell2Cell:
    """The hot path on ``world`` GPUs (world == 1: a single fused C-ABI call)."""

    def __init__(self, handle, M, N, G, world, rank, device, precision="ozaki"):
        self.h, self.M, self.N, self.G = handle, M, N, G
        self.world, self.rank, self.device = world, rank, device
        self.precision = precision
        if precision == "ozaki":
            # the digit format of the fused single-GPU driver; exact int32 accumulation bounds the gene count of the
            # integer path, longer rows take the FP64 pipe there too
            self.nsl, self.rb, exact = handle.ozaki_format(M, N, G)
            if not exact:
                self.precision = "fp64"
        self.lo, self.hi = row_shard(M, world, rank)
        self._bufs = None

    # ---- single GPU: the fused driver does everything ------------------------------------------
    def _single(self, rna, dna, in_space):
        assign, step, objs, stats = self.h.cell2cell(rna, dna, self.M, self.N, self.G, in_space=in_space,
                                                     precision=self.precision)
        return {"assign": assign, "step": step, "objs": objs, "stats": stats.as_dict()}

    def _alloc(self):
        import torch

        if self._bufs is None:
            lib = self.h.lib
            per = -(-self.M // self.world)
            ldc = (self.N + 1) & ~1
            ldct = (self.M + 1) & ~1
            f64 = dict(dtype=torch.float64, device=self.device)
            m_loc = max(1, self.hi - self.lo)  # operand buffers hold exactly this rank's rows
            if self.precision == "fp64":
                ldk = lib.mcd_padded_k(self.G)
                ops = dict(a=torch.empty((m_loc, ldk), **f64), b=torch.empty((self.N, ldk), **f64))
            elif self.precision == "ozaki":
                ldk = lib.mcd_padded_k_split(self.G)
                nsl = self.nsl
                i8 = dict(dtype=torch.int8, device=self.device)
                ops = dict(a=torch.empty((nsl, m_loc, ldk), **i8), b=torch.empty((nsl, self.N, ldk), **i8),
                           sa=torch.empty(m_loc, **f64), sb=torch.empty(self.N, **f64), nsl=nsl)
            else:
                ldk = lib.mcd_padded_k_split(self.G)
                i16 = dict(dtype=torch.int16, device=self.device)
                ops = dict(a=torch.empty((2, m_loc, ldk), **i16), b=torch.empty((2, self.N, ldk), **i16))
            self._bufs = dict(
                per=per, ldk=ldk, ldc=ldc, ldct=ldct,
                na=torch.empty(per, **f64), nb=torch.empty(self.N, **f64),
                c_loc=torch.zeros((per, ldc), **f64), ct=torch.empty((self.N, ldct), **f64),
                rna_dev=None, dna_dev=None, **ops,
            )
        return self._bufs

    def _standardize_and_correlate(self, b, rna_loc, dna, m_loc, events, ext):
        """K1 (both operands) + K2 of this rank's row block in the configured precision; C only (no C^T)."""
        lib, h, chk = self.h.lib, self.h.h, self.h.check
        G, N = self.G, self.N
        pa, pb, na, nb = b["a"].data_ptr(), b["b"].data_ptr(), b["na"].data_ptr(), b["nb"].data_ptr()
        c, ldc, ldk = b["c_loc"].data_ptr(), b["ldc"], b["ldk"]
        if self.precision == "fp64":
            chk(lib.mcd_standardize(h, rna_loc.data_ptr(), m_loc, G, G, pa, na))
            chk(lib.mcd_standardize(h, dna.data_ptr(), N, G, G, pb, nb))
            events[1].record(ext)
            chk(lib.mcd_corr_fp64(h, pa, m_loc, pb, N, G, ldk, na, nb, c, ldc, None, 0))
        elif self.precision == "ozaki":
            sa, sb, nsl, rb = b["sa"].data_ptr(), b["sb"].data_ptr(), b["nsl"], self.rb
            chk(lib.mcd_standardize_ozaki_radix(h, rna_loc.data_ptr(), m_loc, G, G, pa, nsl, rb, sa, na))
            chk(lib.mcd_standardize_ozaki_radix(h, dna.data_ptr(), N, G, G, pb, nsl, rb, sb, nb))
            events[1].record(ext)
            chk(lib.mcd_corr_ozaki_radix(h, pa, m_loc, pb, N, G, ldk, nsl, rb, sa, sb, na, nb, c, ldc, None, 0))
        else:
            chk(lib.mcd_standardize_split(h, rna_loc.data_ptr(), m_loc, G, G, pa, na))
            chk(lib.mcd_standardize_split(h, dna.data_ptr(), N, G, G, pb, nb))
            events[1].record(ext)
            chk(lib.mcd_corr_split(h, pa, m_loc, pb, N, G, ldk, na, nb, c, ldc, None, 0))

    def _sharded(self, rna_loc, dna):
        """rna_loc: this rank's [hi-lo, G] device tensor; dna: [N, G] device tensor."""
        import torch

        b = self._alloc()
        lib, h = self.h.lib, self.h.h
        ext = torch.cuda.ExternalStream(lib.mcd_stream(h), device=self.device)
        m_loc = self.hi - self.lo
        e = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        e[0].record(ext)
        self._standardize_and_correlate(b, rna_loc, dna, m_loc, e, ext)
        e[2].record(ext)
        with torch.cuda.stream(ext):
            c_full = gather_rows(b["c_loc"], self.M, self.world)
        self.h.check(lib.mcd_transpose_f64(h, c_full.data_ptr(), self.M, self.N, b["ldc"], b["ct"].data_ptr(),
                                           b["ldct"]))
        e[3].record(ext)
        assign, step, objs, stats = self.h.lap_steps(c_full.data_ptr(), b["ldc"], b["ct"].data_ptr(), b["ldct"],
                                                     self.M, self.N)
        e[4].record(ext)
        self.h.check(lib.mcd_check_finite(h))
        d = stats.as_dict()
        d["ms_standardize"] = e[0].elapsed_time(e[1])
        d["ms_corr"] = e[1].elapsed_time(e[2])
        d["ms_gather"] = e[2].elapsed_time(e[3])
        d["ms_total"] = e[0].elapsed_time(e[4])
        d["ms_h2d"] = 0.0
        d["kernel_launches"] = d["kernel_launches"] + 4
        return {"assign": assign, "step": step, "objs": objs, "stats": d}

    # ---- public --------------------------------------------------------------------------------
    def run_device(self, rna_loc, dna):
        if self.world == 1:
            return self._single(rna_loc.data_ptr(), dna.data_ptr(), _lib.MEM_DEVICE)
        return self._sharded(rna_loc, dna)

    def run_host(self, rna_host, dna_host):
        """Pinned host tensors in, host numpy results out (H2D and D2H inside the call)."""
        import torch

        if self.world == 1:
            return self._single(rna_host.data_ptr(), dna_host.data_ptr(), _lib.MEM_HOST)
        b = self._alloc()
        ext = torch.cuda.ExternalStream(self.h.lib.mcd_stream(self.h.h), device=self.device)
        dlo, dhi = row_shard(self.N, self.world, self.rank)
        per_d = -(-self.N // self.world)
        if b["rna_dev"] is None:
            b["rna_dev"] = torch.empty(rna_host.shape, dtype=torch.float64, device=self.device)
            b["dna_part"] = torch.zeros((per_d, self.G), dtype=torch.float64, device=self.device)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(ext):
            e0.record(ext)
            # every rank needs the whole DNA operand, but only 1/P of it crosses ITS PCIe link: the rest arrives
            # over NVLink (all-gather of the raw row shards), which is ~10x faster than P redundant host copies
            if dhi > dlo:
                b["dna_part"][: dhi - dlo].copy_(dna_host[dlo:dhi], non_blocking=True)
            b["rna_dev"].copy_(rna_host, non_blocking=True)
            dna_dev = gather_rows(b["dna_part"], self.N, self.world)
            e1.record(ext)
        out = self._sharded(b["rna_dev"], dna_dev)
        out["stats"]["ms_h2d"] = e0.elapsed_time(e1)
        out["stats"]["ms_total"] += out["stats"]["ms_h2d"]
        out["h2d_bytes"] = int(rna_host.numel() * 8 + (dhi - dlo) * self.G * 8)
        return out


def sweep_assignments(handle, rna: np.ndarray, dna: np.ndarray, replicate_cols, world=1, rank=0, precision="ozaki",
                      reuse_corr=True, concurrency=8):
    """Resampling-stability sweep (config 4; reference
    ``Resampling_stability_analyses/CRC_data_analyses/clonal_proportions_resampling.py:172-201``, run there under
    ``multiprocessing.Pool(20)``, ``:297-306``): replicate r is the hot path on ``dna[replicate_cols[r]]`` (DNA cells
    resampled with replacement).  Replicas only: rank ``r mod world`` runs replicate r, no collective.

    ``reuse_corr`` (declared optimisation, SURVEY.md section 8e): a replicate only gathers DNA cells and the genes are
    untouched, so its correlation matrix is a column gather of the base matrix -- the base matrix is computed once
    per rank and the rank's replicates run as ONE ``mcd_subinstance_sweep`` call that keeps ``concurrency`` of them
    in flight on the GPU (same values bit for bit: the same kernels compute them).  ``reuse_corr=False`` recomputes
    everything per replicate like the reference does.
    Returns {replicate index: (assign, step, objs)} for this rank's replicates.
    """
    out = {}
    M, G = rna.shape
    mine = [r for r in range(len(replicate_cols)) if replicate_owner(r, world) == rank]
    if not mine:
        return out
    if reuse_corr:
        handle.cell2cell(rna, dna, M, dna.shape[0], G, precision=precision)
        by_len = {}
        for r in mine:
            by_len.setdefault(len(replicate_cols[r]), []).append(r)
        for n_sub, group in by_len.items():
            cols = np.stack([np.asarray(replicate_cols[r], dtype=np.int32) for r in group])
            assign, step, objs, _, _ = handle.subinstance_sweep(cols, M=M, concurrency=concurrency)
            for k, r in enumerate(group):
                out[r] = (assign[k], step[k], objs[k])
        return out
    for r in mine:
        sub = np.ascontiguousarray(dna[np.asarray(replicate_cols[r])])
        assign, step, objs, _ = handle.cell2cell(rna, sub, M, sub.shape[0], G, precision=precision)
        out[r] = (assign, step, objs)
    return out


def replicate_accuracy(assign, cols, rna_clone, dna_clone):
    """Per-replicate clone accuracy of the reference's sweep (clonal_proportions_resampling.py:191-201): the share of
    RNA cells whose predicted DNA cell carries the RNA cell's own clone label.  ``assign`` holds positions in ``cols``."""
    pred = np.asarray(dna_clone)[np.asarray(cols)[np.asarray(assign)]]
    return float(np.mean(pred == np.asarray(rna_clone)))
