"""Host-side mirror of the reference's public class (the drop-in boundary).

``MaCroDNA(rna_df, dna_df, dna_label)`` with ``cell2cell_assignment()`` /
``cell2clone_assignment()`` / ``tiny_test()`` keeps the constructor, method names,
return schemas and observable side effects of
``/root/reference/src/MaCroDNA/macrodna.py:10-17, 86-199, 201-237``.  Pandas gene
intersection and index bookkeeping stay on the host (north star); everything
numeric -- standardisation, correlation matrix, the per-step assignment solves and
the step loop -- runs in the CUDA library behind the C ABI
(``include/macrodna_b200.h``) through ctypes.  No CPU fallback exists.
"""
from __future__ import annotations

import os

import numpy as np
import pandas as pd

from . import _lib

_HANDLES = {}


def get_handle(device: int = 0, slot: int = 0) -> "_lib.Handle":
    """Per-process, per-device library context (created on first use, so instances pickle).

    The reference's sweep scripts run the class in the parent and then fork a ``multiprocessing.Pool``
    (clonal_proportions_resampling.py:266-267, :300): a CUDA context does not survive ``fork()``, so a handle
    inherited from another process is never touched.  A child that inherited one is told how to run instead
    (CUDA cannot be re-initialised in a forked child); a child of a parent that had not used the GPU yet simply
    creates its own context."""
    key = device if slot == 0 else (device, slot)  # slot > 0: a further context on the same device (devices=[0, 0])
    h = _HANDLES.get(key)
    if h is not None and getattr(h, "pid", None) != os.getpid():
        # inherited over fork(): the parent had already initialised CUDA in this address space
        raise RuntimeError(
            "macrodna_b200: this process was fork()ed from a process that had already used the GPU (pid %s); CUDA "
            "cannot be re-initialised in a forked child.  Start the workers with "
            "multiprocessing.get_context('spawn') (or 'forkserver'), or run the replicates in the parent with "
            "MaCroDNA.subinstance_assignment / macrodna_b200.dist.sweep_assignments, which keep many replicates in "
            "flight on the GPU." % (h.pid,))
    if h is None or h.h is None:
        h = _lib.Handle(device)
        _HANDLES[key] = h
    return h


def get_handles(devices) -> list:
    """One context per entry of ``devices`` (a device may be listed more than once: separate contexts on it)."""
    seen = {}
    out = []
    for d in devices:
        d = int(d)
        out.append(get_handle(d, seen.get(d, 0)))
        seen[d] = seen.get(d, 0) + 1
    return out


def _check_devices(devices):
    """``devices=`` as a list of device ordinals (None stays None); refused before any GPU call if an entry is not a
    non-negative integer."""
    if devices is None:
        return None
    out = []
    for d in devices:
        if isinstance(d, bool) or not isinstance(d, (int, np.integer)) or d < 0:
            raise ValueError("devices must be non-negative CUDA device ordinals, got %r" % (d,))
        out.append(int(d))
    return out


class _StatsDict:
    """Merged stats of a two-call run, with the ``as_dict`` / attribute access of ``_lib.McdStats``."""

    def __init__(self, d):
        self._d = d

    def as_dict(self):
        return dict(self._d)

    def __getattr__(self, k):
        try:
            return self._d[k]
        except KeyError:
            raise AttributeError(k) from None


class MaCroDNA:
    """B200 drop-in for the reference class (``macrodna.py:10``).

    Parameters mirror ``macrodna.py:11``: ``rna_df`` / ``dna_df`` are genes x cells
    frames (index = gene ids, columns = cell ids, ``:13``); ``dna_label`` has columns
    ``clone`` and ``cell`` (``:14``).  Keyword-only extras default to reference behaviour:

    * ``devices``: list of CUDA devices of this node; more than one shards the correlation work by RNA rows
      (``mcd_cell2cell_multi``), results identical to one device, and deals the replicates of
      :meth:`leave_one_out_sweep` and :meth:`subinstance_sweep` over all of them (each device works on its own copy of
      the correlation matrix, made on the first such call after a run);
    * ``precision``: ``"ozaki"`` (default: FP64-equivalent correlations from the int8 tcgen05 tensor cores, exact
      digit-slice products, ~1e-12 absolute), ``"fp64"`` (FP64 tensor pipe, DMMA) or ``"split"`` (tcgen05 fp16
      hi/lo split precision, ~3e-7 absolute);
    * ``clone_column``: ``"predict_clone"`` (README.md:201, CRC_data_analysis/macrodna.py:195) or
      ``"predict"`` (src/MaCroDNA/macrodna.py:198);
    * ``verbose``: print the reference's progress lines (``:95-98,120,124,147``);
    * ``variant``: return signature of ``cell2cell_assignment`` -- the reference repo carries nine copies of the
      class with drifting signatures (SURVEY.md section 2.2): ``"src"`` ``(res, tagged)``;
      ``"objective"`` ``(res, tagged, sum(objVal))`` (random_assignment_test.py:196);
      ``"median"`` ``(res, tagged, sum, median matched corr)`` (random_assignment_test_median.py:196-199);
      ``"loo"`` ``(res, tagged[predicted_dna_cell, step, corr_val] indexed by rna_cell, sum, n_iters)``
      (run_loo_experiment.py:194-199); ``"resampling"`` tagged frame only with columns
      ``predicted_dna_cell, rna_cell, step`` and no index (clonal_proportions_resampling.py:166-169).
    """

    def __init__(self, rna_df=None, dna_df=None, dna_label=None, *, device=0, devices=None, precision="ozaki",
                 clone_column="predict_clone", verbose=False, variant="src"):
        self._genes = None  # shared genes of the last run: the frames below are filtered lazily (see rna_df)
        self.rna_df = rna_df
        self.dna_df = dna_df
        self.dna_label = dna_label
        # devices=[d0, d1, ...]: the RNA rows are sharded over these GPUs for standardisation + correlation (no exchange
        # inside the contraction), the shards meet on d0 over NVLink and d0 runs the step loop (mcd_cell2cell_multi)
        self.devices = _check_devices(devices)
        self.device = self.devices[0] if self.devices else device
        self.precision = precision
        self.clone_column = clone_column
        self.verbose = verbose
        if variant not in ("src", "objective", "median", "loo", "resampling"):
            raise ValueError("unknown variant %r" % (variant,))
        self.variant = variant
        self.keep_corr_val = variant in ("median", "loo")
        self.last_corr_val = None   # matched correlation per RNA cell (variants "median" / "loo")
        self.last_stats = None      # dict of CUDA-event timings / solver counters of the last call
        self.last_objective = None  # per-step objective (the `m.objVal` of each reference `ilp` call)
        self.last_assign = None     # int32 DNA column per RNA cell
        self.last_step = None       # int32 1-based step per RNA cell
        self.last_loo = None        # leave_one_out_sweep: left-out cells, certificate gaps, stats

    # -- the frames.  The reference overwrites self.rna_df / self.dna_df with the gene-filtered frames
    #    (macrodna.py:90-91).  Here the filtering of the DATA happens on the device (index gather in K1), so the
    #    host frames are only re-indexed if somebody actually looks at them after a run.
    @property
    def rna_df(self):
        if self._genes is not None and self._rna_df is not None and not self._rna_filtered:
            self._rna_df = self._rna_df.loc[self._genes, :]
            self._rna_filtered = True
        return self._rna_df

    @rna_df.setter
    def rna_df(self, df):
        self._rna_df = df
        self._rna_filtered = False
        self._genes = None
        self._resident_token = None  # the resident correlation matrix belongs to the old frames

    @property
    def dna_df(self):
        if self._genes is not None and self._dna_df is not None and not self._dna_filtered:
            self._dna_df = self._dna_df.loc[self._genes, :]
            self._dna_filtered = True
        return self._dna_df

    @dna_df.setter
    def dna_df(self, df):
        self._dna_df = df
        self._dna_filtered = False
        self._genes = None
        self._resident_token = None

    # -- host bookkeeping -------------------------------------------------------------------------
    def _shared_genes(self):
        """macrodna.py:89 -- set intersection; canonical order = DNA-frame order.
        Returns (genes, column of each gene in the DNA block, column of each gene in the RNA block)."""
        rna_index = self._rna_df.index
        dna_index = self._dna_df.index
        if not dna_index.is_unique or not rna_index.is_unique:
            raise ValueError("duplicate gene labels in the expression / copy-number index")
        pos_in_rna = rna_index.get_indexer(dna_index)
        keep = pos_in_rna >= 0
        if not keep.any():
            raise ValueError("rna_df and dna_df share no genes")
        dna_pos = np.flatnonzero(keep).astype(np.int32)
        rna_pos = pos_in_rna[keep].astype(np.int32)
        return dna_index[keep], dna_pos, rna_pos

    @staticmethod
    def _duplicate_dna_cells(dna_cells, dna_np):
        """Duplicated DNA cell ids WITH identical data (a frame built by ``dna.loc[:, resampled_names]``).  Returns
        (row of the first copy of every distinct cell, for every column the position of its cell among those) or None."""
        first = {}
        for k, c in enumerate(dna_cells):
            first.setdefault(c, k)
        if len(first) == len(dna_cells):
            return None
        first_pos = np.array([first[c] for c in dna_cells])
        if not np.array_equal(dna_np, dna_np[first_pos]):
            return None  # same label, different data: genuinely different cells
        uniq = np.array(sorted(first.values()))
        rank = {k: r for r, k in enumerate(uniq.tolist())}
        return uniq, np.array([rank[k] for k in first_pos.tolist()], dtype=np.int32)

    @staticmethod
    def _cells_by_genes(df):
        """macrodna.py:93-94 -- ``df.T.to_numpy()`` as C-contiguous float64 (cells x all genes of the frame).
        For a single-dtype float64 frame this is a zero-copy view of the frame's block."""
        try:
            a = df.to_numpy(dtype=np.float64).T
        except (TypeError, ValueError) as e:
            raise ValueError("non-numeric data in input frame: %s" % e) from None
        return np.ascontiguousarray(a)

    def _run(self):
        if self._rna_df is None or self._dna_df is None:
            raise ValueError("rna_df and dna_df are required")
        dna_cells = list(self._dna_df.columns)  # macrodna.py:87
        rna_cells = list(self._rna_df.columns)  # macrodna.py:88
        if len(set(rna_cells)) != len(rna_cells):
            # the reference dies later with "1 is not in list" (macrodna.py:159-160)
            raise ValueError("duplicate RNA cell ids")
        if len(rna_cells) == 0 or len(dna_cells) == 0:
            raise ValueError("empty input frame")
        genes, dna_pos, rna_pos = self._shared_genes()
        dna_np = self._cells_by_genes(self._dna_df)  # [N, all DNA genes]
        rna_np = self._cells_by_genes(self._rna_df)  # [M, all RNA genes]
        M, N, G = rna_np.shape[0], dna_np.shape[0], len(genes)
        # identity gathers are dropped (same genes, same order: the common preprocessed case)
        if G == dna_np.shape[1] and (dna_pos == np.arange(G, dtype=np.int32)).all():
            dna_pos = None
        if G == rna_np.shape[1] and (rna_pos == np.arange(G, dtype=np.int32)).all():
            rna_pos = None
        if self.verbose:
            print("number of cells in dna data %s" % N)
            print("number of cells in rna data %s" % M)
            print("number of genes in dna data %s" % G)
            print("number of genes in rna data %s" % G)
            q, r = divmod(M, N)
            print(q, r)
            print("MaCroDNA will be run for %s steps" % (q + (1 if r else 0)))
        h = get_handle(self.device)
        dup_cols = self._duplicate_dna_cells(dna_cells, dna_np)
        if dup_cols is not None:
            # A resampled DNA frame (`dna.loc[:, names]` with names drawn WITH replacement,
            # clonal_proportions_resampling.py:184-190): the correlation matrix is computed on the distinct cells and
            # the step loop runs on its column gather (exact ties between the copies are broken deterministically,
            # see mcd_subinstance_steps in include/macrodna_b200.h).
            uniq, cols = dup_cols
            dna_u = np.ascontiguousarray(dna_np[uniq])
            h.set_option("corr_only", 1)
            try:
                _, _, _, stats = h.cell2cell(rna_np, dna_u, M, len(uniq), G, ld_rna=rna_np.shape[1],
                                             ld_dna=dna_u.shape[1], precision=self.precision, rna_gene_idx=rna_pos,
                                             dna_gene_idx=dna_pos)
            finally:
                h.set_option("corr_only", 0)
            assign, step, objs, stats2 = h.subinstance(None, cols, M=M, N=len(uniq))
            d = stats.as_dict()
            d2 = stats2.as_dict()
            for k in ("ms_lap", "lap_rounds", "lap_bids", "lap_bytes", "lap_aug_rows", "lap_aug_steps", "cert_rel_gap",
                      "cert_max_violation", "cert_bad", "cert_steps", "step_rounds", "step_bids", "step_cert_gap", "n_steps"):
                d[k] = d2[k]
            d["ms_total"] += d2["ms_total"]
            d["kernel_launches"] += d2["kernel_launches"]
            stats = _StatsDict(d)
        elif self.devices and len(self.devices) > 1:
            assign, step, objs, stats = _lib.cell2cell_multi(get_handles(self.devices), rna_np, dna_np, M, N, G,
                                                             ld_rna=rna_np.shape[1], ld_dna=dna_np.shape[1],
                                                             precision=self.precision, rna_gene_idx=rna_pos,
                                                             dna_gene_idx=dna_pos)
        else:
            assign, step, objs, stats = h.cell2cell(rna_np, dna_np, M, N, G, ld_rna=rna_np.shape[1],
                                                    ld_dna=dna_np.shape[1], precision=self.precision,
                                                    rna_gene_idx=rna_pos, dna_gene_idx=dna_pos)
        # macrodna.py:90-91: from now on the frames are the gene-filtered ones (materialised on first access)
        if not self._rna_filtered or not self._dna_filtered or self._genes is None:
            self._genes = genes
        if (assign < 0).any():
            raise ValueError("unassigned RNA cell")  # list.index(1), macrodna.py:160
        self.last_assign, self.last_step, self.last_objective = assign, step, objs
        self.last_stats = stats.as_dict()
        # the correlation matrix of THIS run stays on the device until the handle's next cell2cell call
        if dup_cols is None:
            h.resident_token = self._resident_token = object()
            self._resident_shape = (M, N)
            self._resident_cells = (rna_cells, dna_cells)
            self.last_corr_val = h.last_match_values(M) if self.keep_corr_val else None
        else:
            self._resident_token = None  # the resident matrix is the distinct-cell one: later views recompute
            self.last_corr_val = (h.corr_pairs(np.arange(M, dtype=np.int32), dup_cols[1][assign])
                                  if self.keep_corr_val else None)
        if self.verbose:
            for o in objs:
                print("Obj: %g" % o)
            print("the number of associations in the correspondence matrix %s" % float(M))
        return rna_cells, dna_cells, assign, step

    # -- public API -------------------------------------------------------------------------------
    def cell2cell_assignment(self):
        """macrodna.py:86-186.  Returns ``(df[predict_cell], df[predict_cell, step])``, index ``cell``,
        rows in RNA input-column order, ``step`` 1-based."""
        rna_cells, dna_cells, assign, step = self._run()
        pred = [dna_cells[j] for j in assign.tolist()]
        tmp_result = pd.DataFrame(list(zip(pred, rna_cells)), columns=["predict_cell", "cell"])
        tmp_result = tmp_result.set_index("cell")  # macrodna.py:164-165
        tmp_result_tagged = pd.DataFrame(list(zip(pred, rna_cells, step.tolist())),
                                         columns=["predict_cell", "cell", "step"])
        if self.variant == "resampling":
            return pd.DataFrame(list(zip(pred, rna_cells, step.tolist())),
                                columns=["predicted_dna_cell", "rna_cell", "step"])
        if self.variant == "loo":
            tagged = pd.DataFrame(list(zip(pred, rna_cells, step.tolist(), self.last_corr_val.tolist())),
                                  columns=["predicted_dna_cell", "rna_cell", "step", "corr_val"]).set_index("rna_cell")
            return tmp_result, tagged, float(np.sum(self.last_objective)), int(len(self.last_objective))
        tmp_result_tagged = tmp_result_tagged.set_index("cell")  # macrodna.py:182-184
        if self.variant == "objective":
            return tmp_result, tmp_result_tagged, float(np.sum(self.last_objective))
        if self.variant == "median":
            return (tmp_result, tmp_result_tagged, float(np.sum(self.last_objective)),
                    float(np.median(self.last_corr_val)))
        return tmp_result, tmp_result_tagged

    # -- views of the resident correlation matrix (replicate sweeps, leave-one-out) -----------------
    def _ensure_resident(self):
        h = get_handle(self.device)
        if getattr(self, "_resident_token", None) is None or getattr(h, "resident_token", None) is not self._resident_token:
            self._run()  # the reference recomputes `corrs` on every call anyway (run_loo_experiment.py:217-221)
        return h

    def _view_handles(self):
        """The handles a sweep deals its replicates over: the one holding the resident matrix, then (``devices=`` with
        more than one entry) one per further device holding a copy of it, made once per run."""
        h = self._ensure_resident()
        if not self.devices or len(self.devices) < 2:
            return [h]
        hs = get_handles(self.devices)
        if self._resident_token is None or any(x.resident_token is not self._resident_token for x in hs[1:]):
            _lib.share_resident(hs)
        return hs

    def _sub_indices(self, rna_cells, dna_cells):
        """Rows / columns of the resident matrix for a replicate of cell ids (None = all cells, in order), and the
        selected ids."""
        all_rna, all_dna = self._resident_cells
        rows = cols = None
        sel_rna, sel_dna = all_rna, all_dna
        if rna_cells is not None:
            pos = {c: k for k, c in enumerate(all_rna)}
            sel_rna = list(rna_cells)
            if len(set(sel_rna)) != len(sel_rna):
                raise ValueError("duplicate RNA cell ids")
            rows = np.array([pos[c] for c in sel_rna], dtype=np.int32)
        if dna_cells is not None:
            pos = self._dna_positions()
            sel_dna = list(dna_cells)
            cols = np.array([pos[c] for c in sel_dna], dtype=np.int32)
        return rows, cols, sel_rna, sel_dna

    def _dna_positions(self):
        """DNA cell id -> column of the resident matrix (its first copy)."""
        pos = {}
        for k, c in enumerate(self._resident_cells[1]):
            pos.setdefault(c, k)
        return pos

    def subinstance_assignment(self, rna_cells=None, dna_cells=None):
        """Re-run the step loop on a replicate that only gathers cells of the frames of the last run: ``dna_cells``
        may repeat and drop DNA cell ids (``new_dna = dna.loc[:, names]``, clonal_proportions_resampling.py:184-190;
        run_dna_batch_removal_exp.py), ``rna_cells`` selects RNA cells.  The correlation matrix is NOT recomputed
        (genes are untouched: the replicate's matrix is an index gather of the resident one).  Returns the
        ``"resampling"`` frame ``[predicted_dna_cell, rna_cell, step]`` (clonal_proportions_resampling.py:166-169)."""
        h = self._ensure_resident()
        M, N = self._resident_shape
        rows, cols, sel_rna, sel_dna = self._sub_indices(rna_cells, dna_cells)
        assign, step, objs, stats = h.subinstance(rows, cols, M=M, N=N)
        self.last_sub = {"assign": assign, "step": step, "objs": objs, "stats": stats.as_dict()}
        pred = [sel_dna[j] for j in assign.tolist()]
        return pd.DataFrame(list(zip(pred, sel_rna, step.tolist())), columns=["predicted_dna_cell", "rna_cell", "step"])

    def subinstance_sweep(self, dna_cells_list, rna_cells=None, concurrency=8):
        """Every replicate of ``dna_cells_list`` (each a list of DNA cell ids of the last run's frames, repeats and
        omissions allowed) against the RNA cells ``rna_cells`` (None = all) in batched calls
        (``mcd_subinstance_sweep``, ``concurrency`` solves in flight per device, over all of ``devices``): the
        reference's resampling and DNA-removal sweeps (clonal_proportions_resampling.py:172-201,
        run_dna_batch_removal_exp.py).  Returns the list of ``"resampling"`` frames a loop of
        :meth:`subinstance_assignment` returns, frame for frame (replicates with duplicated DNA cells have exact ties:
        any of the tied optima is returned, with the same objectives).  Per-replicate objectives, certificate gaps
        and the stats go to ``self.last_sweep``."""
        reps = [list(c) for c in dna_cells_list]
        if not reps:
            raise ValueError("dna_cells_list is empty")
        if any(len(c) == 0 for c in reps):
            raise ValueError("a replicate has no DNA cells")
        hs = self._view_handles()
        M, N = self._resident_shape
        rows, _, sel_rna, _ = self._sub_indices(rna_cells, None)
        m = M if rows is None else rows.size
        pos = self._dna_positions()
        cols = [np.array([pos[c] for c in rep], dtype=np.int32) for rep in reps]
        # one batched call per replicate width (DNA-removal replicates may differ in size)
        by_width = {}
        for r, c in enumerate(cols):
            by_width.setdefault(c.size, []).append(r)
        frames = [None] * len(reps)
        objs, gaps, stats = [None] * len(reps), np.empty(len(reps)), []
        for idx in by_width.values():
            block = np.stack([cols[r] for r in idx])
            if len(hs) == 1:
                a, s, o, g, st = hs[0].subinstance_sweep(block, rna_rows=rows, M=m, concurrency=concurrency)
            else:
                a, s, o, g, st = _lib.subinstance_sweep_multi(hs, block, rna_rows=rows, M=m, concurrency=concurrency)
            stats.append(st.as_dict())
            for k, r in enumerate(idx):
                pred = [reps[r][j] for j in a[k].tolist()]
                frames[r] = pd.DataFrame(list(zip(pred, sel_rna, s[k].tolist())),
                                         columns=["predicted_dna_cell", "rna_cell", "step"])
                objs[r], gaps[r] = o[k], g[k]
        self.last_sweep = {"objs": objs, "cert_gap": gaps, "stats": stats}
        return frames

    def leave_one_out(self, cell_idx, K_steps, biopsy_name=None):
        """run_loo_experiment.py:201-319.  The RNA cell at position ``cell_idx`` is removed, the step loop runs on the
        remaining cells (``np.delete(corrs, cell_idx, 0)``, :224), and the left-out cell takes the DNA cell of
        highest correlation that has at most ``K_steps - 1`` matches (:298-309).  Returns
        ``(frame[predicted_dna_cell, step, corr_val] indexed by rna_cell, sum of the objective values)``; the left-out
        cell's row carries ``step == "TEST"``."""
        h = self._ensure_resident()
        rna_cells, dna_cells = self._resident_cells
        M, N = self._resident_shape
        if not 0 <= cell_idx < M:
            raise IndexError("pop index out of range")  # rna_cells.pop(cell_idx), :206
        rows = np.delete(np.arange(M, dtype=np.int32), cell_idx)
        if rows.size:
            assign, step, objs, _ = h.subinstance(rows, None, M=M, N=N)
            vals = h.corr_pairs(rows, assign)
        else:
            assign = np.empty(0, dtype=np.int32)
            step = np.empty(0, dtype=np.int32)
            objs = vals = np.empty(0)
        cell_corr = h.corr_rows([cell_idx], N)[0]                     # np.take(corrs, cell_idx, axis=0), :226
        cnt = np.bincount(assign, minlength=N)                       # np.count_nonzero(tagged, axis=0), :296
        eligible = cnt <= (K_steps - 1)                              # :298
        test_col, test_corr = -1, 0.0
        for idx_ in np.argsort(cell_corr)[::-1]:                     # :300-309
            if eligible[idx_]:
                test_col, test_corr = int(idx_), float(cell_corr[idx_])
                break
        return self._loo_frame(cell_idx, assign, step, vals, objs, test_col, test_corr, biopsy_name)

    def _loo_frame(self, cell_idx, assign, step, vals, objs, test_col, test_corr, biopsy_name):
        """The ``(tagged, objective)`` of one leave-one-out replicate (run_loo_experiment.py:246-319): the remaining
        cells with their DNA cell, step and matched correlation, then the left-out cell's ``"TEST"`` row if a DNA
        cell was eligible (``test_col >= 0``); the objective is ``float(sum(obj_scores))`` in the reference's order."""
        rna_cells, dna_cells = self._resident_cells
        res_dna = [dna_cells[j] for j in assign.tolist()]
        res_rna = [c for k, c in enumerate(rna_cells) if k != cell_idx]
        res_tag = step.tolist()
        res_val = vals.tolist()
        obj_scores = [float(o) for o in objs]
        if test_col >= 0:
            res_dna.append(dna_cells[test_col])
            res_rna.append(rna_cells[cell_idx])
            res_tag.append("TEST")
            obj_scores.append(test_corr)
            res_val.append(test_corr)
        tagged = pd.DataFrame(list(zip(res_dna, res_rna, res_tag, res_val)),
                              columns=["predicted_dna_cell", "rna_cell", "step", "corr_val"]).set_index("rna_cell")
        if self.verbose:
            print("name of the left-out RNA cell %s from sample %s" % (rna_cells[cell_idx], biopsy_name))
        return tagged, float(sum(obj_scores))

    def leave_one_out_sweep(self, cell_idx=None, K_steps=None, biopsy_name=None, frames=False, concurrency=8):
        """Every leave-one-out replicate of ``cell_idx`` (positions as in :meth:`leave_one_out`; None = every RNA
        cell) in one call (``mcd_loo_sweep``): the solves are kept ``concurrency`` at a time in flight on the GPU.
        ``K_steps`` defaults to ``ceil(M / N)``, what run_loo_experiment.py passes.

        Returns a frame indexed by ``rna_cell`` (the left-out cells, in ``cell_idx`` order) with columns
        ``predicted_dna_cell`` (None when no DNA cell is eligible), ``corr_val`` and ``objective``; per-replicate
        certificate gaps and the stats go to ``self.last_loo``.  ``frames=True`` returns instead the list of
        ``(tagged, objective)`` a loop of ``leave_one_out(q, K_steps, biopsy_name)`` returns."""
        if self._rna_df is None or self._dna_df is None:
            raise ValueError("rna_df and dna_df are required")
        M, N = len(self._rna_df.columns), len(self._dna_df.columns)
        cells = list(range(M)) if cell_idx is None else [int(q) for q in cell_idx]
        if not cells:
            raise ValueError("cell_idx is empty")
        for q in cells:
            if not 0 <= q < M:
                raise IndexError("pop index out of range")  # rna_cells.pop(cell_idx), run_loo_experiment.py:206
        if K_steps is None:
            K_steps = -(-M // N) if N else 1
        K_steps = int(K_steps)
        if K_steps < 1:
            raise ValueError("K_steps must be >= 1")
        dna_cells = list(self._dna_df.columns)
        if len(set(dna_cells)) != len(dna_cells) and \
                self._duplicate_dna_cells(dna_cells, self._cells_by_genes(self._dna_df)) is not None:
            raise ValueError("leave_one_out_sweep: the DNA frame repeats cells with identical data (a resampled frame); "
                             "its correlation matrix is computed on the distinct cells, so leave-one-out replicates "
                             "cannot be taken from it -- pass the frame of distinct DNA cells")
        hs = self._view_handles()
        rna_cells, dna_cells = self._resident_cells
        M, N = self._resident_shape
        if len(hs) == 1:
            res, stats = hs[0].loo_sweep(cells, K_steps, M, N, full=frames, concurrency=concurrency)
        else:
            res, stats = _lib.loo_sweep_multi(hs, cells, K_steps, M, N, full=frames, concurrency=concurrency)
        self.last_loo = {"cells": np.asarray(cells), "cert_gap": res["cert_gap"], "stats": stats.as_dict()}
        if frames:
            return [self._loo_frame(q, res["assign"][r], res["step"][r], res["match_corr"][r], res["step_obj"][r],
                                    int(res["test_col"][r]), float(res["test_corr"][r]), biopsy_name)
                    for r, q in enumerate(cells)]
        if self.verbose:
            for q in cells:
                print("name of the left-out RNA cell %s from sample %s" % (rna_cells[q], biopsy_name))
        pred = [dna_cells[j] if j >= 0 else None for j in res["test_col"].tolist()]
        return pd.DataFrame({"predicted_dna_cell": pred, "corr_val": res["test_corr"], "objective": res["total"]},
                            index=pd.Index([rna_cells[q] for q in cells], name="rna_cell"))

    def cell2clone_assignment(self):
        """macrodna.py:188-199: cell2cell + ``dna_label.set_index("cell").loc[predict_cell]["clone"]``."""
        if self.dna_label is None:
            raise ValueError("dna_label is required for cell2clone_assignment")
        if self.variant != "src":
            raise ValueError("cell2clone_assignment uses the 'src' return signature")
        rna_result, _ = self.cell2cell_assignment()
        dna_label = self.dna_label.set_index("cell")
        rna_result[self.clone_column] = dna_label.loc[rna_result["predict_cell"]]["clone"].tolist()
        return rna_result

    def tiny_test(self):
        """The fixed 4 DNA x 4 RNA x 6-gene case of macrodna.py:201-237 (RNA carries an extra gene g7)."""
        dna_data = pd.DataFrame.from_dict({"cell1": [2, 2, 3, 1, 6, 2], "cell2": [2, 2, 2, 2, 2, 2],
                                           "cell3": [1, 1, 2, 2, 2, 3], "cell4": [2, 2, 2, 2, 2, 6],
                                           "gene": ["g1", "g2", "g3", "g4", "g5", "g6"]}).set_index("gene")
        rna_data = pd.DataFrame.from_dict({"cell1": [0, 0, 10, 0, 20, 0, 0], "cell2": [2, 2, 2, 2, 2, 2, 0],
                                           "cell3": [0, 0, 2, 2, 0, 5, 0], "cell4": [1, 1, 1, 1, 1, 20, 0],
                                           "gene": ["g1", "g2", "g3", "g4", "g5", "g6", "g7"]}).set_index("gene")
        dna_cluster = pd.DataFrame.from_dict({"clone": [0, 1, 2, 3], "cell": ["cell1", "cell2", "cell3", "cell4"]})
        print("******Test DNA data is:")
        print(dna_data)
        print("******Test RNA data is:")
        print(rna_data)
        print("******Clone id for each DNA cell is:")
        print(dna_cluster)
        print("**********")
        print("Start Mapping RNA cells to DNA clones")
        print("**********")
        self.dna_df, self.rna_df, self.dna_label = dna_data, rna_data, dna_cluster
        out = self.cell2clone_assignment()
        print("**********")
        print("Finish Mapping")
        print("Test Success")
        print("**********")
        return out


class random_test:
    """Mirror of ``random_test`` (Resampling_stability_analyses/BE_data_analyses/random_assignment_test.py:198-258):
    random step-wise injective assignments over the correlation matrix, as the null distribution of the objective.
    The matrix is computed once on the device (the constructor runs the hot path); ``assign()`` returns the sum of
    the matched correlations of ONE random assignment like the reference, drawn from batches generated by
    ``mcd_null_assignments``; ``assign_many`` returns a whole batch (optionally with the medians of
    random_assignment_test_median.py).  Same distribution as the reference, not NumPy's random stream; every trial is
    the draw written down at ``mcd_null_assignments`` (include/macrodna_b200.h), up to 2^24 cells a side.
    ``devices=[d0, d1, ...]``: the trials are split over these GPUs (``mcd_null_assignments_multi``), bit for bit
    the draws of one device."""

    def __init__(self, rna_df=None, dna_df=None, *, device=0, devices=None, precision="ozaki", seed=2023, batch=4096):
        self._m = MaCroDNA(rna_df, dna_df, device=device, devices=devices, precision=precision)
        self._m._run()
        self.dna_cells, self.rna_cells = list(self._m._resident_cells[1]), list(self._m._resident_cells[0])
        M, N = self._m._resident_shape
        self.quotient, self.remainder = divmod(M, N)
        self.n_iters = self.quotient + (1 if self.remainder else 0)
        self._seed, self._batch, self._buf, self._pos, self._draws = int(seed), int(batch), None, 0, 0

    def assign_many(self, trials, seed=None, medians=False):
        hs = self._m._view_handles()
        seed = self._seed if seed is None else seed
        if len(hs) == 1:
            return hs[0].null_assignments(trials, seed, medians=medians)
        return _lib.null_assignments_multi(hs, trials, seed, medians=medians)

    def assign(self):
        if self._buf is None or self._pos >= len(self._buf):
            self._buf = self.assign_many(self._batch, seed=self._seed + 7919 * self._draws)
            self._draws += 1
            self._pos = 0
        v = float(self._buf[self._pos])
        self._pos += 1
        return v
