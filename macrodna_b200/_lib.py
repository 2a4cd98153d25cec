"""ctypes binding of ``libmacrodna_b200.so`` (C ABI in ``include/macrodna_b200.h``).

There is no fallback: if the library is missing or no B200 is visible, every
entry point raises.  Nothing here imports torch or the oracle.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmacrodna_b200.so")

MCD_OK = 0
MCD_ERR_INVALID = -1
MCD_ERR_CUDA = -2
MCD_ERR_NOMEM = -3
MCD_ERR_NONFINITE = -4
MCD_ERR_UNSUPPORTED = -5
MCD_ERR_NOT_CONVERGED = -6

PREC = {"fp64": 0, "split": 1, "ozaki": 2}
MEM_HOST, MEM_DEVICE = 0, 1
MAX_STEP_STATS = 64


class McdStats(C.Structure):
    _fields_ = [
        ("ms_h2d", C.c_double),
        ("ms_standardize", C.c_double),
        ("ms_corr", C.c_double),
        ("ms_lap", C.c_double),
        ("ms_d2h", C.c_double),
        ("ms_total", C.c_double),
        ("n_steps", C.c_int64),
        ("kernel_launches", C.c_int64),
        ("lap_rounds", C.c_int64),
        ("lap_bids", C.c_int64),
        ("lap_bytes", C.c_int64),
        ("lap_aug_rows", C.c_int64),
        ("lap_aug_steps", C.c_int64),
        ("lap_cycles", C.c_int64 * 8),
        ("step_ms", C.c_double * MAX_STEP_STATS),
        ("step_rounds", C.c_int64 * MAX_STEP_STATS),
        ("step_bids", C.c_int64 * MAX_STEP_STATS),
        ("cert_rel_gap", C.c_double),
        ("cert_max_violation", C.c_double),
        ("cert_bad", C.c_int64),
        ("cert_steps", C.c_int64),
        ("step_cert_gap", C.c_double * MAX_STEP_STATS),
        ("sweep_fallbacks", C.c_int64),
    ]

    def as_dict(self):
        n = min(int(self.n_steps), MAX_STEP_STATS)
        d = {k: getattr(self, k) for k, _ in self._fields_[:13]}
        d["lap_cycles"] = [self.lap_cycles[i] for i in range(8)]
        d["step_ms"] = [self.step_ms[i] for i in range(n)]
        d["step_rounds"] = [self.step_rounds[i] for i in range(n)]
        d["step_bids"] = [self.step_bids[i] for i in range(n)]
        for k in ("cert_rel_gap", "cert_max_violation", "cert_bad", "cert_steps", "sweep_fallbacks"):
            d[k] = getattr(self, k)
        d["step_cert_gap"] = [self.step_cert_gap[i] for i in range(n)]
        return d


# name -> (restype, argtypes); the exact list of symbols include/macrodna_b200.h declares
_VP, _I, _I64, _D = C.c_void_p, C.c_int, C.c_int64, C.c_double
SIGNATURES = {
    "mcd_abi_version": (_I, []),
    "mcd_strerror": (C.c_char_p, [_I]),
    "mcd_create": (_I, [C.POINTER(_VP), _I]),
    "mcd_destroy": (_I, [_VP]),
    "mcd_last_error": (C.c_char_p, [_VP]),
    "mcd_device_sm_count": (_I, [_VP]),
    "mcd_synchronize": (_I, [_VP]),
    "mcd_stream": (_VP, [_VP]),
    "mcd_set_option": (_I, [_VP, C.c_char_p, _D]),
    "mcd_get_option": (_I, [_VP, C.c_char_p, C.POINTER(_D)]),
    "mcd_padded_k": (_I64, [_I64]),
    "mcd_padded_k_split": (_I64, [_I64]),
    "mcd_num_steps": (_I64, [_I64, _I64]),
    "mcd_standardize": (_I, [_VP, _VP, _I64, _I64, _I64, _VP, _VP]),
    "mcd_standardize_split": (_I, [_VP, _VP, _I64, _I64, _I64, _VP, _VP]),
    "mcd_ozaki_default_slices": (_I, []),
    "mcd_ozaki_slices_for": (_I, [_I64, _I64, _I64]),
    "mcd_ozaki_slices": (_I, [_VP, _I64, _I64, _I64]),
    "mcd_ozaki_format": (_I, [_VP, _I64, _I64, _I64, C.POINTER(_I), C.POINTER(_I)]),
    "mcd_standardize_ozaki": (_I, [_VP, _VP, _I64, _I64, _I64, _VP, _I, _VP, _VP]),
    "mcd_standardize_ozaki_radix": (_I, [_VP, _VP, _I64, _I64, _I64, _VP, _I, _I, _VP, _VP]),
    "mcd_corr_ozaki": (_I, [_VP, _VP, _I64, _VP, _I64, _I64, _I64, _I, _VP, _VP, _VP, _VP, _VP, _I64, _VP, _I64]),
    "mcd_corr_ozaki_radix": (_I, [_VP, _VP, _I64, _VP, _I64, _I64, _I64, _I, _I, _VP, _VP, _VP, _VP, _VP, _I64, _VP,
                                  _I64]),
    "mcd_check_finite": (_I, [_VP]),
    "mcd_corr_fp64": (_I, [_VP, _VP, _I64, _VP, _I64, _I64, _I64, _VP, _VP, _VP, _I64, _VP, _I64]),
    "mcd_corr_split": (_I, [_VP, _VP, _I64, _VP, _I64, _I64, _I64, _VP, _VP, _VP, _I64, _VP, _I64]),
    "mcd_transpose_f64": (_I, [_VP, _VP, _I64, _I64, _I64, _VP, _I64]),
    "mcd_last_match_values": (_I, [_VP, _VP, _I64, _I]),
    "mcd_lap_max": (_I, [_VP, _VP, _I64, _I64, _I64, _VP, _VP]),
    "mcd_lap_max_certified": (_I, [_VP, _VP, _I64, _I64, _I64, _VP, _VP, _VP, _VP]),
    "mcd_lap_certify": (_I, [_VP, _VP, _I64, _I64, _I64, _VP, _VP, _VP]),
    "mcd_subinstance_steps": (_I, [_VP, _VP, _I64, _VP, _I64, _VP, _VP, _VP, _I, C.POINTER(McdStats)]),
    "mcd_subinstance_sweep": (_I, [_VP, _I64, _VP, _I64, _VP, _I64, _VP, _VP, _VP, _VP, _I, C.POINTER(McdStats)]),
    "mcd_loo_sweep": (_I, [_VP, _VP, _I64, _I64, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I, C.POINTER(McdStats)]),
    "mcd_corr_rows": (_I, [_VP, _VP, _I64, _VP, _I]),
    "mcd_corr_pairs": (_I, [_VP, _VP, _VP, _I64, _VP]),
    "mcd_null_assignments": (_I, [_VP, _I64, C.c_uint64, _VP, _VP, _I]),
    "mcd_share_resident": (_I, [C.POINTER(_VP), _I]),
    "mcd_subinstance_sweep_multi": (_I, [C.POINTER(_VP), _I, _I64, _VP, _I64, _VP, _I64, _VP, _VP, _VP, _VP, _I,
                                         C.POINTER(McdStats)]),
    "mcd_loo_sweep_multi": (_I, [C.POINTER(_VP), _I, _VP, _I64, _I64, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _I,
                                 C.POINTER(McdStats)]),
    "mcd_null_assignments_multi": (_I, [C.POINTER(_VP), _I, _I64, C.c_uint64, _VP, _VP]),
    "mcd_lap_steps": (_I, [_VP, _VP, _I64, _VP, _I64, _I64, _I64, _VP, _VP, _VP, _I, C.POINTER(McdStats)]),
    "mcd_cell2cell_gather": (
        _I,
        [_VP, _VP, _I64, _VP, _VP, _I64, _VP, _I64, _I64, _I64, _I, _I, _VP, _VP, _VP, _VP, _I, C.POINTER(McdStats)],
    ),
    "mcd_cell2cell_multi": (
        _I,
        [C.POINTER(_VP), _I, _VP, _I64, _VP, _VP, _I64, _VP, _I64, _I64, _I64, _I, _VP, _VP, _VP, C.POINTER(McdStats)],
    ),
    "mcd_cell2cell": (
        _I,
        [_VP, _VP, _I64, _VP, _I64, _I64, _I64, _I64, _I, _I, _VP, _VP, _VP, _VP, _I, C.POINTER(McdStats)],
    ),
}

_lib = None


def load_library():
    """dlopen the in-tree library and bind every declared symbol.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libmacrodna_b200.so is not built (%s). Run `python -m macrodna_b200.build`; "
            "there is no CPU fallback." % LIB_PATH
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    if lib.mcd_abi_version() != 2:
        raise RuntimeError("libmacrodna_b200.so ABI version mismatch")
    _lib = lib
    return lib


class McdError(RuntimeError):
    def __init__(self, status, detail):
        super().__init__("macrodna_b200 status %d: %s" % (status, detail))
        self.status = status


def _ptr(x):
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        return x.ctypes.data
    return int(x)


def _matrix(x, rows, ld, name):
    """A host operand of the C ABI: C-contiguous float64 [rows, ld].  Anything else (float32, a Fortran-ordered or
    transposed view such as ``df.to_numpy().T``, a wrong shape) would be silently reinterpreted by the pointer
    hand-off, so it is converted (dtype / layout) or rejected (shape) here.  Device pointers pass through."""
    if not isinstance(x, np.ndarray):
        return x
    if x.ndim != 2 or x.shape[0] != rows or x.shape[1] != ld:
        raise ValueError("macrodna_b200: %s must have shape (%d, %d), got %r" % (name, rows, ld, x.shape))
    return np.ascontiguousarray(x, dtype=np.float64)


def _out(x, n, dtype, name):
    """A caller-provided host output vector: must already be a writable C-contiguous array of the right type."""
    if isinstance(x, np.ndarray):
        if x.dtype != dtype or not x.flags.c_contiguous or not x.flags.writeable or x.size < n:
            raise ValueError("macrodna_b200: %s must be a writable C-contiguous %s array of at least %d elements" % (
                name, np.dtype(dtype).name, n))
    return x


def cell2cell_multi(handles, rna, dna, M, N, G, ld_rna=None, ld_dna=None, precision="ozaki", rna_gene_idx=None,
                    dna_gene_idx=None):
    """The hot path on several GPUs of one node from one process (``mcd_cell2cell_multi``): RNA rows sharded over
    ``handles`` (one per device), step loop on ``handles[0]``, where the correlation matrix stays resident."""
    h0 = handles[0]
    for h in handles:
        h.resident_token = None
    nsteps = h0.lib.mcd_num_steps(M, N)
    rna = _matrix(rna, M, ld_rna or G, "rna")
    dna = _matrix(dna, N, ld_dna or G, "dna")
    if not isinstance(rna, np.ndarray) or not isinstance(dna, np.ndarray):
        raise ValueError("macrodna_b200: the multi-GPU driver takes host arrays")
    assign = np.empty(M, dtype=np.int32)
    step = np.empty(M, dtype=np.int32)
    step_obj = np.empty(nsteps, dtype=np.float64)
    if rna_gene_idx is not None:
        rna_gene_idx = np.ascontiguousarray(rna_gene_idx, dtype=np.int32)
    if dna_gene_idx is not None:
        dna_gene_idx = np.ascontiguousarray(dna_gene_idx, dtype=np.int32)
    stats = McdStats()
    arr = (C.c_void_p * len(handles))(*[h.h for h in handles])
    st = h0.lib.mcd_cell2cell_multi(arr, len(handles), _ptr(rna), ld_rna or G, _ptr(rna_gene_idx), _ptr(dna), ld_dna or G,
                                    _ptr(dna_gene_idx), M, N, G, PREC[precision], _ptr(assign), _ptr(step), _ptr(step_obj),
                                    C.byref(stats))
    h0.check(st)
    return assign, step, step_obj, stats


def _handle_array(handles):
    """The ``mcd_handle*`` of a multi-handle call.  An empty list, or one context listed twice (two host threads would
    drive it at once), is refused here, before any GPU call."""
    handles = list(handles)
    if not handles:
        raise ValueError("macrodna_b200: at least one handle is required")
    if len({id(h) for h in handles}) != len(handles):
        raise ValueError("macrodna_b200: a handle is listed twice (list a device twice to get separate contexts on it)")
    return handles, (C.c_void_p * len(handles))(*[h.h for h in handles])


def share_resident(handles):
    """Copy the correlation matrix resident on ``handles[0]`` to every other handle (``mcd_share_resident``): the
    copies let the ``*_multi`` view calls deal their work over all of them.  A copy is valid until the next run on
    ``handles[0]``; a copy carries no assignment (``last_match_values`` refuses it)."""
    handles, arr = _handle_array(handles)
    for h in handles[1:]:
        h.resident_token = None
    handles[0].check(handles[0].lib.mcd_share_resident(arr, len(handles)))
    for h in handles[1:]:
        h.resident_token = handles[0].resident_token  # the same run's matrix


def subinstance_sweep_multi(handles, dna_cols, rna_rows=None, M=None, concurrency=8):
    """:meth:`Handle.subinstance_sweep` with the replicates dealt over ``handles`` (``mcd_subinstance_sweep_multi``;
    ``handles[1:]`` hold copies of ``handles[0]``'s matrix, see :func:`share_resident`)."""
    handles, arr = _handle_array(handles)
    h0 = handles[0]
    return h0._subinstance_sweep(lambda *a: h0.lib.mcd_subinstance_sweep_multi(arr, len(handles), *a), dna_cols,
                                 rna_rows, M, concurrency)


def loo_sweep_multi(handles, cells, k_steps, M, N, full=False, concurrency=8):
    """:meth:`Handle.loo_sweep` with the replicates dealt over ``handles`` (``mcd_loo_sweep_multi``)."""
    handles, arr = _handle_array(handles)
    h0 = handles[0]
    return h0._loo_sweep(lambda *a: h0.lib.mcd_loo_sweep_multi(arr, len(handles), *a), cells, k_steps, M, N, full,
                         concurrency)


def null_assignments_multi(handles, trials, seed=2023, medians=False):
    """:meth:`Handle.null_assignments` with the trials split over ``handles`` (``mcd_null_assignments_multi``): bit
    for bit what ``handles[0]`` alone returns."""
    handles, arr = _handle_array(handles)
    h0 = handles[0]
    sums = np.empty(int(trials), dtype=np.float64)
    med = np.empty(int(trials), dtype=np.float64) if medians else None
    h0.check(h0.lib.mcd_null_assignments_multi(arr, len(handles), int(trials), int(seed), _ptr(sums), _ptr(med)))
    return (sums, med) if medians else sums


class Handle:
    """One CUDA device + stream + workspace.  Created lazily so objects holding it stay picklable."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        st = self.lib.mcd_create(C.byref(h), int(device))
        if st != MCD_OK:
            raise McdError(
                st,
                "mcd_create(device=%d) failed: %s -- a B200 (sm_100a) GPU is required, there is no CPU fallback"
                % (device, self.lib.mcd_strerror(st).decode()),
            )
        self.h = h
        self.device = device
        self.pid = os.getpid()  # a CUDA context does not survive fork(): api.get_handle checks this
        self.resident_token = None  # identifies the run whose correlation matrix is resident (api.MaCroDNA)

    def close(self):
        if getattr(self, "h", None):
            if getattr(self, "pid", None) == os.getpid():  # in a forked child the context is not ours to destroy
                self.lib.mcd_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, st):
        if st != MCD_OK:
            detail = self.lib.mcd_last_error(self.h).decode()
            if st == MCD_ERR_NONFINITE or st == MCD_ERR_INVALID:
                raise ValueError("macrodna_b200: " + detail)
            raise McdError(st, detail)

    def set_option(self, name, value):
        """Tuning / behaviour switch of this handle (``mcd_set_option``; names in include/macrodna_b200.h)."""
        self.check(self.lib.mcd_set_option(self.h, name.encode(), float(value)))

    def get_option(self, name):
        v = C.c_double()
        self.check(self.lib.mcd_get_option(self.h, name.encode(), C.byref(v)))
        return v.value

    def ozaki_format(self, M, N, G):
        """(nsl, radix_bits, exact) of ``mcd_ozaki_format``: the digit format this handle uses for M x N x G, and
        whether its int32 accumulation is exact there (False: the drivers take the FP64 pipe)."""
        nsl, rb = C.c_int(), C.c_int()
        exact = self.lib.mcd_ozaki_format(self.h, M, N, G, C.byref(nsl), C.byref(rb))
        return nsl.value, rb.value, exact == 1

    @property
    def sm_count(self):
        return self.lib.mcd_device_sm_count(self.h)

    def synchronize(self):
        self.check(self.lib.mcd_synchronize(self.h))

    # ---- whole path, host or device buffers -------------------------------------------------
    def cell2cell(self, rna, dna, M, N, G, ld_rna=None, ld_dna=None, in_space=MEM_HOST, precision="ozaki",
                  assign=None, step=None, step_obj=None, corr_out=None, out_space=MEM_HOST, rna_gene_idx=None,
                  dna_gene_idx=None):
        """``rna``/``dna``: numpy arrays (host) or integer device pointers; cells x genes float64.
        ``rna_gene_idx`` / ``dna_gene_idx``: optional int32 arrays [G] -- column of each shared gene in the
        operand's block (the gene intersection is then gathered on the device)."""
        self.resident_token = None  # whoever relied on the previous resident correlation matrix must recompute
        nsteps = self.lib.mcd_num_steps(M, N)
        if in_space == MEM_HOST:
            rna = _matrix(rna, M, ld_rna or G, "rna")
            dna = _matrix(dna, N, ld_dna or G, "dna")
        if out_space == MEM_HOST:
            assign = _out(assign, M, np.int32, "assign")
            step = _out(step, M, np.int32, "step")
            step_obj = _out(step_obj, nsteps, np.float64, "step_obj")
            corr_out = _out(corr_out, M * N, np.float64, "corr_out")
        if assign is None:
            assign = np.empty(M, dtype=np.int32)
        if step is None:
            step = np.empty(M, dtype=np.int32)
        if step_obj is None:
            step_obj = np.empty(nsteps, dtype=np.float64)
        stats = McdStats()
        if rna_gene_idx is not None:
            rna_gene_idx = np.ascontiguousarray(rna_gene_idx, dtype=np.int32)
        if dna_gene_idx is not None:
            dna_gene_idx = np.ascontiguousarray(dna_gene_idx, dtype=np.int32)
        st = self.lib.mcd_cell2cell_gather(
            self.h, _ptr(rna), ld_rna or G, _ptr(rna_gene_idx), _ptr(dna), ld_dna or G, _ptr(dna_gene_idx), M, N, G,
            in_space, PREC[precision], _ptr(assign), _ptr(step), _ptr(step_obj), _ptr(corr_out), out_space,
            C.byref(stats),
        )
        self.check(st)
        return assign, step, step_obj, stats

    def last_match_values(self, M):
        """corr[i, assign[i]] of the last cell2cell call (matrix still resident on the device)."""
        out = np.empty(M, dtype=np.float64)
        self.check(self.lib.mcd_last_match_values(self.h, _ptr(out), M, MEM_HOST))
        return out

    # ---- views of the correlation matrix the last cell2cell call left resident ----------------------
    def subinstance(self, rna_rows=None, dna_cols=None, M=None, N=None):
        """Step loop on C[rna_rows][:, dna_cols] (None = all).  Returns (assign, step, objs, stats); ``assign``
        holds POSITIONS in ``dna_cols``."""
        if rna_rows is not None:
            rna_rows = np.ascontiguousarray(rna_rows, dtype=np.int32)
            m = rna_rows.size
        else:
            m = int(M)
        if dna_cols is not None:
            dna_cols = np.ascontiguousarray(dna_cols, dtype=np.int32)
            n = dna_cols.size
        else:
            n = int(N)
        nsteps = self.lib.mcd_num_steps(m, n)
        assign = np.empty(m, dtype=np.int32)
        step = np.empty(m, dtype=np.int32)
        objs = np.empty(nsteps, dtype=np.float64)
        stats = McdStats()
        self.check(self.lib.mcd_subinstance_steps(self.h, _ptr(rna_rows), m, _ptr(dna_cols), n, _ptr(assign), _ptr(step),
                                                  _ptr(objs), MEM_HOST, C.byref(stats)))
        return assign, step, objs, stats

    def subinstance_sweep(self, dna_cols, rna_rows=None, M=None, concurrency=8):
        """``len(dna_cols)`` replicates of :meth:`subinstance` kept ``concurrency`` at a time in flight
        (``mcd_subinstance_sweep``).  ``dna_cols``: int array [nrep, n_sub] of columns of the resident matrix
        (repeats allowed).  Returns (assign [nrep, m], step [nrep, m], objs [nrep, nsteps], cert_gap [nrep], stats)."""
        return self._subinstance_sweep(lambda *a: self.lib.mcd_subinstance_sweep(self.h, *a), dna_cols, rna_rows, M,
                                       concurrency)

    def _subinstance_sweep(self, call, dna_cols, rna_rows, M, concurrency):
        dna_cols = np.ascontiguousarray(dna_cols, dtype=np.int32)
        if dna_cols.ndim != 2:
            raise ValueError("dna_cols must be a 2-D array [replicates, DNA cells per replicate]")
        nrep, n = dna_cols.shape
        if rna_rows is not None:
            rna_rows = np.ascontiguousarray(rna_rows, dtype=np.int32)
            m = rna_rows.size
        else:
            m = int(M)
        nsteps = self.lib.mcd_num_steps(m, n)
        assign = np.empty((nrep, m), dtype=np.int32)
        step = np.empty((nrep, m), dtype=np.int32)
        objs = np.empty((nrep, nsteps), dtype=np.float64)
        gaps = np.empty(nrep, dtype=np.float64)
        stats = McdStats()
        self.check(call(nrep, _ptr(rna_rows), m, _ptr(dna_cols), n, _ptr(assign), _ptr(step), _ptr(objs), _ptr(gaps),
                        int(concurrency), C.byref(stats)))
        return assign, step, objs, gaps, stats

    def loo_sweep(self, cells, k_steps, M, N, full=False, concurrency=8):
        """Leave-one-out replicates of the resident M x N matrix, one per entry of ``cells`` (``mcd_loo_sweep``).
        Returns (dict of arrays, stats): ``test_col`` [ncells] (-1: no eligible column), ``test_corr``, ``total``,
        ``cert_gap``; with ``full`` also ``assign`` / ``step`` / ``match_corr`` [ncells, M-1] and ``step_obj``
        [ncells, nsteps]."""
        return self._loo_sweep(lambda *a: self.lib.mcd_loo_sweep(self.h, *a), cells, k_steps, M, N, full, concurrency)

    def _loo_sweep(self, call, cells, k_steps, M, N, full, concurrency):
        cells = np.ascontiguousarray(cells, dtype=np.int32).ravel()
        n, m = cells.size, int(M) - 1
        nsteps = self.lib.mcd_num_steps(m, int(N))
        out = {"test_col": np.empty(n, dtype=np.int32), "test_corr": np.empty(n, dtype=np.float64),
               "total": np.empty(n, dtype=np.float64), "cert_gap": np.empty(n, dtype=np.float64)}
        if full:
            out.update(assign=np.empty((n, m), dtype=np.int32), step=np.empty((n, m), dtype=np.int32),
                       step_obj=np.empty((n, nsteps), dtype=np.float64), match_corr=np.empty((n, m), dtype=np.float64))
        stats = McdStats()
        self.check(call(_ptr(cells), n, int(k_steps), _ptr(out["test_col"]), _ptr(out["test_corr"]), _ptr(out["total"]),
                        _ptr(out.get("assign")), _ptr(out.get("step")), _ptr(out.get("step_obj")),
                        _ptr(out.get("match_corr")), _ptr(out["cert_gap"]), int(concurrency), C.byref(stats)))
        return out, stats

    def corr_rows(self, rows, N):
        rows = np.ascontiguousarray(rows, dtype=np.int32)
        out = np.empty((rows.size, int(N)), dtype=np.float64)
        self.check(self.lib.mcd_corr_rows(self.h, _ptr(rows), rows.size, _ptr(out), MEM_HOST))
        return out

    def corr_pairs(self, rows, cols):
        rows = np.ascontiguousarray(rows, dtype=np.int32)
        cols = np.ascontiguousarray(cols, dtype=np.int32)
        out = np.empty(rows.size, dtype=np.float64)
        self.check(self.lib.mcd_corr_pairs(self.h, _ptr(rows), _ptr(cols), rows.size, _ptr(out)))
        return out

    def null_assignments(self, trials, seed=2023, medians=False):
        sums = np.empty(int(trials), dtype=np.float64)
        med = np.empty(int(trials), dtype=np.float64) if medians else None
        self.check(self.lib.mcd_null_assignments(self.h, int(trials), int(seed), _ptr(sums), _ptr(med), MEM_HOST))
        return (sums, med) if medians else sums

    def lap_steps(self, C_ptr, ldc, Ct_ptr, ldct, M, N, out_space=MEM_HOST, assign=None, step=None, step_obj=None):
        self.resident_token = None
        nsteps = self.lib.mcd_num_steps(M, N)
        if assign is None:
            assign = np.empty(M, dtype=np.int32)
        if step is None:
            step = np.empty(M, dtype=np.int32)
        if step_obj is None:
            step_obj = np.empty(nsteps, dtype=np.float64)
        stats = McdStats()
        st = self.lib.mcd_lap_steps(self.h, _ptr(C_ptr), ldc, _ptr(Ct_ptr), ldct, M, N, _ptr(assign), _ptr(step),
                                    _ptr(step_obj), out_space, C.byref(stats))
        self.check(st)
        return assign, step, step_obj, stats
