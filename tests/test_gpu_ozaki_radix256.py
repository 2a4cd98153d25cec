"""GPU tests of the radix-256 digit format of the int8 tcgen05 correlation path: 5 balanced radix-256 slices
(15 products per output, ~5e-12 absolute), the format mcd_ozaki_format picks for large instances.  The handle option
"ozaki.radix" = 256 forces it at small shapes."""
import contextlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _torch():
    import torch

    assert torch.cuda.is_available()
    return torch


@contextlib.contextmanager
def _radix(handle, radix):
    handle.set_option("ozaki.radix", radix)
    try:
        yield
    finally:
        handle.set_option("ozaki.radix", 0)


def _digits256(handle, x_dev, ncells, G, ldx, nsl=5):
    torch = _torch()
    lib, h = handle.lib, handle.h
    ldk = lib.mcd_padded_k_split(G)
    a8 = torch.full((nsl, ncells, ldk), 55, dtype=torch.int8, device="cuda")
    sa = torch.empty(ncells, dtype=torch.float64, device="cuda")
    na = torch.empty(ncells, dtype=torch.float64, device="cuda")
    handle.check(lib.mcd_standardize_ozaki_radix(h, x_dev.data_ptr(), ncells, G, ldx, a8.data_ptr(), nsl, 8,
                                                 sa.data_ptr(), na.data_ptr()))
    handle.synchronize()
    return a8.cpu().numpy(), sa.cpu().numpy(), na.cpu().numpy()


def _value(a8, nsl=5):
    q = np.zeros(a8.shape[1:], dtype=np.float64)  # |q| <= 2^38: exact in float64
    for t in range(nsl):
        q = q * 256.0 + a8[t].astype(np.float64)
    return q


@pytest.mark.parametrize("generic", [0, 1])
@pytest.mark.parametrize("G", [5, 130, 256, 1000, 3000, 4097, 8192, 9001, 13000, 16385, 20000, 24576, 30000])
def test_radix256_digits_reconstruct_unit_rows(handle, G, generic):
    """Every K1 launch shape (fast path and, with k1.generic, the generic kernels; G = 30 000 is the long-row kernel),
    from aligned and from strided / misaligned input: digits reconstruct the unit rows to 2^-39 x the row scale,
    padding and zero-variance rows are zero, the leading digit lies in [-64, 64]."""
    from oracle import restatement as R

    torch = _torch()
    rng = np.random.default_rng(G + 7)
    ncells = 9
    x = np.log1p(rng.poisson(3.0, size=(ncells, G)).astype(np.float64)) + rng.random((ncells, G)) * 1e-3
    x[2] = np.log1p(2.0)
    x[5] = 1.0 / 3.0
    xc, nrm = R.standardise(x)
    flat = np.array([2, 5])
    nrm[flat] = 0.0
    xc[flat] = 0.0
    unit = np.divide(xc, nrm[:, None], out=np.zeros_like(xc), where=nrm[:, None] > 0)
    handle.set_option("k1.generic", generic)
    try:
        for ldx, off in ((G, 0), (G + 3, 1)):
            buf = torch.zeros(ncells * ldx + 8, dtype=torch.float64, device="cuda")
            view = buf[off:off + ncells * ldx].view(ncells, ldx)
            view[:, :G] = torch.from_numpy(x).cuda()
            a8, sa, na = _digits256(handle, view, ncells, G, ldx)
            assert np.abs(a8[0].astype(int)).max() <= 64
            rec = _value(a8)[:, :G] * 2.0 ** -39 * sa[:, None]
            assert np.abs(rec - unit).max() <= max(2.0 ** -39 * sa.max(), 1e-15), (G, ldx)
            assert (a8[:, :, G:] == 0).all()
            assert (a8[:, flat, :] == 0).all()
            assert np.abs(na - nrm).max() <= 1e-12 * nrm.max()
            live = nrm > 0
            top = np.abs(_value(a8)[live]).max(axis=1) * 2.0 ** -39
            assert (top >= 0.25 - 1e-9).all() and (top <= 0.5).all()
    finally:
        handle.set_option("k1.generic", 0)


@pytest.mark.parametrize("shape", [(4, 4, 6), (128, 256, 64), (130, 257, 100), (300, 200, 1000), (515, 700, 4099),
                                   (1000, 249, 20000)])
def test_corr_ozaki_radix256_kernel(handle, shape):
    from oracle import restatement as R

    torch = _torch()
    lib, h = handle.lib, handle.h
    M, N, G = shape
    rng = np.random.default_rng(M + 3 * N)
    rna = np.log1p(rng.poisson(4.0, size=(M, G)).astype(np.float64))
    dna = np.log1p(rng.integers(1, 5, size=(N, G)) * (1 + 0.05 * rng.standard_normal((N, G))))
    if N > 2:
        dna[1] = 2.0
    ref = R.correlation_matrix(rna, dna)
    a8, sa, na = _digits256(handle, torch.from_numpy(rna).cuda(), M, G, G)
    b8, sb, nb = _digits256(handle, torch.from_numpy(dna).cuda(), N, G, G)
    ldk = lib.mcd_padded_k_split(G)
    ldc, ldct = N + 2, M + 2
    c = torch.full((M, ldc), 7.0, dtype=torch.float64, device="cuda")
    ct = torch.full((N, ldct), 7.0, dtype=torch.float64, device="cuda")
    dev = [torch.from_numpy(v).cuda() for v in (a8, b8, sa, sb, na, nb)]
    handle.check(lib.mcd_corr_ozaki_radix(h, dev[0].data_ptr(), M, dev[1].data_ptr(), N, G, ldk, 5, 8, dev[2].data_ptr(),
                                          dev[3].data_ptr(), dev[4].data_ptr(), dev[5].data_ptr(), c.data_ptr(), ldc,
                                          ct.data_ptr(), ldct))
    handle.synchronize()
    c, ct = c.cpu().numpy(), ct.cpu().numpy()
    err = np.abs(c[:, :N] - ref).max()
    print("ozaki int8 radix-256 x5 max |dcorr| for", shape, "=", err)
    assert err < 1e-10
    assert (c[:, N:] == 7.0).all() and (ct[:, M:] == 7.0).all()
    assert (ct[:, :M] == c[:, :N].T).all()
    if N > 2:
        assert (c[:, 1] == 0).all()


def test_corr_ozaki_radix256_int32_bound(handle):
    """Hand-made digits at the bound: slice 0 = -64 and slices 1-4 = -128 in both operands make every term of the
    group g = 4 positive, 65 536 per gene; at ldk8 = 32 704 the accumulators stay exact and the result equals the
    value computed with Python integers.  At ldk8 = 32 768 the kernel refuses."""
    from macrodna_b200 import _lib

    torch = _torch()
    lib, h = handle.lib, handle.h
    M = N = 4
    digit = [-64, -128, -128, -128, -128]
    for ldk8, ok in ((32704, True), (32768, False)):
        a8 = torch.empty((5, M, ldk8), dtype=torch.int8, device="cuda")
        for t in range(5):
            a8[t].fill_(digit[t])
        b8 = a8.clone()
        ones = torch.ones(M, dtype=torch.float64, device="cuda")
        c = torch.zeros((M, N), dtype=torch.float64, device="cuda")
        st = lib.mcd_corr_ozaki_radix(h, a8.data_ptr(), M, b8.data_ptr(), N, ldk8, ldk8, 5, 8, ones.data_ptr(),
                                      ones.data_ptr(), ones.data_ptr(), ones.data_ptr(), c.data_ptr(), N, None, 0)
        if not ok:
            assert st == _lib.MCD_ERR_UNSUPPORTED
            continue
        handle.check(st)
        handle.synchronize()
        acc = [ldk8 * sum(digit[t] * digit[g - t] for t in range(g + 1)) for g in range(5)]
        assert acc[4] == 65536 * ldk8 and acc[4] < 2 ** 31
        exact = sum(acc[g] * 2 ** (8 * (4 - g)) for g in range(5))  # every group sum fits 37 bits: exact in float64
        v = float(exact) / 2.0 ** 32
        assert v * 2.0 ** 32 == exact
        nn = 1.0
        expect = v * (1.0 * 1.0 * 2.0 ** -14) * (nn / (1e-10 + nn))
        assert (c.cpu().numpy() == expect).all()


@pytest.mark.parametrize("name", ["C2", "C3", "C4"])
def test_whole_path_radix256(handle, name):
    from conftest import tie_report
    from macrodna_b200 import synth
    from oracle import restatement as R

    inst = synth.make_config_arrays(name)
    M, G = inst.rna.shape
    N = inst.dna.shape[0]
    corr = np.empty((M, N))
    with _radix(handle, 256):
        assert handle.ozaki_format(M, N, G) == (5, 8, True)
        assign, step, objs, stats = handle.cell2cell(inst.rna, inst.dna, M, N, G, precision="ozaki", corr_out=corr)
    c_ref, a_ref, s_ref, o_ref = R.cell2cell_arrays(inst.rna, inst.dna)
    err = np.abs(corr - c_ref).max()
    print(name, "ozaki radix-256 x5: max |dcorr| %.3g" % err)
    assert err <= 1e-10
    ident, rep = tie_report(c_ref, assign, step, a_ref, s_ref, rel=1e-9)
    assert ident, rep
    assert np.abs(objs - o_ref).max() <= 1e-9 * np.abs(o_ref).max()


def test_format_options_on_a_handle(handle):
    assert handle.ozaki_format(50000, 10000, 20000) == (5, 8, True)
    handle.set_option("ozaki.slices", 6)
    try:
        assert handle.ozaki_format(50000, 10000, 20000) == (6, 7, True)
        assert handle.lib.mcd_ozaki_slices(handle.h, 50000, 10000, 20000) == 6
    finally:
        handle.set_option("ozaki.slices", 0)
    with _radix(handle, 128):
        assert handle.ozaki_format(50000, 10000, 20000) == (6, 7, True)
        assert handle.ozaki_format(300, 70, 500) == (8, 7, True)
    with _radix(handle, 256):
        assert handle.ozaki_format(300, 70, 500) == (5, 8, True)
        assert handle.ozaki_format(300, 70, 40000) == (5, 8, False)


def test_multi_device_radix256_equals_single_device(handle):
    from macrodna_b200 import _lib, synth
    from macrodna_b200.api import get_handles

    inst = synth.make_arrays(1001, 140, 700, 4, seed=23)
    M, G = inst.rna.shape
    N = inst.dna.shape[0]
    hs = get_handles([0, 0])
    assert hs[0] is handle
    with _radix(handle, 256):
        a1, s1, o1, _ = handle.cell2cell(inst.rna, inst.dna, M, N, G, precision="ozaki")
        a2, s2, o2, _ = _lib.cell2cell_multi(hs, inst.rna, inst.dna, M, N, G, precision="ozaki")
    assert (a1 == a2).all() and (s1 == s2).all() and (o1 == o2).all()


def test_sharded_ranks_reproduce_single_gpu_rows(handle):
    """ShardedCell2Cell's per-rank K1 + K2 (the two ranks of a world of 2, run one after the other on this device)
    reproduce the single-GPU correlation rows bit for bit in the radix-256 format."""
    torch = _torch()
    from macrodna_b200 import dist, synth

    inst = synth.make_arrays(1001, 300, 3000, 4, seed=5)
    M, G = inst.rna.shape
    N = inst.dna.shape[0]
    corr = np.empty((M, N))
    with _radix(handle, 256):
        handle.cell2cell(inst.rna, inst.dna, M, N, G, precision="ozaki", corr_out=corr)
        dna = torch.from_numpy(inst.dna).cuda()
        for rank in range(2):
            sh = dist.ShardedCell2Cell(handle, M, N, G, world=2, rank=rank, device=torch.device("cuda", 0))
            assert (sh.nsl, sh.rb, sh.precision) == (5, 8, "ozaki")
            b = sh._alloc()
            ext = torch.cuda.ExternalStream(handle.lib.mcd_stream(handle.h), device=sh.device)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            rna_loc = torch.from_numpy(np.ascontiguousarray(inst.rna[sh.lo:sh.hi])).cuda()
            torch.cuda.synchronize()
            sh._standardize_and_correlate(b, rna_loc, dna, sh.hi - sh.lo, ev, ext)
            handle.synchronize()
            rows = b["c_loc"][: sh.hi - sh.lo, :N].cpu().numpy()
            assert (rows == corr[sh.lo:sh.hi]).all(), rank
