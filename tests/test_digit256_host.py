"""CPU checks of the radix-256 digit format of the int8 correlation path: K1's fma / PRMT packing against a plain
digit decomposition (the device helpers are cut out of standardize.cu and compiled with g++), and the format choice
of mcd_ozaki_format (pure host entry point, no GPU)."""
import ctypes
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "macrodna_b200", "csrc")
HOST = os.path.join(ROOT, "tests", "host")


def _cut(path, start, end):
    src = open(path).read()
    a, b = src.index(start), src.index(end)
    assert a < b
    return src[a:b]


@pytest.mark.skipif(shutil.which("g++") is None, reason="g++ not available")
def test_k1_radix256_packing_matches_plain_digits(tmp_path):
    src = os.path.join(CSRC, "standardize.cu")
    snippet = (_cut(src, "__device__ __forceinline__ void ozaki_digits", "// Split-precision operand") +
               _cut(src, "template <int NSL>\n__device__ __forceinline__ void ozaki_bits", "// T threads per row, NV4 sweeps"))
    snip = tmp_path / "snippet.h"
    snip.write_text(snippet)
    exe = tmp_path / "check"
    subprocess.run(["g++", "-std=c++17", "-O2", "-DDIGIT_SNIPPET=\"%s\"" % snip, os.path.join(HOST, "digit256_check.cpp"),
                    "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "0 mismatches" in out.stdout


def _format(M, N, G):
    from macrodna_b200 import _lib

    lib = _lib.load_library()
    nsl, rb = ctypes.c_int(), ctypes.c_int()
    exact = lib.mcd_ozaki_format(None, M, N, G, ctypes.byref(nsl), ctypes.byref(rb))
    return nsl.value, 1 << rb.value, exact


def test_format_choice_without_handle():
    from macrodna_b200 import _lib

    lib = _lib.load_library()
    assert _format(50000, 10000, 20000) == (5, 256, 1)   # C5
    assert _format(50000, 10000, 32704) == (5, 256, 1)   # ldk8 = 32 704: the radix-256 int32 bound
    assert _format(50000, 10000, 32705) == (6, 128, 1)   # ldk8 = 32 768: 65 536 * ldk8 = 2^31
    assert _format(50000, 10000, 87360) == (6, 128, 1)   # radix 128 x 6 up to its own bound ...
    assert _format(50000, 10000, 87400)[2] == 0          # ... then the FP64 pipe
    assert _format(5000, 1000, 15000) == (8, 128, 1)     # C4: M N G <= 2e11
    assert _format(10000, 1000, 20000) == (8, 128, 1)    # exactly 2e11
    assert _format(40, 17, 90000) == (8, 128, 0)         # long rows below 2e11: FP64 pipe
    assert lib.mcd_ozaki_slices_for(50000, 10000, 20000) == 5
    assert lib.mcd_ozaki_slices_for(5000, 1000, 15000) == 8
    assert lib.mcd_ozaki_slices(None, 50000, 10000, 20000) == 5
