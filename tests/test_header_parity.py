"""Source-level API parity, function by function (SURVEY 8b tier 1).

tests/test_dropin_drivers.py shows that the reference's drivers build unchanged against include/*.h and print the
known-answer sizes on book1.  This goes below that: a C++ harness runs one test body against our headers and requires
every produced stream, every `RansEncSymbol` / `Rans64EncSymbol` / `RansDecSymbol` field (over the whole parameter range
the reference allows), every table row and every decoder state and cursor to be identical to what the same body
recorded against the reference's own headers (digests in tests/golden/reference_vectors.json), for the scalar, the
reciprocal and the SSE4.1 code paths.  The alias harness does the same for include/rans_alias.h; only the check that
runs our step functions on the driver's own SymbolStats includes main_alias.cpp (in place, nothing is copied), so that
one needs the reference checkout.
"""
import json
import os
import shutil
import subprocess

import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.join(ROOT, "tests", "header_parity")
REF = oracle.REFERENCE
VECTORS = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_vectors.json")))
WANT, WANT_ALIAS = VECTORS["header_parity"], VECTORS["alias_parity"]


@pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")
@pytest.mark.parametrize("opt", ["-O0", "-O3"])
def test_every_api_function_matches_the_reference(tmp_path, opt):
    exe = tmp_path / "harness"
    subprocess.check_call(["g++", opt, "-std=c++17", "-msse4.1", "-I" + os.path.join(ROOT, "include"), "-I" + HERE, "-o", str(exe),
                           os.path.join(HERE, "harness.cpp")])
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:]
    assert len(WANT) == 9 and out.stdout.strip().splitlines() == WANT, out.stdout


@pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")
@pytest.mark.parametrize("opt", ["-O0", "-O3"])
def test_rans_alias_header_matches_the_reference_driver(tmp_path, opt):
    """include/rans_alias.h (SURVEY section 7 step 2): the alias tables, RansEncPutAlias and RansDecGetAlias against the
    reference's own code in main_alias.cpp -- tables, encoder states, streams, decoder states and cursors identical at
    scale_bits 8 / 11 / 14 / 16, on the models the reference built (digests and frequencies in reference_vectors.json)."""
    exe = tmp_path / "harness_alias"
    subprocess.check_call(["g++", opt, "-std=c++17", "-w", "-I" + os.path.join(ROOT, "include"), "-o", str(exe),
                           os.path.join(HERE, "harness_alias.cpp")])
    freqs = "\n".join(" ".join(map(str, f)) for f in WANT_ALIAS["freqs"]) + "\n"
    out = subprocess.run([str(exe)], input=freqs, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:]
    assert len(WANT_ALIAS["lines"]) == 16 and out.stdout.strip().splitlines() == WANT_ALIAS["lines"], out.stdout


@pytest.mark.skipif(not os.path.exists(os.path.join(REF, "main_alias.cpp")) or shutil.which("g++") is None,
                    reason="needs the reference's main_alias.cpp and g++")
@pytest.mark.parametrize("opt", ["-O0", "-O3"])
def test_rans_alias_steps_on_the_driver_struct(tmp_path, opt):
    """The part that needs the reference's source: the harness built against main_alias.cpp (included in place) drives
    our RansEncPutAlias / RansDecGetAlias on the driver's own SymbolStats as well as on RansAliasTables, requires both to
    match the driver's functions step by step, and prints the models and digests stored in reference_vectors.json."""
    src = open(os.path.join(HERE, "harness_alias.cpp")).read().replace("REFDIR", REF)
    (tmp_path / "harness_alias.cpp").write_text(src)
    exe = tmp_path / "harness_alias"
    subprocess.check_call(["g++", opt, "-std=c++17", "-w", "-DRANS_REF_DRIVER", "-I" + os.path.join(ROOT, "include"), "-o", str(exe),
                           str(tmp_path / "harness_alias.cpp")], cwd=REF)
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600, cwd=REF)
    assert out.returncode == 0, out.stdout[-3000:]
    lines = out.stdout.strip().splitlines()
    assert [ln for ln in lines if not ln.startswith("freqs ")] == WANT_ALIAS["lines"]
    assert [[int(x) for x in ln.split(":", 1)[1].split()] for ln in lines if ln.startswith("freqs ")] == WANT_ALIAS["freqs"]


def test_rans_alias_header_compiles_for_the_device(tmp_path):
    """The same header under nvcc: RansEncPutAlias / RansDecGetAlias are __host__ __device__ (compile-only, sm_100a)."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    (tmp_path / "k.cu").write_text('''
#include "rans_alias.h"
__global__ void k(RansAliasTables* t, uint8_t* buf, uint32_t* out)
{
    RansState x;
    RansEncInit(&x);
    uint8_t* p = buf + 64;
    RansEncPutAlias(&x, &p, t, 3, 16);
    RansEncFlush(&x, &p);
    RansDecInit(&x, &p);
    out[0] = RansDecGetAlias(&x, t, 16);
}
''')
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-I" + os.path.join(ROOT, "include"), "-c",
                           "-o", str(tmp_path / "k.o"), str(tmp_path / "k.cu")])
