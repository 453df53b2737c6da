"""BASELINE config 1 / SURVEY 8(b).1: the reference's drivers must build UNCHANGED against
this repo's source-level headers (include/rans_byte.h, rans64.h, rans_word_sse41.h,
platform.h) and print the reference's known-answer sizes and 'decode ok!'.

The drivers are copied to a temp dir at test time (a quoted #include looks beside the
including file first, so they cannot be compiled in place) -- nothing from the reference is
ever copied into the repo.  So that test needs the reference checkout (oracle.REFERENCE).
"""
import os
import re
import shutil
import subprocess

import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = oracle.REFERENCE

DRIVERS = [
    ("main.cpp", [], [435113, 435117]),                    # README:48,62
    ("main64.cpp", [], [435116, 435120]),                  # README:82,96
    ("main_simd.cpp", ["-msse4.1"], [435604, 435606, 435626]),   # README:110 for the 8-way stream
    ("main_alias.cpp", [], [435059, 435063]),
]


@pytest.mark.skipif(not os.path.exists(os.path.join(REF, "book1")), reason="needs the reference's driver sources")
@pytest.mark.parametrize("src,flags,sizes", DRIVERS)
def test_reference_driver_builds_unchanged_and_round_trips(tmp_path, src, flags, sizes):
    shutil.copy(os.path.join(REF, src), tmp_path / src)
    os.symlink(os.path.join(REF, "book1"), tmp_path / "book1")
    exe = tmp_path / "exam"
    subprocess.check_call(["g++", "-O3", "-w", *flags, "-I" + os.path.join(ROOT, "include"), "-o", str(exe), str(tmp_path / src),
                           "-lm", "-lrt"])
    # make sure it really used OUR headers
    deps = subprocess.run(["g++", "-MM", *flags, "-I" + os.path.join(ROOT, "include"), str(tmp_path / src)], capture_output=True,
                          text=True).stdout
    assert os.path.join(ROOT, "include") in deps and REF not in deps
    out = subprocess.run([str(exe)], cwd=tmp_path, capture_output=True, text=True, timeout=120).stdout
    assert "ERROR" not in out and out.count("decode ok!") == len(sizes), out[-400:]
    assert [int(x) for x in re.findall(r"rANS: (\d+) bytes", out)] == sizes


def test_headers_compile_for_device(tmp_path):
    """The same step functions are usable inside sm_100a kernels."""
    cu = tmp_path / "t.cu"
    cu.write_text('''
#include <assert.h>
#include "rans_byte.h"
#include "rans64.h"
#include "rans_word_sse41.h"
__global__ void k(uint8_t* b, uint32_t* w32, uint16_t* w16, RansWordTables* tab, RansEncSymbol* es, Rans64EncSymbol* e64)
{
    RansState r; RansEncInit(&r); uint8_t* p = b + 64; RansEncPutSymbol(&r, &p, es); RansEncFlush(&r, &p);
    RansDecInit(&r, &p); RansDecAdvance(&r, &p, 0, 1, 12); RansDecRenorm(&r, &p);
    Rans64State q; Rans64EncInit(&q); uint32_t* pw = w32 + 16; Rans64EncPutSymbol(&q, &pw, e64, 12); Rans64EncFlush(&q, &pw);
    Rans64DecInit(&q, &pw); Rans64DecAdvance(&q, &pw, 0, 1, 12);
    RansWordEnc e = RansWordEncInit(); uint16_t* ph = w16 + 32; RansWordEncPut(&e, &ph, 0, 1); RansWordEncFlush(&e, &ph);
    RansWordDec d; RansWordDecInit(&d, &ph); b[0] = RansWordDecSym(&d, tab); RansWordDecRenorm(&d, &ph);
}
''')
    subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-I" + os.path.join(ROOT, "include"), "-c",
                           "-o", str(tmp_path / "t.o"), str(cu)])
