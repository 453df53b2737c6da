"""CPU tests that PIN the oracle (oracle/rans_oracle.c):
  * against the committed golden fixtures generated from the reference itself
    (tests/golden/make_golden.py -> oracle/_ref = reference headers + drivers compiled in place),
  * against what the reference computed for a grid of inputs, coders and lane counts
    (tests/golden/make_reference_vectors.py -> tests/golden/reference_vectors.json),
  * against the reference's published known-answer sizes for book1 (README:48,62,82,96,110)
    and the sizes the unmodified reference drivers print.
"""
import hashlib
import json
import os
import re
import subprocess

import numpy as np
import pytest

import oracle as orc

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = np.load(os.path.join(HERE, "golden", "golden.npz"))
INDEX = json.load(open(os.path.join(HERE, "golden", "golden.json")))
REFVEC = json.load(open(os.path.join(HERE, "golden", "reference_vectors.json")))
CODERS = {"word": (orc.CODER_WORD, 12), "byte": (orc.CODER_BYTE, 14), "alias": (orc.CODER_ALIAS, 16), "rans64": (orc.CODER_RANS64, 14)}
CASES = [k for k in INDEX if k != "book1"]
README_SIZES = {"byte/N1": 435113, "byte/N2": 435117, "rans64/N1": 435116, "rans64/N2": 435120, "word/N8": 435626}


def _sha(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def _book1(oracle_lib):
    """book1, decoded from the reference's own 32-way stream of it (test_book1_n32_golden_stream checks that stream)."""
    g = np.load(os.path.join(HERE, "golden", "book1_n32.npz"))
    freqs = g["freqs"]
    cum = np.concatenate([[0], np.cumsum(freqs)]).astype(np.uint32)
    return oracle_lib.decode(orc.CODER_WORD, g["stream"], int(g["n"]), freqs, cum, 32)[0]


@pytest.mark.parametrize("case", CASES)
def test_fixture_inputs_are_reproducible(case, gen):
    meta = INDEX[case]
    data = gen(meta["kind"], meta["n"], meta["seed"])
    assert _sha(data) == meta["sha256"]
    assert np.array_equal(data, GOLD[f"{case}/data"])


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("cname", sorted(CODERS))
def test_oracle_matches_reference_golden(oracle_lib, case, cname):
    cid, sb = CODERS[cname]
    data = GOLD[f"{case}/data"]
    freqs, cum = oracle_lib.model(data, sb)
    assert np.array_equal(freqs, GOLD[f"{case}/{cname}/freqs"]), "normalize_freqs differs from the reference"
    for key in INDEX[case]["streams"]:
        if not key.startswith(cname + "/"):
            continue
        nl = int(key.split("/N")[1])
        want = GOLD[f"{case}/{cname}/N{nl}"]
        got = oracle_lib.encode(cid, data, freqs, cum, nl, sb)
        assert np.array_equal(got, want), f"{case} {key}: oracle stream != reference stream"
        dec, used = oracle_lib.decode(cid, want, data.size, freqs, cum, nl, sb)
        assert np.array_equal(dec, data) and used == want.size


@pytest.mark.parametrize("case", CASES)
def test_oracle_alias_tables_golden(oracle_lib, case):
    data = GOLD[f"{case}/data"]
    freqs, cum = oracle_lib.model(data, 16)
    div, adj, sf, sid, remap = oracle_lib.alias_build(freqs, cum)
    assert np.array_equal(div, GOLD[f"{case}/alias_tables/divider"])
    assert np.array_equal(adj, GOLD[f"{case}/alias_tables/slot_adjust"])
    assert np.array_equal(sf, GOLD[f"{case}/alias_tables/slot_freqs"])
    assert np.array_equal(sid, GOLD[f"{case}/alias_tables/sym_id"])
    assert _sha(remap) == INDEX[case]["alias_remap_sha256"]


@pytest.mark.parametrize("kind", ["uniform", "zipf", "text", "two", "skew", "const"])
@pytest.mark.parametrize("n", [0, 1, 7, 64, 1000, 20011])
def test_oracle_vs_reference_live(oracle_lib, gen, kind, n):
    """The oracle's model and streams equal the reference's (recorded in reference_vectors.json: stream sizes and
    SHA-256), and the oracle's decoder consumes exactly what the reference's decoder consumed."""
    want = REFVEC["live"][f"{kind}/{n}"]
    data = gen(kind, max(n, 1), seed=n + 3)[:n] if n else np.zeros(0, np.uint8)
    assert _sha(data) == want["data_sha256"]
    model_src = data if n else gen(kind, 100, 1)
    for cname, (cid, sb) in CODERS.items():
        fo, co = oracle_lib.model(model_src, sb)
        assert _sha(fo, co) == want[cname]["model_sha256"]
        for nl in (1, 2, 3, 8, 32, 64):
            ref = want[cname][f"N{nl}"]
            so = oracle_lib.encode(cid, data, fo, co, nl, sb)
            assert so.size == ref["bytes"] and _sha(so) == ref["sha256"], (cname, nl)
            do, uo = oracle_lib.decode(cid, so, n, fo, co, nl, sb)
            assert np.array_equal(do, data) and uo == ref["used"] == so.size


def test_oracle_simd8_decoder_agrees(oracle_lib, gen):
    """The oracle's N=8 stream is the one the reference's own SSE4.1 2x4-lane decoder (main_simd.cpp:313-332) reads
    back to the input."""
    data = gen("text", 30007, 21)
    assert _sha(data) == REFVEC["simd8"]["data_sha256"]
    f, c = oracle_lib.model(data, 12)
    s = oracle_lib.encode(orc.CODER_WORD, data, f, c, 8)
    assert s.size == REFVEC["simd8"]["bytes"] and _sha(s) == REFVEC["simd8"]["sha256"]


def test_chunked_container_rules(oracle_lib, gen):
    data = gen("zipf", 50000, 8)
    f, c = oracle_lib.model(data, 12)
    blob, offs = oracle_lib.chunked_encode(orc.CODER_WORD, data, f, c, 4096)
    assert blob.size % 16 == 0 and offs[-1] == blob.size
    ends = offs[1:] & ~np.uint64(15)
    for i in range(len(offs) - 1):      # each chunk is exactly the plain N=32 stream, end-aligned
        s = oracle_lib.encode(orc.CODER_WORD, data[i * 4096:(i + 1) * 4096], f, c, 32)
        assert int(ends[i] - offs[i]) == s.size
        assert np.array_equal(blob[int(offs[i]):int(ends[i])], s)
        lo = int(ends[i - 1]) if i else 0
        assert not blob[lo:int(offs[i])].any()
    assert np.array_equal(oracle_lib.chunked_decode(orc.CODER_WORD, blob, offs, data.size, f, c, 4096), data)


def test_book1_n32_golden_stream(oracle_lib):
    """tests/golden/book1_n32.npz is the reference's own 32-way word-coder stream of book1 (435 702 bytes, SURVEY 8a;
    made by make_book1_stream.py).  The C restatement decodes it to bytes with book1's SHA-256 and re-encodes them to
    the identical stream -- the same known answer the GPU test checks through the C-ABI."""
    import hashlib
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "book1_n32.npz"))
    stream, freqs, n = g["stream"], g["freqs"], int(g["n"])
    assert stream.size == 435702 and n == 768771
    cum = np.concatenate([[0], np.cumsum(freqs)]).astype(np.uint32)
    book, used = oracle_lib.decode(orc.CODER_WORD, stream, n, freqs, cum, 32)
    assert used == stream.size
    assert hashlib.sha256(book.tobytes()).hexdigest() == "9ffa47cd93bccd732f20e0c304203cfbc1b8a91bedac536e2d8f6051003d9951"
    f2, c2 = oracle_lib.model(book, 12)
    assert np.array_equal(f2, freqs) and np.array_equal(c2, cum)
    assert np.array_equal(oracle_lib.encode(orc.CODER_WORD, book, freqs, cum, 32), stream)


# ---------------------------------------------------------------- book1, the reference's test file

def test_book1_known_answers(oracle_lib):
    book = _book1(oracle_lib)
    assert _sha(book) == INDEX["book1"]["sha256"] == "9ffa47cd93bccd732f20e0c304203cfbc1b8a91bedac536e2d8f6051003d9951"
    for key, meta in INDEX["book1"]["streams"].items():
        cname, nl = key.split("/N")
        cid, sb = CODERS[cname]
        f, c = oracle_lib.model(book, sb)
        s = oracle_lib.encode(cid, book, f, c, int(nl), sb)
        assert s.size == meta["bytes"] and _sha(s) == meta["sha256"], key
        if key in README_SIZES:
            assert s.size == README_SIZES[key]


@pytest.mark.parametrize("exe,sizes", [("exam", [435113, 435117]), ("exam64", [435116, 435120]),
                                       ("exam_simd_sse41", [435604, 435606, 435626]), ("exam_alias", [435059, 435063])])
def test_unmodified_reference_drivers(oracle_lib, tmp_path, exe, sizes):
    """The four reference drivers, built untouched by oracle/Makefile, print the known sizes and 'decode ok!' for book1.
    Where oracle/_ref was built they run here, on book1 rebuilt from the stored stream; their printed output is also
    stored (reference_vectors.json, whose agreement with `sizes` only checks that fixture).  Either way the oracle's
    book1 streams for the same coders and lane counts must have exactly those sizes."""
    printed = REFVEC["drivers"][exe]
    assert printed["sizes"] == sizes and printed["decode_ok"] == len(sizes)
    book = _book1(oracle_lib)
    path = os.path.join(os.path.dirname(orc.__file__), "_ref", exe)
    if os.path.exists(path):
        book.tofile(tmp_path / "book1")
        out = subprocess.run([path], cwd=tmp_path, capture_output=True, text=True, timeout=120).stdout
        assert "ERROR" not in out and out.count("decode ok!") == len(sizes)
        assert [int(x) for x in re.findall(r"rANS: (\d+) bytes", out)] == sizes
    coder, lanes = {"exam": ("byte", (1, 2)), "exam64": ("rans64", (1, 2)), "exam_simd_sse41": ("word", (1, 2, 8)),
                    "exam_alias": ("alias", (1, 2))}[exe]
    cid, sb = CODERS[coder]
    f, c = oracle_lib.model(book, sb)
    assert [oracle_lib.encode(cid, book, f, c, nl, sb).size for nl in lanes] == sizes
