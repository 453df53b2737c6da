#!/usr/bin/env python
"""Record what the reference itself computes for the tests that compare with it, so that they run without it.

Runs only where the reference checkout exists (oracle.REFERENCE: $REF, else oracle/Makefile's default) and oracle/_ref
is built from it.  Writes tests/golden/reference_vectors.json:

  live           for every input of test_oracle.py::test_oracle_vs_reference_live: the reference's model and, per
                 coder and lane count, its stream (size, SHA-256) and how many bytes its decoder consumed
  simd8          the N = 8 word stream the reference's SSE4.1 decoder reads back to its input
  n32            the reference's N = 32 streams the GPU chunk tests compare with (test_gpu_parity.py)
  drivers        the compressed sizes the four unmodified reference drivers print for book1
  header_parity  the digest lines of tests/header_parity/harness.cpp built against the reference's headers
  alias_parity   tests/header_parity/harness_alias.cpp built against the reference's main_alias.cpp: each model's
                 frequencies ("freqs") and the digest lines ("lines")

    python tests/golden/make_reference_vectors.py
"""
import hashlib
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import oracle  # noqa: E402
from conftest import _gen  # noqa: E402

REF = oracle.REFERENCE

CODERS = {"word": (oracle.CODER_WORD, 12), "byte": (oracle.CODER_BYTE, 14), "alias": (oracle.CODER_ALIAS, 16),
          "rans64": (oracle.CODER_RANS64, 14)}
LIVE_KINDS = ["uniform", "zipf", "text", "two", "skew", "const"]
LIVE_NS = [0, 1, 7, 64, 1000, 20011]
LIVE_LANES = (1, 2, 3, 8, 32, 64)
N32 = {"word": ("text", 50000, 5), "alias": ("zipf", 60000, 6), "byte": ("text", 60000, 8), "rans64": ("text", 60000, 8)}
DRIVERS = ["exam", "exam64", "exam_simd_sse41", "exam_alias"]


def sha(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def stream_entry(ref, cid, data, freqs, cum, nl, sb):
    s = ref.encode(cid, data, freqs, cum, nl, sb)
    dec, used = ref.decode(cid, s, data.size, freqs, cum, nl, sb)
    assert np.array_equal(dec, data) and used == s.size
    return {"bytes": int(s.size), "sha256": sha(s), "used": int(used)}


def main():
    ref = oracle.Reference()
    out = {"live": {}, "n32": {}, "drivers": {}}
    for kind in LIVE_KINDS:
        for n in LIVE_NS:
            data = _gen(kind, max(n, 1), seed=n + 3)[:n] if n else np.zeros(0, np.uint8)
            model_src = data if n else _gen(kind, 100, 1)
            case = {"data_sha256": sha(data)}
            for cname, (cid, sb) in CODERS.items():
                freqs, cum = ref.model(model_src, sb)
                case[cname] = {"model_sha256": sha(freqs, cum)}
                for nl in LIVE_LANES:
                    case[cname][f"N{nl}"] = stream_entry(ref, cid, data, freqs, cum, nl, sb)
            out["live"][f"{kind}/{n}"] = case

    data = _gen("text", 30007, 21)
    freqs, cum = ref.model(data, 12)
    s = ref.encode(oracle.CODER_WORD, data, freqs, cum, 8)
    dec, _ = ref.word_decode_simd8(s, data.size, freqs, cum)
    assert np.array_equal(dec, data)
    out["simd8"] = {"data_sha256": sha(data), "bytes": int(s.size), "sha256": sha(s)}

    for cname, (kind, n, seed) in N32.items():
        cid, sb = CODERS[cname]
        data = _gen(kind, n, seed)
        freqs, cum = ref.model(data, sb)
        out["n32"][cname] = {"data_sha256": sha(data), "model_sha256": sha(freqs, cum),
                             **stream_entry(ref, cid, data, freqs, cum, 32, sb)}

    for exe in DRIVERS:
        text = subprocess.run([os.path.join(ROOT, "oracle", "_ref", exe)], cwd=REF, capture_output=True, text=True,
                              timeout=120).stdout
        assert "ERROR" not in text
        out["drivers"][exe] = {"sizes": [int(x) for x in re.findall(r"rANS: (\d+) bytes", text)],
                               "decode_ok": text.count("decode ok!")}

    with tempfile.TemporaryDirectory() as tmp:
        src = open(os.path.join(HERE, "..", "header_parity", "harness.cpp")).read().replace("REFDIR", REF)
        with open(os.path.join(tmp, "harness.cpp"), "w") as f:
            f.write(src)
        exe = os.path.join(tmp, "harness")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-msse4.1", "-DRANS_REF_HEADERS",
                               "-I" + os.path.join(HERE, "..", "header_parity"), "-o", exe, os.path.join(tmp, "harness.cpp")])
        lines = subprocess.run([exe], capture_output=True, text=True, check=True, timeout=600).stdout.strip().splitlines()
        assert len(lines) == 9 and all("round trips 1" in ln for ln in lines), lines
        out["header_parity"] = lines

        src = open(os.path.join(HERE, "..", "header_parity", "harness_alias.cpp")).read().replace("REFDIR", REF)
        with open(os.path.join(tmp, "harness_alias.cpp"), "w") as f:
            f.write(src)
        exe = os.path.join(tmp, "harness_alias")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-w", "-DRANS_REF_DRIVER", "-I" + os.path.join(ROOT, "include"), "-o", exe,
                               os.path.join(tmp, "harness_alias.cpp")], cwd=REF)
        lines = subprocess.run([exe], capture_output=True, text=True, check=True, timeout=600, cwd=REF).stdout.strip().splitlines()
        freqs = [[int(x) for x in ln.split(":", 1)[1].split()] for ln in lines if ln.startswith("freqs ")]
        lines = [ln for ln in lines if not ln.startswith("freqs ")]
        assert len(freqs) == len(lines) == 16 and all("round trips 1" in ln for ln in lines), lines
        out["alias_parity"] = {"freqs": freqs, "lines": lines}

    path = os.path.join(HERE, "reference_vectors.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
        f.write("\n")
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
