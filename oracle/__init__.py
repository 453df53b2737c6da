"""ctypes bindings for the parity oracle.  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this package.  Nothing under ryg_rans_b200/ does.

Two libraries:
  * liboracle.so        -- oracle/rans_oracle.c, the plain-C restatement (prefix orc_)
  * _ref/libryg_ref.so  -- the reference's own headers/drivers compiled from
                           /root/reference (prefix ref_); present only when built
                           in a container that has the reference checked out (the
                           built .so travels to the GPU box with the snapshot).
"""
import ctypes as C
import os
import subprocess
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_u8p = C.POINTER(C.c_uint8)
_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)

CODER_WORD, CODER_BYTE, CODER_ALIAS, CODER_RANS64 = 0, 1, 2, 3


def _reference_dir():
    """The reference checkout make builds _ref/ from: $REF, else the Makefile's `REF ?=` default."""
    if os.environ.get("REF"):
        return os.environ["REF"]
    with open(os.path.join(_HERE, "Makefile")) as f:
        for line in f:
            if line.startswith("REF ?="):
                return line.split("?=", 1)[1].strip()
    raise RuntimeError("oracle/Makefile defines no REF default")


REFERENCE = _reference_dir()


def build(force=False):
    """Compile liboracle.so (always) and _ref/ (only if the reference checkout REFERENCE is present)."""
    need = force or not os.path.exists(os.path.join(_HERE, "liboracle.so"))
    src = os.path.join(_HERE, "rans_oracle.c")
    lib = os.path.join(_HERE, "liboracle.so")
    if not need and os.path.getmtime(src) > os.path.getmtime(lib):
        need = True
    if need or (os.path.isdir(REFERENCE) and not os.path.exists(os.path.join(_HERE, "_ref", "libryg_ref.so"))):
        subprocess.check_call(["make", "-C", _HERE, "all"], stdout=subprocess.DEVNULL)


def _p(a, t):
    return a.ctypes.data_as(t)


def _u8(a):
    a = np.ascontiguousarray(a, dtype=np.uint8)
    return a


class _Lib:
    """Common surface of liboracle (orc_) and libryg_ref (ref_)."""

    def __init__(self, path, prefix):
        self.lib = C.CDLL(path)
        self.prefix = prefix
        self.path = path
        enc_sig = [_u8p, C.c_size_t, _u32p, _u32p, C.c_uint32, C.c_uint32, _u8p, C.c_size_t]
        dec_sig = [_u8p, C.c_size_t, _u32p, _u32p, C.c_uint32, C.c_uint32, _u8p, C.c_size_t]
        for name in ("byte", "alias", "rans64"):
            for kind, sig in (("encode", enc_sig), ("decode", dec_sig)):
                f = getattr(self.lib, f"{prefix}_{name}_{kind}")
                f.restype = C.c_long
                f.argtypes = sig
        f = getattr(self.lib, f"{prefix}_word_encode")
        f.restype = C.c_long
        f.argtypes = [_u8p, C.c_size_t, _u32p, _u32p, C.c_uint32, _u8p, C.c_size_t]
        f = getattr(self.lib, f"{prefix}_word_decode")
        f.restype = C.c_long
        f.argtypes = [_u8p, C.c_size_t, _u32p, _u32p, C.c_uint32, _u8p, C.c_size_t]
        f = getattr(self.lib, f"{prefix}_normalize_freqs")
        f.restype = C.c_int
        f.argtypes = [_u32p, _u32p, C.c_uint32]
        f = getattr(self.lib, f"{prefix}_count_freqs")
        f.restype = None
        f.argtypes = [_u8p, C.c_size_t, _u32p]
        f = getattr(self.lib, f"{prefix}_word_tables")
        f.restype = None
        f.argtypes = [_u32p, _u32p, _u32p, _u8p]

    # ---- model
    def count_freqs(self, data):
        data = _u8(data)
        freqs = np.zeros(256, np.uint32)
        getattr(self.lib, f"{self.prefix}_count_freqs")(_p(data, _u8p), data.size, _p(freqs, _u32p))
        return freqs

    def normalize_freqs(self, raw_freqs, target_total):
        freqs = np.array(raw_freqs, dtype=np.uint32).copy()
        cum = np.zeros(257, np.uint32)
        rc = getattr(self.lib, f"{self.prefix}_normalize_freqs")(_p(freqs, _u32p), _p(cum, _u32p), target_total)
        if rc != 0:
            raise ValueError(f"normalize_freqs failed rc={rc}")
        return freqs, cum

    def model(self, data, scale_bits):
        return self.normalize_freqs(self.count_freqs(data), 1 << scale_bits)

    def word_tables(self, freqs, cum):
        slots = np.zeros(4096, np.uint32)
        s2s = np.zeros(4096, np.uint8)
        getattr(self.lib, f"{self.prefix}_word_tables")(_p(freqs, _u32p), _p(cum, _u32p), _p(slots, _u32p), _p(s2s, _u8p))
        return slots, s2s

    # ---- N-way streams
    def encode(self, coder, data, freqs, cum, nlanes, scale_bits=12):
        data = _u8(data)
        cap = 2 * data.size + 8 * nlanes + 64
        out = np.zeros(cap, np.uint8)
        if coder == CODER_WORD:
            r = getattr(self.lib, f"{self.prefix}_word_encode")(_p(data, _u8p), data.size, _p(freqs, _u32p), _p(cum, _u32p),
                                                               nlanes, _p(out, _u8p), cap)
        else:
            name = {CODER_BYTE: "byte", CODER_ALIAS: "alias", CODER_RANS64: "rans64"}[coder]
            r = getattr(self.lib, f"{self.prefix}_{name}_encode")(_p(data, _u8p), data.size, _p(freqs, _u32p), _p(cum, _u32p),
                                                                 scale_bits, nlanes, _p(out, _u8p), cap)
        if r < 0:
            raise ValueError(f"encode failed rc={r}")
        return out[:r].copy()

    def decode(self, coder, stream, n, freqs, cum, nlanes, scale_bits=12):
        stream = _u8(stream)
        out = np.zeros(max(n, 1), np.uint8)
        if coder == CODER_WORD:
            r = getattr(self.lib, f"{self.prefix}_word_decode")(_p(stream, _u8p), stream.size, _p(freqs, _u32p), _p(cum, _u32p),
                                                               nlanes, _p(out, _u8p), n)
        else:
            name = {CODER_BYTE: "byte", CODER_ALIAS: "alias", CODER_RANS64: "rans64"}[coder]
            r = getattr(self.lib, f"{self.prefix}_{name}_decode")(_p(stream, _u8p), stream.size, _p(freqs, _u32p), _p(cum, _u32p),
                                                                 scale_bits, nlanes, _p(out, _u8p), n)
        if r < 0:
            raise ValueError(f"decode failed rc={r}")
        return out[:n].copy(), int(r)


class Oracle(_Lib):
    def __init__(self):
        build()
        super().__init__(os.path.join(_HERE, "liboracle.so"), "orc")
        L = self.lib
        L.orc_chunked_encode.restype = C.c_long
        L.orc_chunked_encode.argtypes = [C.c_int, _u8p, C.c_size_t, _u32p, _u32p, C.c_uint32, C.c_uint32, C.c_size_t,
                                         C.c_size_t, _u8p, C.c_size_t, _u64p]
        L.orc_chunked_decode.restype = C.c_long
        L.orc_chunked_decode.argtypes = [C.c_int, _u8p, C.c_size_t, _u64p, _u32p, _u32p, C.c_uint32, C.c_uint32,
                                         C.c_size_t, C.c_size_t, _u8p, C.c_size_t]
        L.orc_alias_build.restype = C.c_int
        L.orc_alias_build.argtypes = [_u32p, _u32p, C.c_void_p, _u32p]

    def alias_build(self, freqs, cum):
        raw = np.zeros(256 * 4 + 512 * 4 + 512 * 4 + 512, np.uint8)
        remap = np.zeros(int(cum[256]), np.uint32)
        rc = self.lib.orc_alias_build(_p(freqs, _u32p), _p(cum, _u32p), raw.ctypes.data, _p(remap, _u32p))
        if rc != 0:
            raise ValueError(f"alias_build rc={rc}")
        divider = raw[:1024].view(np.uint32).copy()
        slot_adjust = raw[1024:3072].view(np.uint32).copy()
        slot_freqs = raw[3072:5120].view(np.uint32).copy()
        sym_id = raw[5120:5632].copy()
        return divider, slot_adjust, slot_freqs, sym_id, remap

    def chunked_encode(self, coder, data, freqs, cum, chunk_syms, nlanes=32, scale_bits=12, align=16):
        data = _u8(data)
        n_chunks = (data.size + chunk_syms - 1) // chunk_syms
        cap = 2 * data.size + n_chunks * (8 * nlanes + 2 * align + 64) + 64
        blob = np.zeros(cap, np.uint8)
        offs = np.zeros(n_chunks + 1, np.uint64)
        r = self.lib.orc_chunked_encode(coder, _p(data, _u8p), data.size, _p(freqs, _u32p), _p(cum, _u32p), scale_bits,
                                        nlanes, chunk_syms, align, _p(blob, _u8p), cap, _p(offs, _u64p))
        if r < 0:
            raise ValueError(f"chunked_encode rc={r}")
        return blob[:r].copy(), offs

    def chunked_decode(self, coder, blob, offsets, n, freqs, cum, chunk_syms, nlanes=32, scale_bits=12, align=16):
        blob = _u8(blob)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        out = np.zeros(max(n, 1), np.uint8)
        r = self.lib.orc_chunked_decode(coder, _p(blob, _u8p), blob.size, _p(offsets, _u64p), _p(freqs, _u32p),
                                        _p(cum, _u32p), scale_bits, nlanes, chunk_syms, align, _p(out, _u8p), n)
        if r < 0:
            raise ValueError(f"chunked_decode rc={r}")
        return out[:n].copy()


class Reference(_Lib):
    """The reference's own code (oracle/_ref/libryg_ref.so)."""

    @staticmethod
    def available():
        build()
        return os.path.exists(os.path.join(_HERE, "_ref", "libryg_ref.so"))

    def __init__(self):
        build()
        super().__init__(os.path.join(_HERE, "_ref", "libryg_ref.so"), "ref")
        L = self.lib
        L.ref_word_decode_simd8.restype = C.c_long
        L.ref_word_decode_simd8.argtypes = [_u8p, C.c_size_t, _u32p, _u32p, _u8p, C.c_size_t]
        L.ref_alias_build.restype = C.c_int
        L.ref_alias_build.argtypes = [_u32p, _u32p, _u32p, _u32p, _u32p, _u8p, _u32p]
        dp = C.POINTER(C.c_double)
        L.ref_cpu_baseline_simd.restype = C.c_int
        L.ref_cpu_baseline_simd.argtypes = [_u8p, C.c_size_t, C.c_int, C.c_int, dp, dp, _u64p]
        for nm in ("ref_cpu_baseline_rans64", "ref_cpu_baseline_alias"):
            f = getattr(L, nm)
            f.restype = C.c_int
            f.argtypes = [_u8p, C.c_size_t, C.c_uint32, C.c_int, C.c_int, dp, dp, _u64p]

    def word_decode_simd8(self, stream, n, freqs, cum):
        stream = _u8(stream)
        out = np.zeros(max(n, 1), np.uint8)
        r = self.lib.ref_word_decode_simd8(_p(stream, _u8p), stream.size, _p(freqs, _u32p), _p(cum, _u32p), _p(out, _u8p), n)
        return out[:n].copy(), int(r)

    def alias_build(self, freqs, cum):
        divider = np.zeros(256, np.uint32)
        slot_adjust = np.zeros(512, np.uint32)
        slot_freqs = np.zeros(512, np.uint32)
        sym_id = np.zeros(512, np.uint8)
        remap = np.zeros(int(cum[256]), np.uint32)
        self.lib.ref_alias_build(_p(freqs, _u32p), _p(cum, _u32p), _p(divider, _u32p), _p(slot_adjust, _u32p),
                                 _p(slot_freqs, _u32p), _p(sym_id, _u8p), _p(remap, _u32p))
        return divider, slot_adjust, slot_freqs, sym_id, remap

    def cpu_baseline(self, which, data, nthreads, runs=3, scale_bits=None):
        """which in {'simd','rans64','alias'} -> dict(enc_s, dec_s, bytes, ok)"""
        data = _u8(data)
        e, d, b = C.c_double(), C.c_double(), C.c_uint64()
        if which == "simd":
            bad = self.lib.ref_cpu_baseline_simd(_p(data, _u8p), data.size, nthreads, runs, C.byref(e), C.byref(d), C.byref(b))
        elif which == "rans64":
            bad = self.lib.ref_cpu_baseline_rans64(_p(data, _u8p), data.size, scale_bits or 14, nthreads, runs,
                                                   C.byref(e), C.byref(d), C.byref(b))
        elif which == "alias":
            bad = self.lib.ref_cpu_baseline_alias(_p(data, _u8p), data.size, scale_bits or 16, nthreads, runs,
                                                  C.byref(e), C.byref(d), C.byref(b))
        else:
            raise ValueError(which)
        return {"enc_s": e.value, "dec_s": d.value, "bytes": int(b.value), "ok": bad == 0}
