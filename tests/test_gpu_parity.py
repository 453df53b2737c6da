"""GPU parity: the C-ABI (include/rans_b200.h) against the oracle, bit-exact.

Mirrors the reference's own verification (decode-output memcmp, main_simd.cpp:340-343)
and strengthens it: the GPU blob must equal the oracle's container byte for byte, the
GPU must decode the oracle's blob, and the oracle must decode the GPU's blob.
"""
import hashlib
import json
import os

import numpy as np
import pytest

import oracle as orc

pytestmark = pytest.mark.gpu

# the reference's own N = 32 streams of the inputs below (tests/golden/make_reference_vectors.py)
REF_N32 = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_vectors.json")))["n32"]

WORD, BYTE, ALIAS, RANS64 = 0, 1, 2, 3


def _model(oracle_lib, data, scale_bits):
    return oracle_lib.model(data, scale_bits)


def _sha(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def _reference_stream_n32(gpu_ctx, oracle_lib, data, coder, ocoder, sb, want):
    """One chunk of the GPU container is the reference's N = 32 stream: same model, same bytes (size and SHA-256 of
    the reference's stream), and it decodes in exactly the bytes the reference's decoder consumed."""
    assert _sha(data) == want["data_sha256"]
    freqs, cum = oracle_lib.model(data, sb)
    assert _sha(freqs, cum) == want["model_sha256"]
    model = gpu_ctx.model(coder, sb, freqs)
    blob, offs = gpu_ctx.encode_host(model, data, 1 << 16)
    stream = blob[int(offs[0]):]
    assert stream.size == want["bytes"] and _sha(stream) == want["sha256"]
    dec, used = oracle_lib.decode(ocoder, stream, data.size, freqs, cum, 32, sb)
    assert np.array_equal(dec, data) and used == want["used"] == stream.size
    model.close()


def _roundtrip(gpu_ctx, oracle_lib, data, coder, scale_bits, chunk):
    import ryg_rans_b200 as rb
    freqs, cum = _model(oracle_lib, data, scale_bits)
    model = gpu_ctx.model(coder, scale_bits, freqs)
    blob, offs = gpu_ctx.encode_host(model, data, chunk)
    oblob, ooffs = oracle_lib.chunked_encode(coder, data, freqs, cum, chunk, nlanes=32, scale_bits=scale_bits)
    assert np.array_equal(offs, ooffs), "directory differs from the oracle container"
    assert blob.size == oblob.size
    assert np.array_equal(blob, oblob), "GPU stream is not byte-identical to the reference-order stream"
    # GPU decodes the oracle's blob; oracle decodes the GPU's blob
    dec = gpu_ctx.decode_host(model, oblob, ooffs, data.size, chunk)
    assert np.array_equal(dec, data)
    dec2 = oracle_lib.chunked_decode(coder, blob, offs, data.size, freqs, cum, chunk, nlanes=32, scale_bits=scale_bits)
    assert np.array_equal(dec2, data)
    model.close()


@pytest.mark.parametrize("kind", ["uniform", "zipf", "text", "two", "skew", "const"])
@pytest.mark.parametrize("n,chunk", [(1, 32), (31, 32), (32, 32), (33, 64), (4096, 4096), (100003, 4096), (300000, 16384)])
def test_word_parity(gpu_ctx, oracle_lib, gen, kind, n, chunk):
    data = gen(kind, n, seed=n * 7 + len(kind))
    _roundtrip(gpu_ctx, oracle_lib, data, WORD, 12, chunk)


def test_word_empty(gpu_ctx, oracle_lib, gen):
    freqs, cum = _model(oracle_lib, gen("uniform", 1000, 1), 12)
    model = gpu_ctx.model(WORD, 12, freqs)
    blob, offs = gpu_ctx.encode_host(model, np.zeros(0, np.uint8), 4096)
    assert blob.size == 0 and offs.tolist() == [0]
    out = gpu_ctx.decode_host(model, blob, offs, 0, 4096)
    assert out.size == 0


def test_word_reference_stream_n32(gpu_ctx, oracle_lib, gen):
    """A single chunk IS the reference's N-way stream with N = 32 (SURVEY 8a layout)."""
    _reference_stream_n32(gpu_ctx, oracle_lib, gen("text", 50000, 5), WORD, orc.CODER_WORD, 12, REF_N32["word"])


def test_book1_known_answer_through_the_gpu(gpu_ctx, oracle_lib):
    """The reference-held known answer, through the GPU (SURVEY 8a): the reference's own 32-way word-coder stream of
    book1 is 435 702 bytes (tests/golden/book1_n32.npz, made by make_book1_stream.py from the reference's primitives).
    The GPU decodes it -- the bytes must hash to book1's SHA-256 -- and re-encoding them as ONE chunk must reproduce
    the stream byte for byte; the oracle agrees on both."""
    import hashlib
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "book1_n32.npz"))
    stream, freqs, n = g["stream"], g["freqs"], int(g["n"])
    assert stream.size == 435702 and n == 768771
    chunk = 1 << 20                                   # one chunk >= n: the container is exactly one reference stream
    gap = (-stream.size) % 16                         # streams are END-aligned to 16 bytes inside a blob
    blob = np.concatenate([np.zeros(gap, np.uint8), stream])
    offs = np.array([gap, blob.size], np.uint64)
    model = gpu_ctx.model(WORD, 12, freqs)
    book = gpu_ctx.decode_host(model, blob, offs, n, chunk)
    assert hashlib.sha256(book.tobytes()).digest() == g["book_sha256"].tobytes()          # "decode ok!"
    assert hashlib.sha256(book.tobytes()).hexdigest() == "9ffa47cd93bccd732f20e0c304203cfbc1b8a91bedac536e2d8f6051003d9951"
    f2, cum = oracle_lib.model(book, 12)
    assert np.array_equal(f2, freqs)                                                     # normalize_freqs(4096) of book1
    gblob, goffs = gpu_ctx.encode_host(model, book, chunk)
    assert gblob.size - int(goffs[0]) == 435702
    assert np.array_equal(gblob[int(goffs[0]):], stream)
    assert np.array_equal(oracle_lib.encode(orc.CODER_WORD, book, freqs, cum, 32), stream)
    model.close()


def test_word_corrupt_stream_is_reported(gpu_ctx, oracle_lib, gen):
    import ryg_rans_b200 as rb
    data = gen("zipf", 20000, 3)
    freqs, cum = _model(oracle_lib, data, 12)
    model = gpu_ctx.model(WORD, 12, freqs)
    blob, offs = gpu_ctx.encode_host(model, data, 4096)
    bad = blob.copy()
    bad[int(offs[1]) + 128:int(offs[1]) + 400] ^= 0x5A
    with pytest.raises(rb.RansError) as ei:
        gpu_ctx.decode_host(model, bad, offs, data.size, 4096)
    assert ei.value.code == -4
    # truncated directory
    offs2 = offs.copy()
    offs2[2] = offs2[3] + 64
    with pytest.raises(rb.RansError):
        gpu_ctx.decode_host(model, blob, offs2, data.size, 4096)
    # context still healthy afterwards
    assert np.array_equal(gpu_ctx.decode_host(model, blob, offs, data.size, 4096), data)


def test_word_zero_freq_symbol_is_reported(gpu_ctx, oracle_lib, gen):
    import ryg_rans_b200 as rb
    data = gen("text", 10000, 2)
    freqs, cum = _model(oracle_lib, data, 12)
    model = gpu_ctx.model(WORD, 12, freqs)
    other = data.copy()
    missing = int(np.flatnonzero(freqs == 0)[0])
    other[1234] = missing
    with pytest.raises(rb.RansError) as ei:
        gpu_ctx.encode_host(model, other, 4096)
    assert ei.value.code == -7


def test_encode_bound_is_tight_enough(gpu_ctx, oracle_lib, gen):
    data = gen("uniform", 70000, 9)
    freqs, cum = _model(oracle_lib, data, 12)
    model = gpu_ctx.model(WORD, 12, freqs)
    blob, offs = gpu_ctx.encode_host(model, data, 4096)
    assert blob.size <= gpu_ctx.encode_bound(data.size, 4096)
    import ryg_rans_b200 as rb
    with pytest.raises(rb.RansError) as ei:
        gpu_ctx.encode_host(model, data, 4096, blob_cap=blob.size - 16)
    assert ei.value.code == -3


# ---------------------------------------------------------------- alias coder (BASELINE config 3)

@pytest.mark.parametrize("kind", ["zipf", "uniform", "text", "two", "const"])
@pytest.mark.parametrize("n,chunk,sb", [(1, 32, 16), (33, 64, 16), (4096, 4096, 16), (100003, 4096, 16), (300000, 16384, 16),
                                        (50001, 2048, 12), (50001, 2048, 8)])
def test_alias_parity(gpu_ctx, oracle_lib, gen, kind, n, chunk, sb):
    data = gen(kind, n, seed=n * 11 + len(kind))
    _roundtrip(gpu_ctx, oracle_lib, data, ALIAS, sb, chunk)


def test_alias_reference_stream_n32(gpu_ctx, oracle_lib, gen):
    _reference_stream_n32(gpu_ctx, oracle_lib, gen("zipf", 60000, 6), ALIAS, orc.CODER_ALIAS, 16, REF_N32["alias"])


def test_alias_corrupt_stream_is_reported(gpu_ctx, oracle_lib, gen):
    import ryg_rans_b200 as rb
    data = gen("zipf", 20000, 3)
    freqs, cum = _model(oracle_lib, data, 16)
    model = gpu_ctx.model(ALIAS, 16, freqs)
    blob, offs = gpu_ctx.encode_host(model, data, 4096)
    bad = blob.copy()
    bad[int(offs[2]) + 128:int(offs[2]) + 300] ^= 0xA5
    with pytest.raises(rb.RansError) as ei:
        gpu_ctx.decode_host(model, bad, offs, data.size, 4096)
    assert ei.value.code == -4


# ---------------------------------------------------------------- rans_byte cum2sym coder (main.cpp) and rans64 (main64.cpp)

@pytest.mark.parametrize("kind", ["zipf", "uniform", "text", "two", "const", "skew"])
@pytest.mark.parametrize("n,chunk,sb", [(1, 32, 14), (33, 64, 14), (4096, 4096, 14), (100003, 4096, 14), (300000, 16384, 14),
                                        (50001, 2048, 12), (50001, 2048, 8), (70001, 8192, 16)])
def test_byte_parity(gpu_ctx, oracle_lib, gen, kind, n, chunk, sb):
    if kind == "const" and sb == 16:
        pytest.skip("a frequency of 65536 does not fit the reference's 16-bit RansDecSymbol.freq")
    data = gen(kind, n, seed=n * 13 + len(kind))
    _roundtrip(gpu_ctx, oracle_lib, data, BYTE, sb, chunk)


def test_byte_rejects_16bit_overflow(gpu_ctx, gen):
    import ryg_rans_b200 as rb
    freqs = np.zeros(256, np.uint32)
    freqs[65] = 65536
    with pytest.raises(rb.RansError) as ei:
        gpu_ctx.model(BYTE, 16, freqs)
    assert ei.value.code == -2


@pytest.mark.parametrize("kind", ["zipf", "uniform", "text", "two", "const", "skew"])
@pytest.mark.parametrize("n,chunk,sb", [(1, 32, 14), (33, 64, 14), (4096, 4096, 14), (100003, 4096, 14), (300000, 16384, 14),
                                        (50001, 2048, 8), (70001, 8192, 16)])
def test_rans64_parity(gpu_ctx, oracle_lib, gen, kind, n, chunk, sb):
    data = gen(kind, n, seed=n * 17 + len(kind))
    _roundtrip(gpu_ctx, oracle_lib, data, RANS64, sb, chunk)


@pytest.mark.parametrize("coder,ocoder,sb", [(BYTE, orc.CODER_BYTE, 14), (RANS64, orc.CODER_RANS64, 14)])
def test_byte_and_rans64_reference_stream_n32(gpu_ctx, oracle_lib, gen, coder, ocoder, sb):
    """The reference's own RansEncPutSymbol / Rans64EncPutSymbol loops (N = 32) produce the GPU's chunk stream,
    and it decodes in exactly the bytes the reference's decoders consumed."""
    _reference_stream_n32(gpu_ctx, oracle_lib, gen("text", 60000, 8), coder, ocoder, sb,
                          REF_N32["byte" if coder == BYTE else "rans64"])


# ---------------------------------------------------------------- device histogram / per-block models (config 5)

@pytest.mark.parametrize("n", [0, 1, 15, 16, 17, 4097, 1 << 20, (1 << 22) + 5])
def test_histogram(gpu_ctx, gen, n):
    data = gen("zipf", n, 4) if n else np.zeros(0, np.uint8)
    counts = gpu_ctx.histogram(data)
    assert np.array_equal(counts, np.bincount(data, minlength=256).astype(np.uint64))


@pytest.mark.parametrize("coder,sb", [(WORD, 12), (BYTE, 14), (ALIAS, 16), (RANS64, 14)])
@pytest.mark.parametrize("kind,n", [("text", 300_001), ("two", 4097), ("uniform", 1 << 20)])
def test_model_from_data(gpu_ctx, oracle_lib, gen, coder, sb, kind, n):
    """rb200_model_from_data = device histogram + the reference's normalize_freqs + tables: the frequencies it
    reports are the oracle's, and a stream encoded with that model is the oracle's stream."""
    import ryg_rans_b200 as rb
    data = gen(kind, n, 21)
    freqs, cum = _model(oracle_lib, data, sb)
    model = rb.Model.from_data(gpu_ctx, coder, sb, data)
    assert np.array_equal(model.freqs, freqs)
    blob, offs = gpu_ctx.encode_host(model, data, 8192)
    ob, oo = oracle_lib.chunked_encode({WORD: orc.CODER_WORD, BYTE: orc.CODER_BYTE, ALIAS: orc.CODER_ALIAS,
                                        RANS64: orc.CODER_RANS64}[coder], data, freqs, cum, 8192, scale_bits=sb)
    assert np.array_equal(offs, oo) and np.array_equal(blob, ob)
    assert np.array_equal(gpu_ctx.decode_host(model, blob, offs, n, 8192), data)
    model.close()


def test_model_from_data_device_and_errors(gpu_ctx, oracle_lib, gen):
    import torch
    import ryg_rans_b200 as rb
    data = gen("zipf", 777_777, 22)
    d = torch.from_numpy(data).cuda()
    model = rb.Model.from_data(gpu_ctx, WORD, 12, device_ptr=d.data_ptr(), n=d.numel())
    assert np.array_equal(model.freqs, _model(oracle_lib, data, 12)[0])
    model.close()
    with pytest.raises(rb.RansError) as e:                         # empty input: nothing to normalise
        rb.Model.from_data(gpu_ctx, WORD, 12, np.zeros(0, np.uint8))
    assert e.value.code == -2
    with pytest.raises(rb.RansError) as e:                         # scale_bits below 8: 256 symbols cannot fit 2^7 slots
        rb.Model.from_data(gpu_ctx, BYTE, 7, gen("uniform", 4096, 1))
    assert e.value.code == -1


def _block_data(gen, n_blocks, block_size):
    kinds = ["zipf", "uniform", "text", "two", "skew", "const"]
    return np.concatenate([gen(kinds[b % len(kinds)], block_size, seed=1000 + b) for b in range(n_blocks)])


@pytest.mark.parametrize("n_blocks,block_size,chunk", [(13, 65536, 8192), (7, 4096, 4096), (6, 16384, 2048), (12, 65536, 65536),
                                                       (5, 65536, 2048),      # 32 chunks per block: the widest CTA (32 warps)
                                                       (5, 17 * 1024, 1024)])  # 17 chunks per block: rounds up to 32 warps

def test_block_models_and_roundtrip(gpu_ctx, oracle_lib, gen, n_blocks, block_size, chunk):
    _check_blocks(gpu_ctx, oracle_lib, _block_data(gen, n_blocks, block_size), n_blocks, block_size, chunk)


@pytest.mark.parametrize("path", ["fused", "split"])
def test_block_paths_and_host_pipeline(cuda_box, path):
    """Per-block encode: the one-launch persistent path (default) and the round-1 sequence (RB200_ENCODE_PATH=split)
    build the identical container; with 1 MiB slices the HOST-mode calls run their 3-stream pipeline over many slices of
    whole blocks (encode, model+encode and decode) and must still match the oracle block by block."""
    import os
    import subprocess
    import sys
    code = r'''
import sys, numpy as np
sys.path.insert(0, %r)
import oracle, ryg_rans_b200 as rb
rng = np.random.default_rng(21)
orc = oracle.Oracle()
ctx = rb.Context(0)
for n_blocks, block_size, chunk in ((200, 65536, 8192), (37, 16384, 4096), (64, 65536, 65536)):
    blocks = []
    for b in range(n_blocks):
        p = 1.0 / np.arange(1, 257) ** (0.6 + 0.1 * (b %% 9))
        blocks.append(rng.permutation(256).astype(np.uint8)[rng.choice(256, block_size, p=p / p.sum())])
    data = np.concatenate(blocks)
    blob, offs, freqs = ctx.blocks_model_encode_host(data, n_blocks, block_size, chunk)
    blob2, offs2 = ctx.blocks_encode_host(data, n_blocks, block_size, freqs, chunk)
    assert np.array_equal(offs, offs2) and np.array_equal(blob, blob2)
    per = block_size // chunk
    for b in range(0, n_blocks, max(1, n_blocks // 7)):
        f, c = orc.model(blocks[b], 12)
        assert np.array_equal(f.astype(np.uint16), freqs[b])
        ob, oo = orc.chunked_encode(oracle.CODER_WORD, blocks[b], f, c, chunk, scale_bits=12)
        lo, hi = int(offs[b * per]) & ~15, int(offs[(b + 1) * per]) & ~15
        assert np.array_equal(blob[lo:hi], ob), b
    assert np.array_equal(ctx.blocks_decode_host(blob, offs, freqs, n_blocks, block_size, chunk), data)
print("block paths ok", ctx.launches)
''' % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RB200_ENCODE_PATH=path, RB200_SLICE_MIB="1")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "block paths ok" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


def test_block_reciprocal_fallback(gpu_ctx, oracle_lib, gen):
    """Per-block encoders pick the 32-bit reciprocal when it is exact for the block's model; blocks whose model has
    a symbol of frequency 2964 or 3005 (the first that are not) must fall back, next to blocks that do not."""
    rng = np.random.default_rng(11)
    blocks = []
    for f0 in (2964, 16, 3005, 2963):
        b = np.concatenate([np.full(f0 * 16, 7, np.uint8), np.full((4096 - f0) * 16, 9, np.uint8)])
        rng.shuffle(b)
        blocks.append(b)
    blocks.append(gen("zipf", 65536, 5))
    data = np.concatenate(blocks)
    freqs16 = _check_blocks(gpu_ctx, oracle_lib, data, len(blocks), 65536, 8192)
    assert [int(freqs16[b][7]) for b in range(4)] == [2964, 16, 3005, 2963]


def _check_blocks(gpu_ctx, oracle_lib, data, n_blocks, block_size, chunk):
    freqs16 = gpu_ctx.blocks_build_models(data, n_blocks, block_size)
    # the one-launch form (model + encode fused, rb200_blocks_model_encode) must give the same models and container
    fblob, foffs, ffreqs = gpu_ctx.blocks_model_encode_host(data, n_blocks, block_size, chunk)
    assert np.array_equal(ffreqs, freqs16)
    want = np.stack([oracle_lib.model(data[b * block_size:(b + 1) * block_size], 12)[0] for b in range(n_blocks)])
    assert np.array_equal(freqs16.astype(np.uint32), want), "device normalize_freqs differs from the reference algorithm"

    blob, offs = gpu_ctx.blocks_encode_host(data, n_blocks, block_size, freqs16, chunk)
    assert np.array_equal(foffs, offs) and np.array_equal(fblob, blob), "fused model+encode container differs"
    # oracle: every block is its own container; containers concatenate because each ends 16-aligned
    parts, all_offs, base = [], [], 0
    for b in range(n_blocks):
        f = want[b]
        c = np.concatenate([[0], np.cumsum(f)]).astype(np.uint32)
        ob, oo = oracle_lib.chunked_encode(orc.CODER_WORD, data[b * block_size:(b + 1) * block_size], f, c, chunk)
        parts.append(ob)
        all_offs.append(oo[:-1] + base)
        base += ob.size
    oblob = np.concatenate(parts)
    ooffs = np.concatenate(all_offs + [[base]]).astype(np.uint64)
    assert np.array_equal(offs, ooffs)
    assert np.array_equal(blob, oblob)
    out = gpu_ctx.blocks_decode_host(oblob, ooffs, freqs16, n_blocks, block_size, chunk)
    assert np.array_equal(out, data)
    return freqs16


# ---------------------------------------------------------------- alternative paths, big sizes

@pytest.mark.parametrize("path", ["fused", "split"])
def test_forced_encode_paths(cuda_box, path):
    """Both word-encode paths (RB200_ENCODE_PATH=fused: persistent encode + scanner warp + deferred placement;
    =split: encode, tile scan, compaction) must produce the identical container at every chunk size."""
    import os
    import subprocess
    import sys
    code = r'''
import sys, numpy as np
sys.path.insert(0, %r)
import oracle, ryg_rans_b200 as rb
rng = np.random.default_rng(3)
p = 1.0 / np.arange(1, 257) ** 1.1
data = rng.choice(256, 3_000_017, p=p / p.sum()).astype(np.uint8)
orc = oracle.Oracle()
ctx = rb.Context(0)
for coder, sb in ((rb.CODER_WORD, 12), (rb.CODER_ALIAS, 16), (rb.CODER_BYTE, 14)):
    f, c = orc.model(data, sb)
    m = ctx.model(coder, sb, f)
    for chunk in (4096, 32, 65536):
        blob, offs = ctx.encode_host(m, data, chunk)
        ob, oo = orc.chunked_encode(coder, data, f, c, chunk, scale_bits=sb)
        assert np.array_equal(offs, oo) and np.array_equal(blob, ob), (coder, chunk)
        assert np.array_equal(ctx.decode_host(m, blob, offs, data.size, chunk), data)
    m.close()
print("fused ok", ctx.launches)
''' % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RB200_ENCODE_PATH=path)
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "fused ok" in out.stdout, out.stderr[-2000:]


@pytest.mark.parametrize("path", ["classic", "persistent"])
def test_forced_decode_paths(cuda_box, path):
    """Both word decoders (RB200_DECODE_PATH=classic: one CTA per 8 chunks, LDG -> STS window; default: persistent grid,
    TMA-staged table, cp.async ring, word_decode_tma.cuh) must decode oracle containers bit-exactly at every chunk size,
    ragged tails and the single-symbol (freq 4096) model included, report corruption, and stay usable afterwards (the
    persistent decoder's work counter re-arms itself)."""
    import os
    import subprocess
    import sys
    code = r'''
import sys, numpy as np
sys.path.insert(0, %r)
import oracle, ryg_rans_b200 as rb
rng = np.random.default_rng(11)
p = 1.0 / np.arange(1, 257) ** 1.1
orc = oracle.Oracle()
ctx = rb.Context(0)
for n in (1, 31, 32, 33, 4097, 1_000_003, 3_000_017):
    for kind in ("zipf", "uniform", "single"):
        if kind == "zipf": data = rng.choice(256, n, p=p / p.sum()).astype(np.uint8)
        elif kind == "uniform": data = rng.integers(0, 256, n, dtype=np.uint8)
        else: data = np.full(n, 65, np.uint8)
        f, c = orc.model(data, 12)
        m = ctx.model(rb.CODER_WORD, 12, f)
        for chunk in (32, 96, 4096, 8192, 65536):
            if n > 200_000 and chunk < 4096: continue
            ob, oo = orc.chunked_encode(oracle.CODER_WORD, data, f, c, chunk, scale_bits=12)
            for rep in range(2):                      # back to back: the chunk counter must have re-armed
                assert np.array_equal(ctx.decode_host(m, ob, oo, n, chunk), data), (n, kind, chunk, rep)
            if n >= 4097 and chunk == 4096:
                bad = ob.copy()
                bad[int(oo[0]) + 128:int(oo[0]) + 400] ^= 0x5a          # inside the first chunk's stream
                try:
                    ctx.decode_host(m, bad, oo, n, chunk)
                    raise SystemExit("corruption not reported")
                except rb.RansError as e:
                    assert e.code == -4, e
                assert np.array_equal(ctx.decode_host(m, ob, oo, n, chunk), data)
        m.close()
print("decode paths ok", ctx.launches)
''' % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RB200_DECODE_PATH=path)
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "decode paths ok" in out.stdout


def test_host_pipeline_many_slices(gpu_ctx, oracle_lib, gen):
    """Host-mode calls are a slice pipeline (32 MiB slices on three streams, ramped at both ends: 4, 8, 16,
    32, 32, 16, 8, 4 MiB here); cross several slice boundaries."""
    n = (32 << 20) * 4 + 12345
    data = gen("text", n, 77)
    freqs, cum = _model(oracle_lib, data, 12)
    model = gpu_ctx.model(WORD, 12, freqs)
    blob, offs = gpu_ctx.encode_host(model, data, 8192)
    assert blob.size % 16 == 0 and offs[-1] == blob.size
    # slices are independent containers that were concatenated: check a chunk on each side of a slice boundary
    for c in (0, 511, 512, 1535, 1536, 3583, 3584, 7679, 7680, 11775, 11776, 13823, 13824, len(offs) - 2):
        lo = c * 8192
        s = oracle_lib.encode(orc.CODER_WORD, data[lo:lo + 8192], freqs, cum, 32)
        end = int(offs[c + 1]) & ~15
        assert np.array_equal(blob[int(offs[c]):end], s), c
    out = gpu_ctx.decode_host(model, blob, offs, n, 8192)
    assert np.array_equal(out, data)
    model.close()


@pytest.mark.parametrize("f0", [1, 2963, 2964, 3005, 4095])
def test_word_reciprocal_variants(gpu_ctx, oracle_lib, f0):
    """The word encoder divides by a 32-bit reciprocal where that is exact on x < freq << 20 (every freq <= 2963 and
    most above; freq 1 through the x - 1 identity) and by the any-x 33-bit one otherwise (2964 and 3005 are the
    first frequencies that need it).  Hand-built models put one symbol on exactly that frequency."""
    rng = np.random.default_rng(f0)
    freqs = np.zeros(256, np.uint32)
    freqs[7] = f0
    rest = 4096 - f0
    freqs[200] = rest // 2
    freqs[13] = rest - rest // 2
    cum = np.concatenate([[0], np.cumsum(freqs)]).astype(np.uint32)
    p = freqs / 4096.0
    data = rng.choice(256, 300_011, p=p).astype(np.uint8)
    data[:2] = (7, 13)                       # both present even when rare
    model = gpu_ctx.model(WORD, 12, freqs)
    for chunk in (8192, 999):
        blob, offs = gpu_ctx.encode_host(model, data, chunk)
        ob, oo = oracle_lib.chunked_encode(orc.CODER_WORD, data, freqs, cum, chunk)
        assert np.array_equal(offs, oo) and np.array_equal(blob, ob), (f0, chunk)
        assert np.array_equal(gpu_ctx.decode_host(model, blob, offs, data.size, chunk), data)
    model.close()


def test_word_reciprocal_forced_33bit(cuda_box):
    """RB200_WORD_RECIPROCAL=33 forces the any-x reciprocal for every model; the container must not change."""
    import os
    import subprocess
    import sys
    code = r'''
import sys, numpy as np
sys.path.insert(0, %r)
import oracle, ryg_rans_b200 as rb
rng = np.random.default_rng(9)
orc = oracle.Oracle()
ctx = rb.Context(0)
for kind in range(3):
    if kind == 0:
        data = rng.integers(0, 256, 2_000_003, dtype=np.uint8)
    elif kind == 1:
        p = 1.0 / np.arange(1, 257) ** 1.1
        data = rng.choice(256, 2_000_003, p=p / p.sum()).astype(np.uint8)
    else:
        data = rng.choice(256, 2_000_003, p=[0.97] + [0.03 / 255] * 255).astype(np.uint8)
    f, c = orc.model(data, 12)
    m = ctx.model(rb.CODER_WORD, 12, f)
    for chunk in (8192, 2048):
        blob, offs = ctx.encode_host(m, data, chunk)
        ob, oo = orc.chunked_encode(rb.CODER_WORD, data, f, c, chunk, scale_bits=12)
        assert np.array_equal(offs, oo) and np.array_equal(blob, ob), (kind, chunk)
    m.close()
print("r33 ok")
''' % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RB200_WORD_RECIPROCAL="33")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "r33 ok" in out.stdout, out.stderr[-2000:]


def test_host_pipeline_ramped_slices(cuda_box):
    """The host pipeline ramps its first and last three slices (1/8, 1/4, 1/2 of RB200_SLICE_MIB).  With 1 MiB
    slices a 9 MB input takes the ramped plan; the container must not depend on the slicing: equal to the
    oracle's for every coder, also with tiny and ragged chunks and a non-pinned directory."""
    import os
    import subprocess
    import sys
    code = r'''
import sys, numpy as np
sys.path.insert(0, %r)
import oracle, ryg_rans_b200 as rb
rng = np.random.default_rng(5)
p = 1.0 / np.arange(1, 257) ** 1.1
data = rng.choice(256, 9_000_017, p=p / p.sum()).astype(np.uint8)
orc = oracle.Oracle()
ctx = rb.Context(0)
for coder, sb, chunks in ((rb.CODER_WORD, 12, (8192, 1000, 32)), (rb.CODER_ALIAS, 16, (8192,)), (rb.CODER_BYTE, 14, (4096,)),
                          (rb.CODER_RANS64, 14, (8192,))):
    f, c = orc.model(data, sb)
    m = ctx.model(coder, sb, f)
    for chunk in chunks:
        blob, offs = ctx.encode_host(m, data, chunk)
        ob, oo = orc.chunked_encode(coder, data, f, c, chunk, scale_bits=sb)
        assert np.array_equal(offs, oo) and np.array_equal(blob, ob), (coder, chunk)
        assert np.array_equal(ctx.decode_host(m, blob, offs, data.size, chunk), data)
    m.close()
print("ramped ok", ctx.launches)
''' % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RB200_SLICE_MIB="1")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ramped ok" in out.stdout, out.stderr[-2000:]
    # 9 MB / 1 MiB slices with ramps = 6 ramp + 7 steady slices per call; far more launches than one per call
    assert int(out.stdout.split()[-1]) > 100


@pytest.mark.parametrize("coder,sb,kind", [(WORD, 12, "uniform"), (ALIAS, 16, "zipf")])
def test_full_size_roundtrip_properties(gpu_ctx, coder, sb, kind):
    """BASELINE sizes (1 GiB per GPU), checked through size-independent properties: device round trip is the
    identity, the directory is monotone and 16-byte end-aligned, the blob size equals the directory's last
    entry, and decoding after corrupting one stream is reported."""
    import torch
    import ryg_rans_b200 as rb
    n, chunk = 1 << 30, 8192
    g = torch.Generator(device="cuda")
    g.manual_seed(1234)
    if kind == "uniform":
        data = torch.randint(0, 256, (n,), dtype=torch.uint8, device="cuda", generator=g)
    else:
        p = 1.0 / torch.arange(1, 257, dtype=torch.float64) ** 1.1
        cdf = torch.cumsum(p / p.sum(), 0).to(device="cuda", dtype=torch.float32)
        data = torch.empty(n, dtype=torch.uint8, device="cuda")
        for lo in range(0, n, 1 << 26):
            u = torch.rand(1 << 26, device="cuda", generator=g)
            data[lo:lo + (1 << 26)] = torch.searchsorted(cdf, u).clamp_(max=255).to(torch.uint8)
    counts = gpu_ctx.histogram_device(data.data_ptr(), n)
    assert int(counts.sum()) == n
    assert np.array_equal(counts, torch.bincount(data.view(torch.uint8).to(torch.int64), minlength=256).cpu().numpy().astype(np.uint64))
    st = rb.SymbolStats()
    st.freqs[:] = counts.astype(np.uint32)
    st.normalize_freqs(1 << sb)
    model = gpu_ctx.model(coder, sb, st.freqs)
    n_chunks = gpu_ctx.chunk_count(n, chunk)
    cap = gpu_ctx.encode_bound(n, chunk)
    blob = torch.empty(cap, dtype=torch.uint8, device="cuda")
    offsets = torch.zeros(n_chunks + 1, dtype=torch.int64, device="cuda")
    out = torch.zeros(n, dtype=torch.uint8, device="cuda")
    gpu_ctx.encode_device(model, data.data_ptr(), n, chunk, blob.data_ptr(), cap, offsets.data_ptr())
    gpu_ctx.sync()
    size = int(offsets[-1])
    assert size % 16 == 0 and 0 < size <= cap
    d = offsets[1:] - offsets[:-1]
    assert bool((d > 0).all())                                   # monotone
    ends = offsets[1:] & ~15
    sizes = ends - offsets[:-1]
    assert int(sizes.min()) >= 128 and int((ends[1:] - ends[:-1] - ((sizes[1:] + 15) & ~15)).abs().max()) == 0
    gpu_ctx.decode_device(model, blob.data_ptr(), size, offsets.data_ptr(), chunk, out.data_ptr(), n)
    gpu_ctx.sync()
    assert torch.equal(out, data)
    # a sample of the 131 072 chunk streams against the oracle, byte for byte: first, last, the chunks either side of
    # every 2^32-byte boundary the blob crosses (none at 1 GiB, but the indexing is 64-bit clean) and 64 random ones
    import oracle as orc_mod
    oracle_lib = orc_mod.Oracle()
    freqs = st.freqs.copy()
    cum = np.concatenate([[0], np.cumsum(freqs)]).astype(np.uint32)
    offs_h = offsets.cpu().numpy().astype(np.uint64)
    rng = np.random.default_rng(99)
    picks = sorted(set([0, 1, n_chunks // 2, n_chunks - 2, n_chunks - 1] + [int(c) for c in rng.integers(0, n_chunks, 64)]))
    ocoder = {WORD: orc_mod.CODER_WORD, ALIAS: orc_mod.CODER_ALIAS}[coder]
    for c in picks:
        lo, hi = c * chunk, min(n, (c + 1) * chunk)
        sym = data[lo:hi].cpu().numpy()
        want = oracle_lib.encode(ocoder, sym, freqs, cum, 32, sb)
        b0, b1 = int(offs_h[c]), int(offs_h[c + 1]) & ~15
        got = blob[b0:b1].cpu().numpy()
        assert got.size == want.size and np.array_equal(got, want), f"chunk {c}: GPU stream != oracle stream"
    # corrupt one stream in the middle of the blob
    mid = int(offsets[n_chunks // 2]) + 200
    blob[mid:mid + 64] ^= 0x3C
    gpu_ctx.decode_device(model, blob.data_ptr(), size, offsets.data_ptr(), chunk, out.data_ptr(), n)
    with pytest.raises(rb.RansError) as ei:
        gpu_ctx.sync()
    assert ei.value.code == -4
    model.close()
    del data, blob, out, offsets
    torch.cuda.empty_cache()


@pytest.mark.parametrize("coder,sb", [(WORD, 12), (BYTE, 14), (ALIAS, 16), (RANS64, 14)])
@pytest.mark.parametrize("chunk", [1000, 4104])
def test_unaligned_chunk_sizes(gpu_ctx, oracle_lib, gen, coder, sb, chunk):
    """chunk_syms that are not multiples of 16: chunk starts are unaligned, so the encoders' 128-bit staging
    falls back to byte loads and ragged tails appear in every chunk."""
    data = gen("zipf", 23456, seed=chunk)
    _roundtrip(gpu_ctx, oracle_lib, data, coder, sb, chunk)


def test_device_pointers_with_offset_views(gpu_ctx, oracle_lib, gen):
    """DEVICE mode on sub-buffers: input at an odd device address (unaligned staging path), outputs 16-byte aligned."""
    import torch
    data = gen("text", 70001, 31)
    freqs, cum = _model(oracle_lib, data, 12)
    model = gpu_ctx.model(WORD, 12, freqs)
    d_all = torch.zeros(data.size + 64, dtype=torch.uint8, device="cuda")
    d_in = d_all[3:3 + data.size]
    d_in.copy_(torch.from_numpy(data))
    n_chunks = gpu_ctx.chunk_count(data.size, 4096)
    cap = gpu_ctx.encode_bound(data.size, 4096)
    blob = torch.zeros(cap, dtype=torch.uint8, device="cuda")
    offs = torch.zeros(n_chunks + 1, dtype=torch.int64, device="cuda")
    out = torch.zeros(data.size + 7, dtype=torch.uint8, device="cuda")
    gpu_ctx.encode_device(model, d_in.data_ptr(), data.size, 4096, blob.data_ptr(), cap, offs.data_ptr())
    gpu_ctx.sync()
    size = int(offs[-1])
    oblob, ooffs = oracle_lib.chunked_encode(orc.CODER_WORD, data, freqs, cum, 4096)
    assert np.array_equal(blob[:size].cpu().numpy(), oblob) and np.array_equal(offs.cpu().numpy().astype(np.uint64), ooffs)
    gpu_ctx.decode_device(model, blob.data_ptr(), size, offs.data_ptr(), 4096, out[5:].data_ptr(), data.size)
    gpu_ctx.sync()
    assert np.array_equal(out[5:5 + data.size].cpu().numpy(), data)
    model.close()


@pytest.mark.parametrize("coder", ["word", "alias"])
def test_cpp_driver_exam_gpu(cuda_box, coder):
    """The reference-style C++ driver (csrc/exam_gpu.cpp) over the C-ABI: host code in C++, no Python in the path."""
    import os
    import subprocess
    import ryg_rans_b200 as rb
    exe = os.path.join(os.path.dirname(rb.LIB_PATH), "exam_gpu")
    if not os.path.exists(exe):
        rb.build()
    assert os.path.exists(exe)
    out = subprocess.run([exe, "-", coder, "8192", str(8 << 20)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    assert "decode ok!" in out.stdout and "ERROR" not in out.stdout
    assert "GPU rANS:" in out.stdout


def test_large_chunks_use_bounded_scratch(gpu_ctx, oracle_lib, gen):
    """chunk_syms above 64 Ki symbols must not blow up the encoder's scratch (two slots per resident warp in the
    fused path): such geometries take the split path, whose scratch is 2x the input."""
    data = gen("zipf", (1 << 20) + 77, 5)
    for coder, sb in ((WORD, 12), (ALIAS, 16)):
        _roundtrip(gpu_ctx, oracle_lib, data, coder, sb, 1 << 18)


def test_shards_concatenate_on_one_gpu(gpu_ctx, oracle_lib, gen):
    """SURVEY 8(e) degraded to one GPU: encode N shards one after the other (what N ranks would do), concatenate
    blobs and directories the way ryg_rans_b200.shard.gather_blobs does, and decode the whole thing in one call."""
    from ryg_rans_b200.shard import shard_bounds
    n, chunk, world = 1_000_003, 4096, 4
    data = gen("text", n, 41)
    freqs, cum = _model(oracle_lib, data, 12)
    model = gpu_ctx.model(WORD, 12, freqs)
    blobs, dirs, base = [], [], 0
    for r in range(world):
        lo, hi = shard_bounds(n, world, r, chunk)
        b, o = gpu_ctx.encode_host(model, data[lo:hi], chunk)
        assert b.size % 16 == 0
        blobs.append(b)
        dirs.append(o[:-1] + np.uint64(base))
        base += b.size
    blob = np.concatenate(blobs)
    offs = np.concatenate(dirs + [np.array([base], np.uint64)])
    whole, woffs = gpu_ctx.encode_host(model, data, chunk)
    assert np.array_equal(blob, whole) and np.array_equal(offs, woffs)
    assert np.array_equal(gpu_ctx.decode_host(model, blob, offs, n, chunk), data)
    model.close()
