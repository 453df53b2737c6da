import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _gen(kind, n, seed):
    """Seeded synthetic byte buffers in the shapes SURVEY 8(d) names."""
    rng = np.random.default_rng(seed)
    if kind == "uniform":
        return rng.integers(0, 256, n, dtype=np.uint8)
    if kind == "zipf":           # p(r) ~ (r+1)^-1.1 over 256 symbols, permuted
        p = 1.0 / np.arange(1, 257) ** 1.1
        p /= p.sum()
        perm = np.random.default_rng(1234).permutation(256)
        return perm[rng.choice(256, n, p=p)].astype(np.uint8)
    if kind == "text":           # order-0 text-like: 82 symbols, skewed
        syms = np.random.default_rng(99).permutation(256)[:82]
        p = np.random.default_rng(98).dirichlet(np.full(82, 0.35))
        return syms[rng.choice(82, n, p=p)].astype(np.uint8)
    if kind == "const":
        return np.full(n, 0x41, np.uint8)
    if kind == "two":            # two symbols, one very rare
        return np.where(rng.random(n) < 0.001, 7, 200).astype(np.uint8)
    if kind == "skew":           # one symbol with p > 0.5 (freq > 2048: exercises the wide reciprocal)
        return np.where(rng.random(n) < 0.7, 3, rng.integers(0, 256, n)).astype(np.uint8)
    raise ValueError(kind)


@pytest.fixture(scope="session")
def gen():
    return _gen


@pytest.fixture(scope="session")
def oracle_lib():
    import oracle
    return oracle.Oracle()


@pytest.fixture(scope="session")
def cuda_box():
    """For GPU tests that drive the library from a child process: skip (rather than fail) where there is no GPU."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


@pytest.fixture(scope="session")
def gpu_ctx():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ryg_rans_b200 as rb
    ctx = rb.Context(0)
    yield ctx
    ctx.close()
