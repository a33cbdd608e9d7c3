"""CPU checks of half-precision embedding input: argument validation of the _ex entries, and that fp16 embeddings reach
the indexer unconverted while the dataset keeps the reference's fp32 rows."""
import os
import warnings

import numpy as np
import pytest
import torch


@pytest.fixture(scope="module")
def lib():
    from lcrec_b200 import _lib, build
    if not os.path.exists(_lib.LIB_PATH):
        build.build()
    return _lib.load()


@pytest.mark.parametrize("dtype", [3, -1])
def test_ex_entries_refuse_bad_dtype(lib, dtype):
    """dtype outside {0, 1, 2} is LCREC_ERR_ARG with a message naming it, before any handle or device is touched (the
    handles below are dummies that must never be dereferenced)."""
    import ctypes as C
    one = C.c_void_p(8)
    codes = (C.c_int64 * 8)()
    calls = {
        "mlp_forward_ex": lambda: lib.lcrec_mlp_forward_ex(one, one, dtype, 4, one, None, one, 1 << 20, None),
        "indexer_pass0_ex": lambda: lib.lcrec_indexer_pass0_ex(one, one, dtype, 4, 0, None),
        "indexer_run_device_ex": lambda: lib.lcrec_indexer_run_device_ex(one, one, dtype, 4, 20, one, codes, None),
        "indexer_run_host_ex": lambda: lib.lcrec_indexer_run_host_ex(one, one, dtype, 4, 20, one, codes, None),
    }
    for name, call in calls.items():
        assert call() == 1, name
        msg = lib.lcrec_last_error()
        assert b"bad argument" in msg and b"dtype" in msg, (name, msg)


class _FakeIndexer:
    """Records what generate_codes hands to the host path."""

    L = 4

    def __init__(self):
        self.seen = None

    def run_host(self, data, max_rounds=20):
        self.seen = data
        n = int(data.shape[0])
        return torch.zeros((n, self.L), dtype=torch.int64), {"n_unique": n, "max_multiplicity": 1}


def _emb(n=37, d=24, dtype=np.float16):
    return np.random.default_rng(1).standard_normal((n, d)).astype(dtype)


def test_generate_codes_keeps_fp16_ndarray():
    from lcrec_b200 import generate_indices as G
    x = _emb()
    fake = _FakeIndexer()
    codes, stats = G.generate_codes(None, x, indexer=fake)
    assert fake.seen.dtype == torch.float16 and not fake.seen.is_cuda
    assert fake.seen.data_ptr() == x.ctypes.data                         # the caller's array itself, no host copy
    assert codes.shape == (x.shape[0], 4) and stats["collision_rate"] == 0.0


@pytest.mark.parametrize("mmap", [False, True])
def test_generate_codes_keeps_fp16_dataset(tmp_path, mmap):
    from lcrec_b200 import generate_indices as G
    from lcrec_b200.datasets import EmbDataset
    x = _emb()
    path = str(tmp_path / "emb.npy")
    np.save(path, x)
    data = EmbDataset(path, mmap=mmap)
    fake = _FakeIndexer()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)                    # torch.from_numpy of a read-only memory map
        G.generate_codes(None, data, indexer=fake)
    assert fake.seen.dtype == torch.float16
    assert np.array_equal(fake.seen.numpy(), x)
    if mmap:
        assert fake.seen.data_ptr() == data.embeddings.ctypes.data        # still the mapped file, not a copy


def test_generate_codes_converts_other_dtypes_to_fp32():
    from lcrec_b200 import generate_indices as G
    x = _emb(dtype=np.float64)
    fake = _FakeIndexer()
    G.generate_codes(None, x, indexer=fake)
    assert fake.seen.dtype == torch.float32
    assert np.array_equal(fake.seen.numpy(), x.astype(np.float32))


def test_emb_dataset_returns_fp32_rows_of_fp16_file(tmp_path):
    from lcrec_b200.datasets import EmbDataset
    x = _emb()
    path = str(tmp_path / "emb.npy")
    np.save(path, x)
    for mmap in (False, True):
        data = EmbDataset(path, mmap=mmap)
        assert data.dim == x.shape[1] and len(data) == x.shape[0]
        row, rows = data[3], data[[0, 5, 7]]
        assert row.dtype == torch.float32 and rows.dtype == torch.float32
        assert np.array_equal(row.numpy(), x[3].astype(np.float32))
        assert np.array_equal(rows.numpy(), x[[0, 5, 7]].astype(np.float32))
