"""CPU checks of the data-parallel EMA entry: every violated argument condition of lcrec_ema_update_dist is LCREC_ERR_ARG,
raised before any device work (the pointers below are dummies that must never be dereferenced), and the symmetric buffer
size formula."""
import ctypes as C
import os

import pytest
import torch


@pytest.fixture(scope="module")
def lib():
    from lcrec_b200 import _lib, build
    if not os.path.exists(_lib.LIB_PATH):
        build.build()
    return _lib.load()


GOOD = dict(latent=8, indices=8, n_local=3, n_global=5, n_codes=4, e_dim=8, decay=0.99, eps=1e-5, cluster_size=8,
            ema_w=8, codebook=8, gathered_latent=8, gathered_indices=8, flags=8, peers=8, world=2, rank=1,
            rows_per_rank=3, epoch=0)

BAD = [
    ("world", 0), ("world", 65), ("rank", -1), ("rank", 2),
    ("rows_per_rank", 0), ("n_local", -1), ("n_local", 4),
    ("n_global", -1), ("n_global", 7),
    ("e_dim", 0), ("e_dim", 8193), ("n_codes", 0),
    ("peers", None), ("cluster_size", None), ("ema_w", None), ("codebook", None), ("gathered_latent", None),
    ("gathered_indices", None), ("flags", None), ("latent", None), ("indices", None),
]


def _call(lib, a):
    p = lambda v: C.c_void_p(v)                                        # noqa: E731
    return lib.lcrec_ema_update_dist(p(a["latent"]), p(a["indices"]), a["n_local"], a["n_global"], a["n_codes"],
                                     a["e_dim"], a["decay"], a["eps"], p(a["cluster_size"]), p(a["ema_w"]),
                                     p(a["codebook"]), p(a["gathered_latent"]), p(a["gathered_indices"]), p(a["flags"]),
                                     p(a["peers"]), a["world"], a["rank"], a["rows_per_rank"], C.c_uint64(a["epoch"]), None)


@pytest.mark.parametrize("field,value", BAD)
def test_ema_update_dist_refuses_bad_arguments(lib, field, value):
    a = dict(GOOD, **{field: value})
    assert _call(lib, a) == 1, (field, value)
    assert b"bad argument" in lib.lcrec_last_error()


def test_ema_update_dist_refuses_global_batch_beyond_2_31(lib):
    a = dict(GOOD, world=64, rank=0, n_local=0, rows_per_rank=1 << 30, n_global=1 << 31)
    assert _call(lib, a) == 1 and b"bad argument" in lib.lcrec_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="with a GPU the call would go on to launch on the dummy pointers")
def test_ema_update_dist_without_local_rows_needs_no_latent(lib):
    """n_local = 0 with null latent / indices passes the argument checks and stops at the device check."""
    a = dict(GOOD, latent=None, indices=None, n_local=0)
    assert _call(lib, a) == 2                                          # LCREC_ERR_CUDA: no device here, not LCREC_ERR_ARG
    assert b"bad argument" not in lib.lcrec_last_error()


@pytest.mark.parametrize("rows,e_dim", [(1, 1), (3, 8), (512, 32), (513, 100), (4097, 7)])
def test_ema_dist_symmetric_bytes(lib, rows, e_dim):
    def a16(b):
        return (b + 15) // 16 * 16
    slot = a16(a16(8 + 8 * rows) + 4 * rows * e_dim)
    assert lib.lcrec_ema_dist_symmetric_bytes(rows, e_dim) == 256 + 2 * slot
    assert slot % 16 == 0 and a16(8 + 8 * rows) % 16 == 0


@pytest.mark.parametrize("rows,e_dim", [(0, 8), (4, 0), (-1, 8)])
def test_ema_dist_symmetric_bytes_refuses_empty_layout(lib, rows, e_dim):
    assert lib.lcrec_ema_dist_symmetric_bytes(rows, e_dim) == -1
