"""Sharded `generate_indices` on CPU: the parallel assembly of the `.index.json` (write_index_json_parts) with gloo on 2 and
3 ranks, empty ranks included, against the bytes of the reference's json.dump; and the argument checks of the new C entries
(lcrec_indexer_pass0_host_ex, lcrec_index_json_ex), which refuse bad arguments before anything touches a device."""
import ctypes as C
import json
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from lcrec_b200 import generate_indices as G
from lcrec_b200.distributed import ShardPlan


def _table(n, L, seed):
    rng = np.random.default_rng(seed)
    codes = rng.integers(0, 300, size=(n, L)).astype(np.int64)
    if n > 3:
        codes[1] = 0; codes[2] = 299
    return codes


def _dump(codes, base=0):
    return json.dumps({base + i: [G.PREFIX[l].format(int(v)) for l, v in enumerate(row)] for i, row in enumerate(codes.tolist())})


def _fragment(codes, base):
    """What ops.index_json_bytes(codes, base, braces=False) formats on the device: the rows without braces, ", " in front
    of every row whose key is not 0."""
    if codes.shape[0] == 0:
        return b""
    return ((", " if base else "") + _dump(codes, base)[1:-1]).encode()


def _worker(rank, world, port, n, L, path):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        plan = ShardPlan(n, world)
        codes = _table(n, L, n + L)[plan.slice(rank)]
        G.write_index_json_parts(_fragment(codes, plan.start(rank)), path)
        assert os.path.getsize(path) == len(_dump(_table(n, L, n + L)))      # complete on every rank when it returns
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("world,n,L", [(2, 0, 3), (2, 1, 4), (2, 7, 1), (3, 2, 5), (3, 101, 4), (3, 12, 2)])
def test_parallel_file_write_equals_json_dump(tmp_path, world, n, L):
    """n < world leaves ranks empty; n = 101 on 3 ranks crosses the 2- and 3-digit keys inside blocks."""
    path = str(tmp_path / "Toy.index.json")
    with open(path, "wb") as f:                                   # an older, longer file is replaced, not patched
        f.write(b"x" * 10000)
    mp.spawn(_worker, args=(world, _free_port(), n, L, path), nprocs=world, join=True)
    codes = _table(n, L, n + L)
    want = _dump(codes)
    assert open(path, "rb").read() == want.encode()
    assert json.loads(want) == {str(k): v for k, v in G.codes_to_index_dict(codes).items()}


def test_fragment_stand_in_concatenates_to_the_table():
    codes = _table(23, 3, 0)
    for cuts in ([0, 23], [0, 9, 10, 23], [0, 0, 5, 5, 23]):
        body = b"".join(_fragment(codes[a:b], a) for a, b in zip(cuts[:-1], cuts[1:]))
        assert b"{" + body + b"}" == _dump(codes).encode()


@pytest.fixture(scope="module")
def lib():
    from lcrec_b200 import _lib, build
    if not os.path.exists(_lib.LIB_PATH):
        build.build()
    return _lib.load()


def test_new_entries_refuse_bad_arguments(lib):
    null, one = C.c_void_p(0), C.c_void_p(8)      # a non-null dummy: never dereferenced on these paths
    cases = {
        "pass0_host null indexer": lambda: lib.lcrec_indexer_pass0_host_ex(null, one, 0, 10, 0, 10, null),
        "pass0_host dtype": lambda: lib.lcrec_indexer_pass0_host_ex(one, one, 3, 10, 0, 10, null),
        "pass0_host row_begin < 0": lambda: lib.lcrec_indexer_pass0_host_ex(one, one, 0, 10, -1, 2, null),
        "pass0_host past n_total": lambda: lib.lcrec_indexer_pass0_host_ex(one, one, 1, 10, 8, 3, null),
        "pass0_host row_begin > n_total": lambda: lib.lcrec_indexer_pass0_host_ex(one, one, 0, 10, 11, 0, null),
        "pass0_host n < 0": lambda: lib.lcrec_indexer_pass0_host_ex(one, one, 0, 10, 0, -1, null),
        "json_ex levels": lambda: lib.lcrec_index_json_ex(one, 4, 6, 0, 1, one, 100, one, one, 100, null),
        "json_ex item_base < 0": lambda: lib.lcrec_index_json_ex(one, 4, 4, -1, 0, one, 100, one, one, 100, null),
        "json_ex braces": lambda: lib.lcrec_index_json_ex(one, 4, 4, 0, 2, one, 100, one, one, 100, null),
        "json_ex key overflow": lambda: lib.lcrec_index_json_ex(one, 4, 4, (1 << 63) - 2, 0, one, 100, one, one, 100, null),
        "json_ex n < 0": lambda: lib.lcrec_index_json_ex(one, -1, 4, 0, 0, one, 100, one, one, 100, null),
    }
    for name, call in cases.items():
        assert call() == 1, name
        assert b"bad argument" in lib.lcrec_last_error(), name
