"""bench.py on CPU: the pieces both arms must agree on (no GPU, no timing)."""
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    sys.path.insert(0, ROOT)
    return importlib.import_module("bench")


def test_reference_sample_is_a_pure_function_of_steps_and_warmup():
    b = _bench()
    assert b.reference_sample_items(3, 3) == 25000 and b.reference_sample_items(5, 1) == 25000        # C1 in full
    assert b.reference_sample_items(5, 3) == 18750 and b.reference_sample_items(20, 5) == 6000
    assert b.reference_sample_items(1000, 0) == 2048
    for k, w in ((5, 3), (20, 5), (3, 3)):
        a, c = b.workload_config(1, 1_000_000, k, w), b.workload_config(1, 1_000_000, k, w)
        assert a == c and str(b.reference_sample_items(k, w)) in a["workload"] and a["reference_sample_items"] == b.reference_sample_items(k, w)


def test_config_switch_sets_the_c5_shape():
    b = _bench()
    try:
        b.set_config("c5")
        assert b.DIMS[-1] == 256 and b.N_CODES == [8192] * 4 and b.E_DIM == 256
        assert b.FLOP_PER_ITEM == 2 * sum(x * y for x, y in zip(b.DIMS[:-1], b.DIMS[1:])) + 4 * 2 * 8192 * 256
        assert "8192" in b.workload_config(8, 250000, 2, 2)["workload"]
    finally:
        b.DIMS = [4096, 2048, 1024, 512, 256, 128, 64, 32]; b.N_CODES = [256] * 4; b.E_DIM = 32
        b.set_config("c3")
    assert b.FLOP_PER_ITEM == 22433792 and b.BYTES_PER_ITEM == 16416            # SURVEY 8(d)


def test_reference_arm_runs_the_staged_reference_script(tmp_path):
    """`bench.py --impl reference` on a tiny sample: one JSON line, kind "reference" when baseline/_ref is staged (build container),
    the numpy port otherwise; never touches a GPU."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample", "256"],
                       capture_output=True, text=True, timeout=600, env=env, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-500:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    staged = os.path.isfile(os.path.join(ROOT, "baseline", "_ref", "index", "generate_indices.py"))
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] == ("reference" if staged else "port")
    assert line["value"] > 0 and line["e2e"]["h2d_bytes_per_step"] == 0 and line["config"]["reference_sample_items"] == 256
    assert line["cpu_baseline"]["cores"] >= 1


def test_dump_outputs_writes_float_arrays_within_the_budget(tmp_path):
    """--dump-outputs: codes come back exactly as float32; above the byte budget the same seeded rows are kept in every run."""
    b = _bench()
    codes = (np.arange(4000, dtype=np.int64) * 7919 % 256).reshape(1000, 4)
    b.dump_outputs(str(tmp_path / "all"), {"codes": codes}, 1 << 20)
    got = np.load(tmp_path / "all" / "codes.npy")
    assert got.dtype == np.float32 and np.array_equal(got, codes) and not (tmp_path / "all" / "codes_rows.npy").exists()
    for run in ("s1", "s2"):
        b.dump_outputs(str(tmp_path / run), {"codes": torch.from_numpy(codes)}, 6000)
    rows = np.load(tmp_path / "s1" / "codes_rows.npy")
    got = np.load(tmp_path / "s1" / "codes.npy")
    assert rows.dtype == np.float64 and got.nbytes + rows.nbytes <= 6000 and len(rows) == 250 and (np.diff(rows) > 0).all()
    assert np.array_equal(got, codes[rows.astype(np.int64)])
    assert np.array_equal(rows, np.load(tmp_path / "s2" / "codes_rows.npy")) and np.array_equal(got, np.load(tmp_path / "s2" / "codes.npy"))


def test_bench_rejects_zero_steps_and_dumps_outside_the_gpu_arm(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)], ["--config", "c2", "--dump-outputs", str(tmp_path)]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120,
                           env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), cwd=str(tmp_path))
        assert r.returncode == 2 and ("--steps" in r.stderr or "--dump-outputs" in r.stderr), r.stderr[-300:]
