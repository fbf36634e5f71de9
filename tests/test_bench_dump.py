"""bench.py --dump-outputs: the PSM table of the last timed step, one float32 / float64 .npy per field, the same from run to
run with the same arguments, and never more than bench.DUMP_BYTES in all.  CPU only: the reference arm (the oracle)
times the same workload, and the size cap is checked on a synthetic table."""
import importlib.util
import os
import subprocess
import sys

import numpy as np

from maxdecoy import _abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def _bench_module():
    spec = importlib.util.spec_from_file_location("bench", BENCH)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_reference_arm_dump_is_reproducible(tmp_path):
    runs = []
    for k in range(2):
        out = tmp_path / ("run%d" % k)
        subprocess.check_call([sys.executable, BENCH, "--impl", "reference", "--config", "c1", "--spectra", "12", "--ref-sample", "12",
                               "--steps", "2", "--warmup", "0", "--dump-outputs", str(out)], stdout=subprocess.DEVNULL, timeout=600)
        runs.append(_load(out))
    a, b = runs
    assert set(a) == set(b) and {"raw_score", "candidate", "rank", "score", "spectrum_row"} <= set(a)
    for name, arr in a.items():
        assert arr.dtype in (np.float32, np.float64), name
        assert np.array_equal(arr, b[name]), name
    assert a["rank"].shape == (12, 5) and np.array_equal(a["spectrum_row"], np.arange(12))
    assert np.all(a["rank"][:, 0] == 1) and np.all(a["raw_score"][:, 0] > 0)


def test_dump_is_capped_by_a_seeded_sample(tmp_path):
    bench = _bench_module()
    n, k = 160_000, 5
    table = np.zeros((n, k), dtype=_abi.PSM_DTYPE)
    table["spectrum_id"] = np.arange(n, dtype=np.uint32)[:, None]
    table["rank"] = np.arange(1, k + 1, dtype=np.uint16)
    table["var_mask"] = np.uint64(1 << 59) | np.arange(n, dtype=np.uint64)[:, None]
    table["raw_score"] = np.arange(n * k, dtype=np.int64).reshape(n, k) * 1000
    for d in ("a", "b"):
        bench.dump_outputs(table, str(tmp_path / d))
    total = sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a"))
    assert total <= bench.DUMP_BYTES
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert all(np.array_equal(a[f], b[f]) for f in a)
    rows = a["spectrum_row"].astype(np.int64)
    assert 100_000 < len(rows) < n and np.all(np.diff(rows) > 0)
    assert np.array_equal(a["spectrum_id"][:, 0], rows)
    assert np.array_equal(a["raw_score"], table["raw_score"][rows].astype(np.float64))
    vm = a["var_mask_hi32"].astype(np.uint64) << np.uint64(32) | a["var_mask_lo32"].astype(np.uint64)
    assert np.array_equal(vm, table["var_mask"][rows])
