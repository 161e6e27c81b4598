"""bench.py --dump-outputs: what the last timed step returned, written so that two builds can be compared output for output.  Two runs
with the same arguments write the same files; at this size the dump holds every number and the whole file, which decode back to the
bench's seeded inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHUNKS = 4
NAMES = ("chunk_compressed_bytes", "compressed", "decompressed", "index")


def _bench(out_dir):
    argv = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "0", "--chunks", str(CHUNKS),
            "--no-e2e", "--no-cpu-baseline", "--no-index-free", "--dump-outputs", str(out_dir)]
    res = subprocess.run(argv, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-4000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    return {name: np.load(os.path.join(out_dir, name + ".npy")) for name in NAMES}


def test_dump_is_repeatable_and_decodes_to_the_inputs(oracle, tmp_path):
    from pcodec_b200 import datagen

    first, second = _bench(tmp_path / "a"), _bench(tmp_path / "b")
    assert sorted(os.listdir(tmp_path / "a")) == sorted(n + ".npy" for n in NAMES)
    assert sum(os.path.getsize(tmp_path / "a" / (n + ".npy")) for n in NAMES) <= 64 << 20
    for name in NAMES:
        assert first[name].dtype in (np.float32, np.float64), name
        np.testing.assert_array_equal(first[name], second[name], err_msg=name)

    nums = np.concatenate([datagen.c2_u64_cumsum_geometric(datagen.CHUNK_N, seed=c) for c in range(CHUNKS)])
    np.testing.assert_array_equal(first["decompressed"], nums.astype(np.float64))
    file = first["compressed"].astype(np.uint8).tobytes()
    assert first["chunk_compressed_bytes"].size == CHUNKS and 0 < first["chunk_compressed_bytes"].sum() < len(file)
    np.testing.assert_array_equal(oracle.simple_decompress(file, np.uint64), nums)
