"""CPU check of bench.py --dump-outputs on the reference arm: the files hold, in float32 / float64, the digests of a row
sample of the benchmark's keys that is fixed by its seed, so that two builds run with the same arguments can be compared."""
import os
import subprocess
import sys

import numpy as np

import oracle
from bench import DUMP_MAX_BYTES, DUMP_ROWS, dump_rows
from tests.util import random_keys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_rows_seeded_sample():
    n = 10 * DUMP_ROWS
    rows = dump_rows(n)
    assert len(rows) == DUMP_ROWS and (np.diff(rows) > 0).all() and rows[-1] < n
    assert (rows == dump_rows(n)).all()
    assert (dump_rows(100) == np.arange(100)).all()
    assert DUMP_ROWS * 32 * 4 + DUMP_ROWS * 8 <= DUMP_MAX_BYTES


def test_reference_arm_dumps_its_digests(tmp_path):
    n = DUMP_ROWS + 5000
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--keys", str(n),
                        "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    digests = np.load(tmp_path / "keccak_digests.npy")
    rows = np.load(tmp_path / "keccak_digest_rows.npy")
    assert digests.dtype == np.float32 and digests.shape == (DUMP_ROWS, 32)
    assert rows.dtype == np.float64 and (rows == dump_rows(n)).all()
    want = oracle.keccak256_fixed(random_keys(2, n)[rows.astype(np.int64)])
    assert (digests == want).all()
