"""bench.py --dump-outputs: what the last timed step returned, as float32 .npy files under a size cap, identical
from run to run.  Exercised on the CPU arm (oracle/cpu); the GPU arm writes the same files plus the verdicts of
its timed verify leg."""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_dump(out):
    subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--workload', 'config1',
                    '--steps', '1', '--warmup', '0', '--dump-outputs', str(out)], check=True, stdout=subprocess.DEVNULL)
    return {n[:-4]: np.load(os.path.join(out, n)) for n in sorted(os.listdir(out))}


def test_dump_outputs_reproducible(tmp_path):
    import __graft_entry__ as g
    g.build_oracle_cpu()
    a = _bench_dump(tmp_path / 'a')
    b = _bench_dump(tmp_path / 'b')
    assert sorted(a) == ['proof_len', 'proof_rows', 'proofs', 'status']
    for name in a:
        assert a[name].dtype == np.float32 and np.array_equal(a[name], b[name]), name
    assert sum(os.path.getsize(tmp_path / 'a' / (n + '.npy')) for n in a) <= 64 * 10 ** 6
    assert not a['status'].any()
    for row, b_idx in enumerate(a['proof_rows'].astype(int)):
        ln = int(a['proof_len'][b_idx])
        assert ln > 0 and a['proofs'][row, :ln].any() and not a['proofs'][row, ln:].any()


def test_dump_rows_seeded_sample_within_budget():
    import bench
    B, row_bytes, fixed = 8192, 160000, 5 * 4 * 8192
    rows = bench.dump_rows(B, row_bytes, fixed)
    assert 1 <= len(rows) < B and np.all(np.diff(rows) > 0) and rows[-1] < B
    assert 4 * row_bytes * len(rows) + fixed <= bench.DUMP_BYTES
    assert np.array_equal(rows, bench.dump_rows(B, row_bytes, fixed))
    assert np.array_equal(bench.dump_rows(8, 100, 0), np.arange(8))
