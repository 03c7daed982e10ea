"""bench.py --dump-outputs: the proofs of the last timed step, written as float32 arrays of proof bytes."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def test_dump_outputs_writes_exact_bytes_and_a_fixed_sample(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    rng = np.random.default_rng(3)
    recs = {"a": [rng.bytes(40) for _ in range(10)], "b": [rng.bytes(24) for _ in range(6)]}
    bench.dump_outputs(str(tmp_path / "full"), recs)
    for name, rows in recs.items():
        got = np.load(tmp_path / "full" / (name + ".npy"))
        assert got.dtype == np.float32 and got.shape == (len(rows), len(rows[0]))
        assert got.astype(np.uint8).tobytes() == b"".join(rows)
    # over the limit: the same share of every array's rows, the same rows from run to run
    limit = 4 * (5 * 40 + 3 * 24)
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", limit)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), recs)
    total = 0
    for name, rows in recs.items():
        s1, s2 = np.load(tmp_path / "s1" / (name + ".npy")), np.load(tmp_path / "s2" / (name + ".npy"))
        assert s1.tobytes() == s2.tobytes() and len(s1) == len(rows) // 2
        assert all(r.astype(np.uint8).tobytes() in rows for r in s1)
        total += s1.nbytes
    assert total <= limit


@pytest.mark.gpu
def test_bench_dumps_the_proofs_of_its_last_timed_step(tmp_path, oracle_cpu, srs_fixture):
    from taiga_b200 import circuits_taiga
    out = tmp_path / "out"
    env = dict(os.environ, TB_SYNTH_PROCS="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "0", "--ptx", "1",
                        "--no-sweep", "--no-cpu", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=1200, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    # one partial transaction: 2 Compliance-shaped and 4 VP-shaped proofs; witness seeds as in ProverService.synthesize_ptx (rank 0)
    for compliance, name, rows, plen, seed0 in ((True, "compliance_proofs", 2, 4480, 0), (False, "vp_proofs", 4, 4448, 50000)):
        a = np.load(out / (name + ".npy"))
        assert a.dtype == np.float32 and a.shape == (rows, plen)
        assert np.all((a >= 0) & (a <= 255) & (a == np.round(a)))
        kd, make = circuits_taiga.build(compliance)
        key = oracle_cpu.OracleKey(kd, srs_fixture)
        for i in (0, rows - 1):
            _, inst, lens = kd.witness_arrays(make(seed0 + i))
            assert key.verify(inst, lens, a[i].astype(np.uint8).tobytes()) == 0, (name, i)
