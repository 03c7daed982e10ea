"""GPU: tb_check_batch (MockProver::verify on the device) against the Python restatement (oracle/mock_prover.py) array
for array, against what the prover and verifier do with the same witnesses, across threads and internal chunks."""
import ctypes
import os
import random
import threading

import numpy as np
import pytest

from conftest import GOLDEN

from oracle import mock_prover as mp
from taiga_b200 import circuits_mini as cm
from taiga_b200 import lib
from taiga_b200.circuit import P

pytestmark = pytest.mark.gpu

S_ROT, S_LK = 5, 6   # selector columns of circuits_mini.standard_plonk

_SRS = {}


@pytest.fixture(scope="module")
def mini_srs(oracle_cpu, gpu_ctx):
    def get(k):
        if k not in _SRS:
            s = oracle_cpu.synthetic_srs(k, seed=k)
            _SRS[k] = gpu_ctx.load_srs(k, s["g"], s["g_lagrange"], s["w"], s["u"])
        return _SRS[k]
    return get


def device_arrays(reports):
    return np.stack([r.fail_rows for r in reports]), np.stack([r.first_row for r in reports])


def corrupt(kd, asg, cls, rnd):
    """One seeded corruption of the given class on an Assignment of standard_plonk."""
    if cls == "gate":       # any advice cell of the gate regions (rows 0..9)
        asg.advice[rnd.randrange(kd.cs.num_advice)][rnd.randrange(10)] = rnd.randrange(P)
    elif cls == "copy":     # a cell of a copy constraint
        (col, row), _ = rnd.choice(asg.copies)     # the first cell of every copy of standard_plonk is an advice cell
        asg.advice[col.index][row] = rnd.randrange(P)
    elif cls == "lookup":   # a lookup row, often outside the table
        rows = [r for r, v in asg.fixed[S_LK].items() if v == 1]
        asg.advice[rnd.randrange(2)][rnd.choice(rows)] = rnd.randrange(24)
    return asg


def witnesses(kd, make, B, seed):
    """B witnesses: every third satisfying, the others with one seeded corruption of a class in turn; blinding rows random."""
    rnd = random.Random(seed)
    adv, inst = [], []
    for b in range(B):
        asg = make(1000 + b)
        if b % 3:
            corrupt(kd, asg, ("gate", "copy", "lookup")[(b + b // 3) % 3], rnd)
        a, i, lens = kd.witness_arrays(asg)
        a[:, asg.usable:] = np.frombuffer(rnd.randbytes(a[:, asg.usable:].size), np.uint8).reshape(a[:, asg.usable:].shape)
        a[:, asg.usable:, 31] &= 0x3F
        adv.append(a)
        inst.append(i)
    return np.stack(adv), np.stack(inst), lens


@pytest.mark.parametrize("k,wide,nl,B", [(6, False, 2, 1), (6, False, 2, 3), (7, True, 1, 33), (6, False, 2, 70), (9, True, 2, 3), (6, False, 0, 33)])
def test_parity_with_restatement_mini(mini_srs, k, wide, nl, B):
    kd, make = cm.standard_plonk(k=k, wide=wide, n_lookups=nl)
    pk = mini_srs(k).load_circuit(kd)
    adv, inst, lens = witnesses(kd, make, B, seed=k * 1000 + B)
    fail, first = device_arrays(pk.check_batch(adv, inst, lens))
    ref_fail, ref_first = mp.check(kd, adv, inst, lens)
    np.testing.assert_array_equal(fail, ref_fail)
    np.testing.assert_array_equal(first, ref_first)
    assert ref_fail[0::3].sum() == 0 and (B == 1 or ref_fail.any())


@pytest.mark.parametrize("k", [6, 7])
def test_parity_with_restatement_seeded_corruptions(mini_srs, k):
    """20 seeded random corruptions of each class in one batch of 60 (two internal chunks)."""
    kd, make = cm.standard_plonk(k=k, wide=(k == 7), n_lookups=2)
    pk = mini_srs(k).load_circuit(kd)
    rnd = random.Random(k)
    wit = [kd.witness_arrays(corrupt(kd, make(5), cls, rnd)) for cls in ("gate", "copy", "lookup") for _ in range(20)]
    adv, inst, lens = np.stack([w[0] for w in wit]), np.stack([w[1] for w in wit]), wit[0][2]
    fail, first = device_arrays(pk.check_batch(adv, inst, lens))
    ref_fail, ref_first = mp.check(kd, adv, inst, lens)
    np.testing.assert_array_equal(fail, ref_fail)
    np.testing.assert_array_equal(first, ref_first)


def test_parity_poison_in_the_key(mini_srs):
    """Selector set in a blinding row and a rotation reaching past the usable rows: poisoned, never unsatisfied."""
    kd, make = cm.standard_plonk(k=6, n_lookups=1)
    C = sum(len(ps) for _, ps in kd.cs.gates)
    usable = kd.n - kd.blinding_factors - 1
    for row in (usable - 1, kd.n - 2):
        kd.fixed[S_ROT, row] = 0
        kd.fixed[S_ROT, row, 0] = 1
    pk = mini_srs(6).load_circuit(kd)
    adv, inst, lens = kd.witness_arrays(make(3))
    rep = pk.check_batch(adv[None], inst[None], lens)[0]
    ref_fail, ref_first = mp.check(kd, adv[None], inst[None], lens)
    np.testing.assert_array_equal(rep.fail_rows, ref_fail[0])
    np.testing.assert_array_equal(rep.first_row, ref_first[0])
    assert {f[0] for f in rep.failures} == {"poisoned"}
    assert any("poisoned" in line for line in rep.describe(kd))


@pytest.mark.parametrize("compliance", [True, False])
def test_taiga_shapes(gpu_srs, compliance):
    from taiga_b200 import circuits_taiga as ct
    kd, make = ct.build(compliance)
    pk = gpu_srs.load_circuit(kd)
    wit = [kd.witness_arrays(make(40 + b)) for b in range(3)]
    adv, inst, lens = np.stack([w[0] for w in wit]), np.stack([w[1] for w in wit]), wit[0][2]
    assert all(r.ok for r in pk.check_batch(adv, inst, lens))
    # one corrupted witness under the Python reference: a cell of a copy constraint and a cell of a used row
    asg = make(40)
    (col, row), _ = next(c for c in asg.copies if c[0][0].kind == 0)
    asg.advice[col.index][row] = (asg.advice[col.index][row] + 1) % P
    asg.advice[0][1] = (asg.advice[0].get(1, 0) + 5) % P
    bad = kd.witness_arrays(asg)[0]
    adv[1] = bad
    reps = pk.check_batch(adv, inst, lens)
    ref_fail, ref_first = mp.check(kd, bad[None], inst[1:2], lens)
    np.testing.assert_array_equal(reps[1].fail_rows, ref_fail[0])
    np.testing.assert_array_equal(reps[1].first_row, ref_first[0])
    assert [r.ok for r in reps] == [True, False, True]
    assert "copy" in {f[0] for f in reps[1].failures}


@pytest.mark.parametrize("nl", [0, 1])
def test_agrees_with_prover_and_verifier(mini_srs, nl):
    """Gate / copy corruptions: reported ok <=> the proof of that witness verifies.  Single-expression lookups:
    a lookup failure <=> tb_prove_batch raises ConstraintSystemFailure."""
    kd, make = cm.standard_plonk(k=6, n_lookups=nl)
    pk = mini_srs(6).load_circuit(kd)
    rnd = random.Random(nl)
    classes = ("gate", "copy") + (("lookup",) if nl else ())
    for i in range(12):
        cls = classes[i % len(classes)]
        adv, inst, lens = kd.witness_arrays(corrupt(kd, make(7 + i), cls, rnd) if i % 4 else make(7 + i))
        rep = pk.check_batch(adv[None], inst[None], lens)[0]
        lookup_fail = any(f[0] == "lookup" for f in rep.failures)
        try:
            proof = pk.prove_batch(adv[None], inst[None], lens, bytes(range(32)))
        except lib.ConstraintSystemFailure:
            assert lookup_fail
            continue
        assert not lookup_fail
        assert pk.verify_batch(inst[None], lens, proof) == [rep.ok], (cls, rep)


def test_determinism_threads_and_golden_proof(mini_srs, gpu_ctx):
    kd, make = cm.standard_plonk(k=6, n_lookups=2)
    pk = mini_srs(6).load_circuit(kd)
    adv, inst, lens = witnesses(kd, make, 40, seed=3)
    first = device_arrays(pk.check_batch(adv, inst, lens))
    again = device_arrays(pk.check_batch(adv, inst, lens))
    np.testing.assert_array_equal(first[0], again[0])
    np.testing.assert_array_equal(first[1], again[1])
    ctxs = [lib.Context(0), lib.Context(0)]
    out, errs = [None, None], []

    def run(i):
        try:
            out[i] = [device_arrays(pk.check_batch(adv, inst, lens, ctx=ctxs[i])) for _ in range(3)]
        except BaseException as e:  # re-raised below
            errs.append(e)
    th = [threading.Thread(target=run, args=(i,)) for i in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errs, errs
    for res in out:
        for f, r in res:
            np.testing.assert_array_equal(f, first[0])
            np.testing.assert_array_equal(r, first[1])
    for c in ctxs:
        c.close()
    # the prover on the same context still reproduces the committed golden proof (witness 100, proof index 5)
    a, i, l = kd.witness_arrays(make(100))
    proof = pk.prove_batch(a[None], i[None], l, bytes((7 * j + 1) & 0xFF for j in range(32)), first_proof_index=5)[0]
    assert proof == open(os.path.join(GOLDEN, "proof_k6_plonk.bin"), "rb").read()


def test_argument_errors_launch_nothing(mini_srs, gpu_ctx):
    kd, make = cm.standard_plonk(k=6, n_lookups=2)
    pk = mini_srs(6).load_circuit(kd)
    adv, inst, lens = kd.witness_arrays(make(1))
    L = gpu_ctx._lib
    S = L.tb_pk_check_slots(pk._h)
    fail, first = np.zeros(S, np.uint32), np.zeros(S, np.uint32)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)   # noqa: E731
    big = np.array([kd.n], np.uint32)
    before = gpu_ctx.launch_count
    assert L.tb_check_batch(gpu_ctx._h, pk._h, 0, p(adv), p(inst), p(lens), p(fail), p(first)) == lib.TB_ERR_INVALID
    assert L.tb_check_batch(gpu_ctx._h, pk._h, 1, p(adv), p(inst), p(lens), None, p(first)) == lib.TB_ERR_INVALID
    assert L.tb_check_batch(gpu_ctx._h, pk._h, 1, p(adv), p(inst), p(lens), p(fail), None) == lib.TB_ERR_INVALID
    assert L.tb_check_batch(gpu_ctx._h, pk._h, 1, p(adv), p(np.zeros(kd.n * 32, np.uint8)), p(big), p(fail), p(first)) == lib.TB_ERR_INVALID
    assert L.tb_check_batch(gpu_ctx._h, pk._h, 4097, p(adv), p(inst), p(lens), p(fail), p(first)) == lib.TB_ERR_INVALID
    assert gpu_ctx.launch_count == before


def test_service_check_ptx_batch(srs_fixture):
    from oracle.mock_prover import decode_sigma
    from taiga_b200.ptx import ProverService
    svc = ProverService(0, srs_fixture, c_workers=1, v_workers=1)
    wit = svc.synthesize_ptx(2, wseed=3, procs=1)
    creps, vreps = svc.check_ptx_batch(wit)
    assert len(creps) == 4 and len(vreps) == 8 and all(r.ok for r in creps + vreps)
    # flip one byte of an advice cell that a copy constraint ties to another cell
    to_c, to_r = decode_sigma(svc.kd_c)
    cols = svc.kd_c.cs.perm_columns
    p, r = next((p, r) for p in range(len(cols)) if cols[p].kind == 0 for r in range(svc.kd_c.n) if (to_c[p, r], to_r[p, r]) != (p, r))
    wit["c_adv"][2, cols[p].index, r, 0] ^= 1
    creps, vreps = svc.check_ptx_batch(wit)
    assert [rep.ok for rep in creps] == [True, True, False, True] and all(rep.ok for rep in vreps)
    assert any(f[0] == "copy" for f in creps[2].failures)
