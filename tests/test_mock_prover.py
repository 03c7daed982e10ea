"""CPU: the Python restatement of halo2 MockProver::verify (oracle/mock_prover.py), the reference tb_check_batch is
tested against, accepts satisfying witnesses, decodes sigma back to the copy classes it was built from, and reports
hand-made corruptions in the expected slot and row."""
import numpy as np
import pytest

from oracle import mock_prover as mp
from taiga_b200 import circuits_mini as cm
from taiga_b200.circuit import ADVICE, P

A, B_, C_ = 0, 1, 2            # advice columns a, b, c of standard_plonk
S_ROT, S_LK = 5, 6              # fixed columns of its selectors


def slots(kd):
    C = sum(len(ps) for _, ps in kd.cs.gates)
    return C, len(kd.cs.lookups), len(kd.cs.perm_columns)


def failures(kd, asg, lens=None, inst=None):
    adv, inst_, lens_ = kd.witness_arrays(asg)
    fail, first = mp.check(kd, adv[None], inst_[None] if inst is None else inst[None], lens_ if lens is None else lens)
    return {int(s): (int(first[0, s]), int(fail[0, s])) for s in np.flatnonzero(fail[0])}


def copy_classes(cs, copies):
    """Union-find over the cells of Assignment.copies: the non-trivial equality classes as frozensets of (column index, row)."""
    idx = {c: i for i, c in enumerate(cs.perm_columns)}
    parent = {}

    def find(x):
        while parent.setdefault(x, x) != x:
            x = parent[x]
        return x
    for (ca, ra), (cb, rb) in copies:
        parent[find((idx[ca], ra))] = find((idx[cb], rb))
    groups = {}
    for x in parent:
        groups.setdefault(find(x), set()).add(x)
    return {frozenset(g) for g in groups.values() if len(g) > 1}


def sigma_cycles(kd):
    to_c, to_r = mp.decode_sigma(kd)
    seen, cycles = set(), set()
    for c in range(to_c.shape[0]):
        for r in range(kd.n):
            if (c, r) in seen or (int(to_c[c, r]), int(to_r[c, r])) == (c, r):
                continue
            cyc, x = set(), (c, r)
            while x not in cyc:
                cyc.add(x)
                x = (int(to_c[x]), int(to_r[x]))
            seen |= cyc
            cycles.add(frozenset(cyc))
    return cycles


@pytest.mark.parametrize("k,wide,nl", [(6, False, 2), (7, True, 1), (6, False, 0), (9, True, 2), (12, False, 1)])
def test_accepts_satisfying_mini_witnesses(k, wide, nl):
    kd, make = cm.standard_plonk(k=k, wide=wide, n_lookups=nl)
    wit = [kd.witness_arrays(make(100 + b)) for b in range(2)]
    fail, first = mp.check(kd, np.stack([w[0] for w in wit]), np.stack([w[1] for w in wit]), wit[0][2])
    assert fail.shape == (2, 2 * slots(kd)[0] + slots(kd)[1] + slots(kd)[2])
    assert not fail.any() and (first == mp.NO_ROW).all()


def test_accepts_satisfying_vp_shape_witness():
    from taiga_b200 import circuits_taiga as ct
    kd, make = ct.build(False)
    adv, inst, lens = kd.witness_arrays(make(41))
    fail, _ = mp.check(kd, adv[None], inst[None], lens)
    assert not fail.any()


@pytest.mark.parametrize("k,wide,nl", [(6, False, 2), (7, True, 1)])
def test_sigma_decode_gives_the_copy_classes_mini(k, wide, nl):
    kd, make = cm.standard_plonk(k=k, wide=wide, n_lookups=nl)
    assert sigma_cycles(kd) == copy_classes(kd.cs, make(1).copies)


@pytest.mark.parametrize("compliance", [True, False])
def test_sigma_decode_gives_the_copy_classes_taiga(compliance):
    from taiga_b200 import circuits_taiga as ct
    kd, make = ct.build(compliance)
    assert sigma_cycles(kd) == copy_classes(kd.cs, make(1).copies)


def test_malformed_sigma_is_rejected():
    kd, make = cm.standard_plonk(k=6)
    kd.sigma[1, 3, 0] ^= 1
    adv, inst, lens = kd.witness_arrays(make(1))
    with pytest.raises(ValueError):
        mp.check(kd, adv[None], inst[None], lens)


def test_gate_corruption_fails_at_the_reading_rows():
    kd, make = cm.standard_plonk(k=6, n_lookups=0)
    asg = make(1)
    R = next(r for r, v in asg.fixed[S_ROT].items() if v == 1)
    asg.advice[C_][R + 1] = (asg.advice[C_][R + 1] + 1) % P        # read as c(next) by the rotation gate at row R only
    assert failures(kd, asg) == {1: (R, 1)}                          # "rot" polynomial 0, unsatisfied
    asg = make(1)
    asg.advice[B_][R] = 2                                            # b at R: both rotation polynomials read it
    assert failures(kd, asg) == {1: (R, 1), 2: (R, 1)}


def test_broken_copy_fails_at_the_cells_of_its_cycle():
    kd, make = cm.standard_plonk(k=6, n_lookups=0)
    C, L, _ = slots(kd)
    asg = make(1)
    row = 6                                                          # a == 7, copied from the constants column
    assert asg.advice[A][row] == 7
    cyc = next(c for c in sigma_cycles(kd) if (0, row) in c)
    asg.advice[A][row] = 8
    assert failures(kd, asg) == {2 * C + L + col: (r, 1) for col, r in cyc}


def test_lookup_input_outside_the_table():
    kd, make = cm.standard_plonk(k=6, n_lookups=1)
    C, _, _ = slots(kd)
    asg = make(1)
    row = max(r for r, v in asg.fixed[S_LK].items() if v == 1)
    asg.advice[A][row] = 999
    assert failures(kd, asg) == {2 * C: (row, 1)}


def test_lookup_membership_is_exact_on_tuples():
    """(a, b) = (2, 9): 2 is in the first table column and 9 in the second, but (2, 9) is not a table row."""
    kd, make = cm.standard_plonk(k=6, n_lookups=2)
    C, _, _ = slots(kd)
    asg = make(1)
    row = max(r for r, v in asg.fixed[S_LK].items() if v == 1)
    asg.advice[A][row], asg.advice[B_][row] = 2, 9
    assert failures(kd, asg) == {2 * C + 1: (row, 1)}


def test_selector_in_a_blinding_row_is_poisoned_not_unsatisfied():
    kd, make = cm.standard_plonk(k=6, n_lookups=0)
    C, _, _ = slots(kd)
    row = kd.n - 2
    kd.fixed[S_ROT, row] = 0
    kd.fixed[S_ROT, row, 0] = 1
    assert failures(kd, make(1)) == {C + 1: (row, 1), C + 2: (row, 1)}


def test_rotation_past_usable_is_poisoned_not_unsatisfied():
    kd, make = cm.standard_plonk(k=6, n_lookups=0)
    C, _, _ = slots(kd)
    usable = kd.n - kd.blinding_factors - 1
    kd.fixed[S_ROT, usable - 1] = 0
    kd.fixed[S_ROT, usable - 1, 0] = 1                               # c(next) of that row is the first blinding row
    assert failures(kd, make(1)) == {C + 1: (usable - 1, 1)}         # b(1 - b) reads only row usable - 1: real zero


def test_instance_beyond_its_length_reads_zero():
    kd, make = cm.standard_plonk(k=6, n_lookups=0)
    C, L, _ = slots(kd)
    asg = make(1)
    adv, inst, lens = kd.witness_arrays(asg)
    inst_col = kd.cs.perm_columns.index(next(c for c in kd.cs.perm_columns if c.kind == 2))
    cyc = next(c for c in sigma_cycles(kd) if (inst_col, 2) in c)
    fail, first = mp.check(kd, adv[None], inst[None, :64], np.array([2], np.uint32))
    got = {int(s): (int(first[0, s]), int(fail[0, s])) for s in np.flatnonzero(fail[0])}
    assert got == {2 * C + L + col: (r, 1) for col, r in cyc}        # row 2 of the instance column reads zero


def test_instance_too_large():
    kd, make = cm.standard_plonk(k=6)
    adv, inst, lens = kd.witness_arrays(make(1))
    with pytest.raises(ValueError):
        mp.check(kd, adv[None], np.zeros((1, 64 * 32), np.uint8), np.array([64], np.uint32))
