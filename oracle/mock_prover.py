"""Pure-Python restatement of halo2 `dev::MockProver::verify` (halo2_proofs 0.3 lineage, dev.rs) for the data-driven
tb_cs_desc: the test reference of tb_check_batch.  Shares no code with the device path.

  n = 2^k, usable = n - blinding_factors - 1, rotations wrap modulo n.
  Fixed cells hold the key's values; instance cells the given values, then zeros; advice cells in rows < usable the
  given values, advice cells in rows >= usable are POISON (the prover overwrites them with blinding scalars).
  Poison follows dev::Value: negation, addition and scaling propagate it; a product is a real zero when either factor
  is a real zero, else poison when a factor is poison.
  gates    every constraint at every row: slot j if real and non-zero, slot C + j if poison;
  lookups  rows < usable: the input tuple must equal, element for element, a table tuple of a row < usable that holds
           no poison (exact membership); a poisoned input fails;
  copies   sigma decoded back to cells (sigma[c][r] = DELTA^c' * omega^r'); for rows r < usable, fails when
           value(p, r) != value(sigma(p, r)) or either is poison.

Evaluation is vectorised over rows: one object-array operation per expression node, with a poison mask beside it.
"""
import numpy as np

from taiga_b200.circuit import (ADVICE, DELTA, EX_ADD, EX_ADVICE, EX_CONST, EX_FIXED, EX_INSTANCE, EX_MUL, EX_NEG,
                                EX_SCALE, FIXED, P, ROOT)

NO_ROW = 0xFFFFFFFF


def to_ints(a):
    """[..., 32] little-endian bytes -> object array of Python ints of shape [...]."""
    a = np.ascontiguousarray(a, dtype=np.uint8)
    w = a.reshape(-1, 32).view("<u8")
    out = w[:, 0].astype(object)
    for i in range(1, 4):
        out = out + (w[:, i].astype(object) << (64 * i))
    return out.reshape(a.shape[:-1])


def decode_sigma(kd):
    """(column index, row) arrays [P, n]: the cell each sigma value names.  Raises ValueError for a value naming no cell."""
    n, m = kd.n, len(kd.cs.perm_columns)
    omega = pow(ROOT, 1 << (32 - kd.k), P)
    cell = {}
    d = 1
    for c in range(m):
        v = d
        for r in range(n):
            cell[v] = (c, r)
            v = v * omega % P
        d = d * DELTA % P
    sig = to_ints(kd.sigma.reshape(m, n, 32)) if m else np.zeros((0, n), object)
    to_c = np.zeros((m, n), np.int64)
    to_r = np.zeros((m, n), np.int64)
    for c in range(m):
        for r in range(n):
            hit = cell.get(sig[c, r])
            if hit is None:
                raise ValueError("malformed key: sigma[%d][%d] names no cell" % (c, r))
            to_c[c, r], to_r[c, r] = hit
    return to_c, to_r


def _children(op, a, b):
    return [a] if op in (EX_NEG, EX_SCALE) else sorted({a, b}) if op in (EX_ADD, EX_MUL) else []


class _Eval:
    """Values and poison masks of the expression nodes over all n rows, freed after their last use."""

    def __init__(self, kd, adv, inst, fixed, usable):
        self.cs, self.n = kd.cs, kd.n
        self.cols = {ADVICE: adv, FIXED: fixed}
        self.inst = inst
        self.adv_poison = np.arange(self.n) >= usable

    def leaf(self, kind, q):
        col, rot = q
        if kind == EX_ADVICE:
            return np.roll(self.cols[ADVICE][col], -rot), np.roll(self.adv_poison, -rot)
        src = self.cols[FIXED][col] if kind == EX_FIXED else self.inst[col]
        return np.roll(src, -rot), np.zeros(self.n, bool)

    def run(self, roots, on_root):
        """Evaluates every node reachable from `roots` (dict node -> list of tags) in topological order and calls
        on_root(tag, values, poison) for each tag of each root."""
        cs = self.cs
        need, stack = set(), list(roots)
        while stack:
            i = stack.pop()
            if i in need:
                continue
            need.add(i)
            op, a, b = cs.nodes[i]
            stack += _children(op, a, b)
        last = {}
        for i in sorted(need):
            op, a, b = cs.nodes[i]
            for c in _children(op, a, b):
                last[c] = i
        val = {}
        queries = {EX_ADVICE: cs.advice_queries, EX_FIXED: cs.fixed_queries, EX_INSTANCE: cs.instance_queries}
        for i in sorted(need):
            op, a, b = cs.nodes[i]
            if op == EX_CONST:
                v, p = np.full(self.n, cs.constants[a], dtype=object), np.zeros(self.n, bool)
            elif op in queries:
                v, p = self.leaf(op, queries[op][a])
            elif op == EX_NEG:
                v, p = (P - val[a][0]) % P, val[a][1]
            elif op == EX_SCALE:
                v, p = val[a][0] * cs.constants[b] % P, val[a][1]
            elif op == EX_ADD:
                v, p = (val[a][0] + val[b][0]) % P, val[a][1] | val[b][1]
            else:
                (va, pa), (vb, pb) = val[a], val[b]
                v = va * vb % P
                p = (pa | pb) & ~(~pa & (va == 0)) & ~(~pb & (vb == 0))
            val[i] = (v, p)
            for tag in roots.get(i, ()):
                on_root(tag, v, p)
            for c in _children(op, a, b):
                if last[c] == i:
                    del val[c]
            if i not in last:
                del val[i]


def check(kd, advice, instance, instance_len):
    """MockProver::verify of B witnesses: (fail_rows, first_row), uint32 [B, 2C + L + P], the layout of tb_check_batch."""
    cs, n = kd.cs, kd.n
    usable = n - kd.blinding_factors - 1
    advice = np.asarray(advice, np.uint8).reshape(-1, cs.num_advice, n, 32)
    B = advice.shape[0]
    lens = [int(x) for x in np.asarray(instance_len).reshape(-1)[:cs.num_instance]]
    if any(x > usable for x in lens):
        raise ValueError("InstanceTooLarge")
    instance = np.asarray(instance, np.uint8).reshape(B, -1)
    roots = [p.node for _, polys in cs.gates for p in polys]
    C, L, Pn = len(roots), len(cs.lookups), len(cs.perm_columns)
    S = 2 * C + L + Pn
    fail = np.zeros((B, S), np.uint32)
    first = np.full((B, S), NO_ROW, np.uint32)
    fixed = to_ints(kd.fixed) if cs.num_fixed else np.zeros((0, n), object)
    to_c, to_r = decode_sigma(kd)
    rows = np.arange(n)

    def record(b, slot, bad):
        idx = np.flatnonzero(bad)
        if len(idx):
            fail[b, slot] = len(idx)
            first[b, slot] = int(rows[idx[0]])

    for b in range(B):
        adv = to_ints(advice[b])
        inst = np.zeros((cs.num_instance, n), object)
        off = 0
        for c, ln in enumerate(lens):
            if ln:
                inst[c, :ln] = to_ints(instance[b, 32 * off:32 * (off + ln)].reshape(ln, 32))
            off += ln
        targets = {}
        for j, r in enumerate(roots):
            targets.setdefault(r, []).append(("gate", j))
        for l, pairs in enumerate(cs.lookups):
            for e, (i_, t_) in enumerate(pairs):
                targets.setdefault(i_.node, []).append(("in", l, e))
                targets.setdefault(t_.node, []).append(("tab", l, e))
        tuples = {}

        def on_root(tag, v, p):
            if tag[0] == "gate":
                record(b, tag[1], ~p & (v != 0))
                record(b, C + tag[1], p)
            else:
                tuples[tag] = (v[:usable], p[:usable])
        _Eval(kd, adv, inst, fixed, usable).run(targets, on_root)
        for l, pairs in enumerate(cs.lookups):
            m = len(pairs)
            tin = [tuples[("in", l, e)] for e in range(m)]
            ttab = [tuples[("tab", l, e)] for e in range(m)]
            tab_pois = np.logical_or.reduce([p for _, p in ttab])
            table = set(t for t, bad in zip(zip(*[v for v, _ in ttab]), tab_pois) if not bad)
            in_pois = np.logical_or.reduce([p for _, p in tin])
            missing = np.array([t not in table for t in zip(*[v for v, _ in tin])], bool)
            record(b, 2 * C + l, in_pois | missing)
        if Pn:
            vals = np.empty((Pn, n), object)
            pois = np.zeros((Pn, n), bool)
            for i, col in enumerate(cs.perm_columns):
                vals[i] = adv[col.index] if col.kind == ADVICE else fixed[col.index] if col.kind == FIXED else inst[col.index]
                pois[i] = (rows >= usable) if col.kind == ADVICE else False
            for i in range(Pn):
                tc, tr = to_c[i, :usable], to_r[i, :usable]
                bad = pois[i, :usable] | pois[tc, tr] | (vals[i, :usable] != vals[tc, tr])
                record(b, 2 * C + L + i, bad)
    return fail, first
