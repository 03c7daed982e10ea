"""ctypes binding of libtaiga_b200.so (C ABI declared in include/taiga_b200.h).

The product path has no CPU fallback: if the CUDA library is missing or no sm_100 device is usable this
module raises instead of computing anything on the host.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtaiga_b200.so")

TB_FP, TB_FQ = 0, 1
TB_VESTA, TB_PALLAS = 0, 1
TB_OK, TB_ERR_INVALID, TB_ERR_CUDA, TB_ERR_CONSTRAINT, TB_ERR_INTERNAL = 0, 1, 2, 3, 4


class TaigaB200Error(RuntimeError):
    def __init__(self, status, msg):
        super().__init__("libtaiga_b200 status %d: %s" % (status, msg))
        self.status = status


class ConstraintSystemFailure(TaigaB200Error):
    """Mirror of halo2 `plonk::Error::ConstraintSystemFailure` (the witness does not satisfy the circuit)."""


_lib = None
_vp, _sz, _u32, _i, _u64 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_int, ctypes.c_uint64

_SIGS = {
    "tb_ctx_create": (_i, [_i, ctypes.POINTER(_vp)]),
    "tb_ctx_destroy": (None, [_vp]),
    "tb_last_error": (ctypes.c_char_p, [_vp]),
    "tb_version": (ctypes.c_char_p, []),
    "tb_ctx_sync": (_i, [_vp]),
    "tb_ctx_stream": (_u64, [_vp]),
    "tb_ctx_launch_count": (_u64, [_vp]),
    "tb_prof_categories": (_i, []),
    "tb_prof_category_name": (ctypes.c_char_p, [_i]),
    "tb_prof_enable": (_i, [_vp, _i]),
    "tb_prof_read": (_i, [_vp, _vp, _vp]),
    "tb_prof_work": (_i, [_vp, _vp]),
    "tb_ntt": (_i, [_vp, _i, _u32, _i, _i, _u32, _vp, _vp]),
    "tb_msm": (_i, [_vp, _i, _sz, _u32, _vp, _vp, _u32, _vp]),
    "tb_dev_to_mont": (_i, [_vp, _i, _vp, _sz]),
    "tb_dev_from_mont": (_i, [_vp, _i, _vp, _sz]),
    "tb_dev_ntt": (_i, [_vp, _i, _u32, _i, _i, _u32, _vp, _vp, _vp]),
    "tb_dev_msm": (_i, [_vp, _i, _sz, _u32, _vp, _vp, _u32, _vp]),
    "tb_srs_load": (_i, [_vp, _u32, _vp, _vp, _vp, _vp, ctypes.POINTER(_vp)]),
    "tb_srs_free": (None, [_vp]),
    "tb_srs_commit": (_i, [_vp, _vp, _i, _u32, _vp, _vp, _vp]),
    "tb_circuit_load": (_i, [_vp, _vp, _vp, _vp, _vp, ctypes.POINTER(_vp)]),
    "tb_pk_free": (None, [_vp]),
    "tb_pk_proof_len": (_sz, [_vp]),
    "tb_pk_commitments": (_i, [_vp, _vp, _vp, _vp]),
    "tb_prove_batch": (_i, [_vp, _vp, _u32, _vp, _vp, _vp, _vp, _u32, _vp, _sz]),
    "tb_verify_batch": (_i, [_vp, _vp, _u32, _vp, _vp, _vp, _sz, _sz, _vp]),
    "tb_pk_check_slots": (_sz, [_vp]),
    "tb_check_batch": (_i, [_vp, _vp, _u32, _vp, _vp, _vp, _vp, _vp]),
}


class CheckReport:
    """Constraint-check result of one witness (halo2 `MockProver::verify`).  `fail_rows` / `first_row` are the witness's
    tb_check_batch slots; `failures` lists (kind, index, first_row, rows) with kind "gate" (constraint unsatisfied),
    "poisoned" (constraint reads a blinding-row advice cell), "lookup" or "copy" (permutation column index)."""

    def __init__(self, fail_rows, first_row, num_constraints, num_lookups):
        self.fail_rows, self.first_row = fail_rows, first_row
        C, L = num_constraints, num_lookups
        self.failures = []
        for s in np.flatnonzero(fail_rows):
            s = int(s)
            kind, idx = ("gate", s) if s < C else ("poisoned", s - C) if s < 2 * C else ("lookup", s - 2 * C) if s < 2 * C + L else ("copy", s - 2 * C - L)
            self.failures.append((kind, idx, int(first_row[s]), int(fail_rows[s])))
        self.ok = not self.failures

    def describe(self, keydata):
        """One line per failure, named as MockProver names it: gate name and polynomial index, lookup index, permutation column."""
        cs = keydata.cs
        polys = [(name, i) for name, ps in cs.gates for i in range(len(ps))]
        out = []
        for kind, idx, row, rows in self.failures:
            if kind in ("gate", "poisoned"):
                name, i = polys[idx]
                what = "constraint %d of gate %r %s" % (i, name, "not satisfied" if kind == "gate" else "reads a poisoned cell")
            elif kind == "lookup":
                what = "lookup %d input not in its table" % idx
            else:
                what = "copy constraint on column %r broken" % cs.perm_columns[idx]
            out.append("%s: first at row %d (%d rows)" % (what, row, rows))
        return out

    def __repr__(self):
        return "CheckReport(ok=%s, failures=%r)" % (self.ok, self.failures)


def exported_symbols():
    """Every symbol include/taiga_b200.h declares (checked by the CPU test-suite)."""
    return sorted(_SIGS)


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("libtaiga_b200.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                              "there is no CPU fallback for the prover path")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        assert a.flags["C_CONTIGUOUS"]
        return a.ctypes.data_as(_vp)
    if hasattr(a, "data_ptr"):  # torch tensor
        return _vp(a.data_ptr())
    return _vp(int(a))


def _u8(a):
    return np.ascontiguousarray(a, dtype=np.uint8)


class Context:
    """One GPU, one stream (tb_ctx)."""

    def __init__(self, device=0):
        self._lib = load()
        h = _vp()
        st = self._lib.tb_ctx_create(int(device), ctypes.byref(h))
        if st != TB_OK:
            raise TaigaB200Error(st, "tb_ctx_create failed: no usable sm_100 CUDA device (no CPU fallback exists)")
        self._h = h
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            self._lib.tb_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st):
        if st != TB_OK:
            msg = self._lib.tb_last_error(self._h).decode(errors="replace")
            raise (ConstraintSystemFailure if st == TB_ERR_CONSTRAINT else TaigaB200Error)(st, msg)

    @property
    def stream(self):
        return int(self._lib.tb_ctx_stream(self._h))

    @property
    def launch_count(self):
        return int(self._lib.tb_ctx_launch_count(self._h))

    def sync(self):
        self._check(self._lib.tb_ctx_sync(self._h))

    def prof_enable(self, on=True):
        self._check(self._lib.tb_prof_enable(self._h, int(on)))

    def prof_read(self):
        """{category: (milliseconds, kernel groups)} since the last read, measured with CUDA events on the context's stream."""
        n = self._lib.tb_prof_categories()
        ms = np.zeros(n, np.float64)
        cnt = np.zeros(n, np.uint64)
        self._check(self._lib.tb_prof_read(self._h, _ptr(ms), _ptr(cnt)))
        return {self._lib.tb_prof_category_name(i).decode(): (float(ms[i]), int(cnt[i])) for i in range(n)}

    def work_read(self):
        """{category: Montgomery multiplications executed since the last read} (the numerator of the integer-pipe roofline)."""
        n = self._lib.tb_prof_categories()
        mm = np.zeros(n, np.float64)
        self._check(self._lib.tb_prof_work(self._h, _ptr(mm)))
        return {self._lib.tb_prof_category_name(i).decode(): float(mm[i]) for i in range(n)}

    # ---- host-buffer primitives
    def ntt(self, field, data, inverse=False, coset=False, batch=1):
        d = _u8(data)
        n = d.size // 32 // batch
        logn = n.bit_length() - 1
        assert (1 << logn) == n and d.size == batch * n * 32
        out = np.empty_like(d)
        self._check(self._lib.tb_ntt(self._h, field, logn, int(inverse), int(coset), batch, _ptr(d), _ptr(out)))
        return out.reshape(batch * n, 32) if batch > 1 else out.reshape(n, 32)

    def msm(self, curve, scalars, points, batch=1, window_bits=0):
        s, p = _u8(scalars), _u8(points)
        n = p.size // 64
        assert s.size == batch * n * 32
        out = np.zeros((batch, 64), np.uint8)
        self._check(self._lib.tb_msm(self._h, curve, n, batch, _ptr(s), _ptr(p), window_bits, _ptr(out)))
        return out

    # ---- device-buffer primitives (torch tensors / raw device pointers)
    def dev_to_mont(self, field, t, n):
        self._check(self._lib.tb_dev_to_mont(self._h, field, _ptr(t), n))

    def dev_from_mont(self, field, t, n):
        self._check(self._lib.tb_dev_from_mont(self._h, field, _ptr(t), n))

    def dev_ntt(self, field, logn, d_in, d_out, d_scratch, inverse=False, coset=False, batch=1):
        self._check(self._lib.tb_dev_ntt(self._h, field, logn, int(inverse), int(coset), batch, _ptr(d_in), _ptr(d_out), _ptr(d_scratch)))

    def dev_msm(self, curve, n, d_scalars, d_points, d_out, batch=1, window_bits=0):
        self._check(self._lib.tb_dev_msm(self._h, curve, n, batch, _ptr(d_scalars), _ptr(d_points), window_bits, _ptr(d_out)))

    def load_srs(self, k, g, g_lagrange, w, u):
        return Srs(self, k, g, g_lagrange, w, u)


class Srs:
    """Device-resident Params<vesta::Affine> (constant.rs:128-139) with fixed-base tables."""

    def __init__(self, ctx, k, g, g_lagrange, w, u):
        self.ctx, self.k, self.n = ctx, k, 1 << k
        g, gl, w, u = _u8(g), _u8(g_lagrange), _u8(w), _u8(u)
        assert g.size == 64 * self.n and gl.size == 64 * self.n and w.size == 64 and u.size == 64
        h = _vp()
        ctx._check(ctx._lib.tb_srs_load(ctx._h, k, _ptr(g), _ptr(gl), _ptr(w), _ptr(u), ctypes.byref(h)))
        self._h = h

    def commit(self, scalars, blinds=None, lagrange=False, batch=1):
        """Params::commit / commit_lagrange: MSM(scalars, g | g_lagrange) + blind * w, per batch item."""
        s = _u8(scalars)
        assert s.size == batch * self.n * 32
        b = _u8(blinds) if blinds is not None else None
        out = np.zeros((batch, 64), np.uint8)
        self.ctx._check(self.ctx._lib.tb_srs_commit(self.ctx._h, self._h, int(lagrange), batch, _ptr(s), _ptr(b), _ptr(out)))
        return out

    def load_circuit(self, keydata):
        return ProvingKey(self, keydata)

    def close(self):
        if getattr(self, "_h", None):
            self.ctx._lib.tb_srs_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ProvingKey:
    """Device-resident proving key of one circuit (tb_pk): the stand-in for halo2's ProvingKey<vesta::Affine>
    (COMPLIANCE_PROVING_KEY / TRIVIAL_RESOURCE_LOGIC_PK, constant.rs:145-152, resource_logic_examples.rs:50-61).
    `keydata` is a taiga_b200.circuit.CircuitKeyData (descriptor + fixed columns + sigma)."""

    def __init__(self, srs, keydata):
        self.srs, self.ctx, self.keydata = srs, srs.ctx, keydata
        self._fixed, self._sigma = _u8(keydata.fixed), _u8(keydata.sigma)
        h = _vp()
        self.ctx._check(self.ctx._lib.tb_circuit_load(self.ctx._h, srs._h, ctypes.byref(keydata.desc), _ptr(self._fixed), _ptr(self._sigma), ctypes.byref(h)))
        self._h = h
        self.proof_len = int(self.ctx._lib.tb_pk_proof_len(h))

    def commitments(self):
        """keygen_vk: (fixed column commitments [num_fixed, 64], sigma commitments [P, 64])."""
        kd = self.keydata
        f = np.zeros((max(1, kd.cs.num_fixed), 64), np.uint8)
        s = np.zeros((max(1, len(kd.cs.perm_columns)), 64), np.uint8)
        self.ctx._check(self.ctx._lib.tb_pk_commitments(self.ctx._h, self._h, _ptr(f), _ptr(s)))
        return f[: kd.cs.num_fixed], s[: len(kd.cs.perm_columns)]

    def prove_batch(self, advice, instance, instance_len, seed, first_proof_index=0):
        """Proof::create for a batch: advice uint8 [B, num_advice, n, 32]; instance uint8 [B, sum(instance_len), 32].
        Returns a list of B proof byte strings."""
        adv = _u8(advice)
        kd = self.keydata
        per = kd.cs.num_advice * kd.n * 32
        assert adv.size % per == 0
        return self.prove_batch_raw(adv, adv.size // per, instance, instance_len, seed, first_proof_index)

    def prove_batch_raw(self, advice, B, instance, instance_len, seed, first_proof_index=0, ctx=None):
        """Same, with `advice` given as anything exposing its address (numpy array, pinned-host or DEVICE torch tensor).
        `ctx`: run on another Context (= another CUDA stream) of the same device, e.g. to overlap two circuits."""
        ctx = ctx or self.ctx
        inst = _u8(instance)
        lens = np.ascontiguousarray(instance_len, dtype=np.uint32)
        assert inst.size >= B * int(lens.sum()) * 32
        seed = _u8(np.frombuffer(bytes(seed), np.uint8))
        assert seed.size == 32
        out = np.zeros((B, self.proof_len), np.uint8)
        ctx._check(ctx._lib.tb_prove_batch(ctx._h, self._h, B, _ptr(advice), _ptr(inst), _ptr(lens), _ptr(seed), first_proof_index,
                                           _ptr(out), self.proof_len))
        return [out[b].tobytes() for b in range(B)]

    def verify_batch(self, instance, instance_len, proofs, ctx=None):
        """Proof::verify for a batch: proofs = list of byte strings; returns a list of booleans."""
        ctx = ctx or self.ctx
        B = len(proofs)
        plen = len(proofs[0])
        assert all(len(p) == plen for p in proofs)
        buf = np.frombuffer(b"".join(proofs), np.uint8).copy()
        inst = _u8(instance)
        lens = np.ascontiguousarray(instance_len, dtype=np.uint32)
        ok = np.zeros(B, np.uint8)
        ctx._check(ctx._lib.tb_verify_batch(ctx._h, self._h, B, _ptr(inst), _ptr(lens), _ptr(buf), plen, plen, _ptr(ok)))
        return [bool(v) for v in ok]

    def check_batch(self, advice, instance, instance_len, ctx=None):
        """MockProver::verify for a batch: advice uint8 [B, num_advice, n, 32]; instance uint8 [B, sum(instance_len), 32].
        Returns one CheckReport per witness."""
        adv = _u8(advice)
        kd = self.keydata
        per = kd.cs.num_advice * kd.n * 32
        assert adv.size % per == 0
        return self.check_batch_raw(adv, adv.size // per, instance, instance_len, ctx=ctx)

    def check_batch_raw(self, advice, B, instance, instance_len, ctx=None):
        """Same, with `advice` given as anything exposing its address (numpy array, pinned-host or DEVICE torch tensor)."""
        ctx = ctx or self.ctx
        inst = _u8(instance)
        lens = np.ascontiguousarray(instance_len, dtype=np.uint32)
        assert inst.size >= B * int(lens.sum()) * 32
        S = int(ctx._lib.tb_pk_check_slots(self._h))
        fail = np.zeros((B, max(1, S)), np.uint32)
        first = np.zeros((B, max(1, S)), np.uint32)
        ctx._check(ctx._lib.tb_check_batch(ctx._h, self._h, B, _ptr(advice), _ptr(inst), _ptr(lens), _ptr(fail), _ptr(first)))
        cs = self.keydata.cs
        C = sum(len(ps) for _, ps in cs.gates)
        return [CheckReport(fail[b, :S], first[b, :S], C, len(cs.lookups)) for b in range(B)]

    def close(self):
        if getattr(self, "_h", None):
            self.ctx._lib.tb_pk_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
