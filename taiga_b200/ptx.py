"""Host-side mirror of the reference's proving surface for the hot path.

  reference (taiga_halo2)                                       here
  ------------------------------------------------------------  -------------------------------------------
  Proof::create(pk, params, circuit, instance, rng)  proof.rs:25-42      Proof.create(pk, witness, seed)
  Proof::verify(vk, params, instance)                proof.rs:45-54      (oracle verifier in tests / bench only)
  SETUP_PARAMS_MAP / COMPLIANCE_PROVING_KEY          constant.rs:128-152 ProverService (SRS + both proving keys, device resident)
  ShieldedPartialTransaction::build                  shielded_ptx.rs:98-134
      2 x ComplianceVerifyingInfo::create + 4 x get_verifying_info, sequential
                                                                         ProverService.build_ptx_batch: all 2P Compliance proofs
                                                                         in one batched call, all 4P VP proofs in another
  verify_transparently  resource_logic_circuit.rs:597-606      ProverService.check_ptx_batch (MockProver::verify on the GPU)

The circuits are the Taiga-shaped ones of circuits_taiga.py (the real ones need the Rust `synthesize`).  Witness
synthesis happens on the host before the call, exactly as `Circuit::synthesize` does in the reference; it is not part
of the proving hot path and not part of any timed region.
"""
import os
import threading

import numpy as np

from . import circuits_taiga, lib

COMPLIANCE_PER_PTX = 2   # shielded_ptx.rs:107-113
VP_PER_PTX = 4           # taiga_api.rs:256-352 (ptx_example_test: 4 trivial application VPs)


class Proof:
    """`Proof(Vec<u8>)` (proof.rs:21)."""

    def __init__(self, data):
        self.data = bytes(data)

    @classmethod
    def create(cls, pk, advice, instance, instance_len, seed):
        """One proof (the reference's call shape).  pk: lib.ProvingKey."""
        return cls(pk.prove_batch(advice[None], instance[None], instance_len, seed)[0])

    def inner(self):
        return self.data


class ProverService:
    """SRS + Compliance / Resource-Logic proving keys resident on one GPU.

    `c_workers` / `v_workers` independent (context = CUDA stream, proving key) pairs per circuit: the proofs of a batch
    are split among them and proved concurrently, so the latency-bound phases of one proof (transcript, bucket
    reductions, IPA rounds) overlap with the throughput-bound phases of the others.  For large batches one worker per
    circuit is enough (the kernels already fill the GPU)."""

    def __init__(self, device=0, srs_arrays=None, c_workers=2, v_workers=2, serial=False):
        s = srs_arrays
        self.serial = serial   # prove the jobs one after the other on the calling thread (profiling under ncu)
        self.ctx = lib.Context(device)
        self.srs = self.ctx.load_srs(s["k"], s["g"], s["g_lagrange"], s["w"], s["u"])
        self.kd_c, self.make_c = circuits_taiga.build(True)
        self.kd_v, self.make_v = circuits_taiga.build(False)
        self.c_workers = [(self.ctx if i == 0 else lib.Context(device), self.srs.load_circuit(self.kd_c)) for i in range(c_workers)]
        self.v_workers = [(lib.Context(device), self.srs.load_circuit(self.kd_v)) for _ in range(v_workers)]
        self.pk_c, self.pk_v = self.c_workers[0][1], self.v_workers[0][1]
        self.contexts = [w[0] for w in self.c_workers + self.v_workers]

    def synthesize_ptx(self, n_ptx, wseed=0, procs=None, pool=None):
        """Witness tables for n_ptx partial transactions: dict of stacked numpy arrays (host).  The advice tables (60 MiB per ptx)
        are written by the worker processes straight into shared memory; only the small instance vectors travel through pipes.
        `pool`: a SynthPool started before any CUDA work (no fork from a multi-threaded process); default: fork here."""
        if pool is not None:
            return pool.synthesize(n_ptx, wseed)
        nc, nv = COMPLIANCE_PER_PTX * n_ptx, VP_PER_PTX * n_ptx
        jobs = [(True, wseed * 100000 + i, i) for i in range(nc)] + [(False, wseed * 100000 + 50000 + i, i) for i in range(nv)]
        c_adv = _shared_array((nc, self.kd_c.cs.num_advice, self.kd_c.n, 32))
        v_adv = _shared_array((nv, self.kd_v.cs.num_advice, self.kd_v.n, 32))
        res = _synthesize_many(self, jobs, procs, c_adv, v_adv)
        cw, vw = res[:nc], res[nc:]
        return {
            "c_adv": c_adv, "c_inst": np.stack([w[0] for w in cw]), "c_len": cw[0][1],
            "v_adv": v_adv, "v_inst": np.stack([w[0] for w in vw]), "v_len": vw[0][1],
        }

    def build_ptx_batch(self, wit, seed, c_adv=None, v_adv=None, max_batch=64, workers_per_circuit=None):
        """ShieldedPartialTransaction::build for a batch: returns (compliance proofs, vp proofs) as lists of bytes.
        c_adv / v_adv may override the advice buffers (e.g. pinned host or device-resident torch tensors).
        workers_per_circuit limits how many of the service's (stream, key) pairs share the batch (large batches fill
        the GPU from one stream per circuit; single partial transactions want two, to overlap their latency-bound phases)."""
        c_adv = wit["c_adv"] if c_adv is None else c_adv
        v_adv = wit["v_adv"] if v_adv is None else v_adv
        jobs = []   # (result slot, worker, first proof, last proof, ...)
        for kind, workers, adv, inst, lens, index0 in (("c", self.c_workers, c_adv, wit["c_inst"], wit["c_len"], 0),
                                                       ("v", self.v_workers, v_adv, wit["v_inst"], wit["v_len"], 1 << 20)):
            total = len(inst)
            nw = min(len(workers) if not workers_per_circuit else min(len(workers), workers_per_circuit), total)
            for w in range(nw):
                lo, hi = total * w // nw, total * (w + 1) // nw
                jobs.append((kind, lo, hi, workers[w], adv, inst, lens, index0))
        results, errors = {}, []

        def run(job):
            kind, lo, hi, (ctx, pk), adv, inst, lens, index0 = job
            try:
                results[(kind, lo)] = self._prove_range(pk, ctx, adv, inst, lens, seed, max_batch, index0, lo, hi)
            except BaseException as ex:  # re-raised in the caller's thread
                errors.append(ex)
        if self.serial:
            for j in jobs:
                run(j)
        else:
            threads = [threading.Thread(target=run, args=(j,)) for j in jobs[1:]]
            for th in threads:
                th.start()   # ctypes releases the GIL inside tb_prove_batch: every worker enqueues on its own stream
            run(jobs[0])
            for th in threads:
                th.join()
        if errors:
            raise errors[0]
        out = {"c": [], "v": []}
        for (kind, lo) in sorted(results):
            out[kind] += results[(kind, lo)]
        return out["c"], out["v"]

    def check_ptx_batch(self, wit):
        """The batched counterpart of `verify_transparently` (resource_logic_circuit.rs:597-606): MockProver::verify of every
        witness of a synthesized batch.  Returns (compliance CheckReports, vp CheckReports)."""
        return (self.pk_c.check_batch(wit["c_adv"], wit["c_inst"], wit["c_len"]),
                self.pk_v.check_batch(wit["v_adv"], wit["v_inst"], wit["v_len"]))

    @property
    def launch_count(self):
        return sum(c.launch_count for c in self.contexts)

    def prof_enable(self, on=True):
        for c in self.contexts:
            c.prof_enable(on)

    def prof_read(self):
        tot = {}
        for c in self.contexts:
            for k_, v_ in c.prof_read().items():
                a = tot.get(k_, (0.0, 0))
                tot[k_] = (a[0] + v_[0], a[1] + v_[1])
        return tot

    def work_read(self):
        tot = {}
        for c in self.contexts:
            for k_, v_ in c.work_read().items():
                tot[k_] = tot.get(k_, 0.0) + v_
        return tot

    @staticmethod
    def _prove_range(pk, ctx, adv, inst, lens, seed, max_batch, index0, lo, hi):
        kd = pk.keydata
        per = kd.cs.num_advice * kd.n * 32
        total = len(inst)
        out = []
        for s in range(lo, hi, max_batch):
            e = min(hi, s + max_batch)
            if hasattr(adv, "data_ptr"):  # torch tensor (pinned host or device)
                chunk = _TensorSlice(adv, s * per, (e - s) * per)
            else:
                chunk = adv.reshape(total, -1)[s:e]
            out += pk.prove_batch_raw(chunk, e - s, inst[s:e], lens, seed, index0 + s, ctx=ctx)
        return out


_SYNTH = None


def _shared_array(shape):
    """uint8 array in anonymous shared memory (inherited by forked workers; unlinked at once, freed with the last mapping)."""
    from multiprocessing import shared_memory
    size = int(np.prod(shape))
    shm = shared_memory.SharedMemory(create=True, size=max(1, size))
    arr = np.ndarray(shape, dtype=np.uint8, buffer=shm.buf)
    try:
        shm.unlink()
    except Exception:
        pass
    _KEEP.append(shm)   # the mapping must outlive the array
    return arr


_KEEP = []


def _synth_one(job):
    comp, seed, slot = job
    svc, c_adv, v_adv = _SYNTH
    kd, make, out = (svc.kd_c, svc.make_c, c_adv) if comp else (svc.kd_v, svc.make_v, v_adv)
    adv, inst, lens = kd.witness_arrays(make(seed))
    out[slot] = adv
    return inst, lens


def _synthesize_many(svc, jobs, procs, c_adv, v_adv):
    """Host witness synthesis (the stand-in for the Rust `Circuit::synthesize`, compliance_circuit.rs:174-327) of many
    proofs: forked worker processes, one witness per task."""
    global _SYNTH
    import multiprocessing as mp
    import os
    procs = procs or min(len(jobs), max(1, (os.cpu_count() or 2) - 2), 64)
    _SYNTH = (svc, c_adv, v_adv)
    try:
        if procs <= 1 or len(jobs) <= 6:
            return [_synth_one(j) for j in jobs]
        with mp.get_context("fork").Pool(procs) as pool:
            return pool.map(_synth_one, jobs, chunksize=max(1, len(jobs) // (4 * procs)))
    finally:
        _SYNTH = None


# ---- persistent pool of synthesis workers (started before CUDA is initialised; the workers build the circuits themselves)
_W = {}


def _pool_init():
    _W["c"] = circuits_taiga.build(True)
    _W["v"] = circuits_taiga.build(False)


def _pool_job(job):
    comp, seed, slot, name, shape = job
    import mmap
    kd, make = _W["c" if comp else "v"]
    adv, inst, lens = kd.witness_arrays(make(seed))
    key = "map_c" if comp else "map_v"
    m = _W.get(key)
    if m is None or m[0] != name:   # map the batch's segment once per worker (plain mmap: no resource-tracker traffic)
        if m is not None:
            del _W[key]
            m = None
        fd = os.open("/dev/shm/" + name.lstrip("/"), os.O_RDWR)
        try:
            mm = mmap.mmap(fd, int(np.prod(shape)))
        finally:
            os.close(fd)
        m = _W[key] = (name, np.frombuffer(mm, dtype=np.uint8).reshape(shape), mm)
    m[1][slot] = adv
    return inst, lens


class SynthPool:
    """Worker processes for host witness synthesis (stand-in for the Rust `Circuit::synthesize`).  Create it BEFORE torch / CUDA
    are touched: the workers are forked once from a single-threaded parent and live for the whole run."""

    def __init__(self, procs=None):
        import multiprocessing as mp
        import os
        self.procs = procs or min(64, max(1, (os.cpu_count() or 2) - 2))
        self.pool = mp.get_context("fork").Pool(self.procs, initializer=_pool_init)

    def synthesize(self, n_ptx, wseed=0):
        from multiprocessing import shared_memory
        nc, nv = COMPLIANCE_PER_PTX * n_ptx, VP_PER_PTX * n_ptx
        n15 = 1 << 15
        shapes = {True: (nc, 10, n15, 32), False: (nv, 10, n15, 32)}
        shms = {c: shared_memory.SharedMemory(create=True, size=int(np.prod(sh))) for c, sh in shapes.items()}
        try:
            jobs = [(True, wseed * 100000 + i, i, shms[True].name, shapes[True]) for i in range(nc)] + \
                   [(False, wseed * 100000 + 50000 + i, i, shms[False].name, shapes[False]) for i in range(nv)]
            res = self.pool.map(_pool_job, jobs, chunksize=max(1, len(jobs) // (4 * self.procs)))
        finally:
            for sh in shms.values():
                try:
                    sh.unlink()
                except Exception:
                    pass
        c_adv = np.ndarray(shapes[True], dtype=np.uint8, buffer=shms[True].buf)
        v_adv = np.ndarray(shapes[False], dtype=np.uint8, buffer=shms[False].buf)
        cw, vw = res[:nc], res[nc:]
        return {"c_adv": c_adv, "c_inst": np.stack([w[0] for w in cw]), "c_len": cw[0][1],
                "v_adv": v_adv, "v_inst": np.stack([w[0] for w in vw]), "v_len": vw[0][1],
                "_shm": list(shms.values())}   # the (already unlinked) segments live exactly as long as this dictionary

    def close(self):
        self.pool.terminate()


class _TensorSlice:
    """A byte range of a torch uint8 tensor, passed to the C ABI by address (host-pinned or device memory)."""

    def __init__(self, t, offset, nbytes):
        self.t, self.offset, self.nbytes = t, offset, nbytes

    def data_ptr(self):
        return self.t.data_ptr() + self.offset
