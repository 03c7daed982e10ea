#!/usr/bin/env python
"""Prints one JSON line: the device constraint check (tb_check_batch, halo2 MockProver::verify) of 64 partial
transactions' worth of witnesses, 128 Compliance-shaped and 256 Resource-Logic-shaped (k = 15), on one GPU.

  ms_per_batch   host clock around whole batches (both circuits) ending in tb_ctx_sync, after one warm-up batch, repeated
                 for at least a second: advice device-resident, and advice read from pinned host memory.
  modmul         Montgomery products per batch counted from the expression DAG: MUL / SCALE nodes reachable from the
                 gate roots x n rows + from the lookup input roots x usable rows, x witnesses (the fixed-column lookup
                 tables are evaluated once per key, not per batch).  int_util uses bench.py's constants.
  python_restatement_s_per_witness   oracle/mock_prover.py on one witness of each shape on this host's CPU: the
                 test reference, not a baseline for the Rust MockProver.
The check does the same work whether or not a witness is satisfying, so a few distinct satisfying witnesses are
synthesized and repeated to fill the batch.
"""
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (SRS fixture loader and the integer-pipe constants)
from oracle import mock_prover  # noqa: E402
from taiga_b200 import circuits_taiga, lib  # noqa: E402
from taiga_b200.circuit import EX_ADD, EX_MUL, EX_NEG, EX_SCALE  # noqa: E402

PTX, C_PER_PTX, V_PER_PTX, DISTINCT = 64, 2, 4, 4


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, mhz = [x.strip() for x in q.split(",")]
    return name, float(power), float(mhz)


def products(kd):
    """Montgomery products the check of one witness executes, from the DAG."""
    cs = kd.cs

    def muls(roots):
        seen, stack = set(), list(roots)
        while stack:
            i = stack.pop()
            if i not in seen:
                seen.add(i)
                op, a, b = cs.nodes[i]
                stack += [a] if op in (EX_NEG, EX_SCALE) else [a, b] if op in (EX_ADD, EX_MUL) else []
        return sum(1 for i in seen if cs.nodes[i][0] in (EX_MUL, EX_SCALE))
    usable = kd.n - kd.blinding_factors - 1
    return muls([p.node for _, ps in cs.gates for p in ps]) * kd.n + muls([i.node for lk in cs.lookups for i, _ in lk]) * usable


def main():
    import torch
    name, power, mhz = card()
    s = bench.load_srs()
    ctx = lib.Context(0)
    srs = ctx.load_srs(s["k"], s["g"], s["g_lagrange"], s["w"], s["u"])
    jobs, restate = [], {}
    for comp, count in ((True, C_PER_PTX * PTX), (False, V_PER_PTX * PTX)):
        kd, make = circuits_taiga.build(comp)
        pk = srs.load_circuit(kd)
        wit = [kd.witness_arrays(make(10 + i)) for i in range(DISTINCT)]
        adv = np.stack([wit[i % DISTINCT][0] for i in range(count)])
        inst = np.stack([wit[i % DISTINCT][1] for i in range(count)])
        t = time.perf_counter()
        f, _ = mock_prover.check(kd, wit[0][0][None], wit[0][1][None], wit[0][2])
        restate["compliance" if comp else "vp"] = round(time.perf_counter() - t, 2)
        assert not f.any()
        S = int(ctx._lib.tb_pk_check_slots(pk._h))
        jobs.append(dict(kd=kd, pk=pk, B=count, lens=np.ascontiguousarray(wit[0][2], np.uint32), inst=np.ascontiguousarray(inst),
                         dev=torch.from_numpy(adv).cuda(), pinned=torch.from_numpy(adv).pin_memory(),
                         fail=np.zeros((count, S), np.uint32), first=np.zeros((count, S), np.uint32)))
        del adv
    vp = ctypes.c_void_p

    def batch(where):
        for j in jobs:
            ctx._check(ctx._lib.tb_check_batch(ctx._h, j["pk"]._h, j["B"], vp(j[where].data_ptr()), j["inst"].ctypes.data_as(vp),
                                               j["lens"].ctypes.data_as(vp), j["fail"].ctypes.data_as(vp), j["first"].ctypes.data_as(vp)))
        ctx.sync()

    out = {}
    for where in ("dev", "pinned"):
        batch(where)   # warm-up: key set-up, module load
        assert all(not j["fail"].any() for j in jobs), "a satisfying witness was reported"
        reps, t0 = 0, time.perf_counter()
        while True:
            batch(where)
            reps += 1
            el = time.perf_counter() - t0
            if el >= 1.0 and reps >= 3:
                break
        out[where] = el / reps * 1e3
    witnesses = sum(j["B"] for j in jobs)
    mm = float(sum(products(j["kd"]) * j["B"] for j in jobs))
    int_peak = 148 * bench.INT_LANES_PER_SM * mhz * 1e6
    print(json.dumps({
        "metric": "constraint_check_batch", "gpu": name, "power_limit_w": power, "clocks_max_sm_mhz": mhz,
        "batch": {"ptx": PTX, "compliance_witnesses": C_PER_PTX * PTX, "vp_witnesses": V_PER_PTX * PTX, "k": 15},
        "ms_per_batch": {"advice_device": round(out["dev"], 2), "advice_pinned_host": round(out["pinned"], 2)},
        "witnesses_per_s": {"advice_device": round(witnesses / out["dev"] * 1e3, 1), "advice_pinned_host": round(witnesses / out["pinned"] * 1e3, 1)},
        "ptx_per_s": {"advice_device": round(PTX / out["dev"] * 1e3, 1), "advice_pinned_host": round(PTX / out["pinned"] * 1e3, 1)},
        "modmul_per_batch": mm,
        "int_util_advice_device": round(mm * bench.SASS_PER_MODMUL / (out["dev"] * 1e-3) / int_peak, 4),
        "python_restatement_s_per_witness": restate,
        "launches": ctx.launch_count}))
    ctx.close()


if __name__ == "__main__":
    main()
