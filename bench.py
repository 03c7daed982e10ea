#!/usr/bin/env python
"""bench.py - partial-transaction proofs/sec of the B200-native Taiga prover hot path.

Contract (driver): `python bench.py --gpus N --steps K --warmup W [--impl reference]`; for N > 1 it is launched under
torch.distributed.run, one rank per GPU.  Rank 0 prints ONE JSON line.

  step      one pass of the hot path over one batch: `--ptx P` shielded partial transactions per GPU, default 64
            (BASELINE.json configs[2]; 128 per GPU at 8 GPUs = the 1024 ptx of configs[4]).  One ptx = 2 Compliance
            ("Action")-shaped + 4 Resource-Logic ("VP")-shaped Halo2/IPA proofs, k = 15, Taiga's own SRS, i.e.
            ShieldedPartialTransaction::build (shielded_ptx.rs:98-134).  All proofs of a circuit go through
            tb_prove_batch in chunks of 64: MSMs, NTTs and the gate evaluation are batched across proofs.
  value     whole-job ptx/s with the advice tables already resident in HBM when the timed region starts
            (wall clock between device synchronisations around the K steps, max over ranks; CUDA-event time beside it).
  e2e       the same metric through the C ABI with HOST (pinned) advice buffers: host->device copies of the advice
            tables and the device->host read of the proof bytes are inside the timed region.
  latency   configs[1]: ONE partial transaction per step (two streams per circuit), the latency-bound secondary figure.
  roofline  dominant kernel group of a profiled step (CUDA events on the library's streams).  `achieved` = SURVEY 8d
            algorithmic bytes / time against the measured HBM peak (MEASURED_PEAKS.json) because the metric asks for
            it; the binding resource is the INTEGER pipe (tools/modmul_bench.cu: 0.5 integer instructions per cycle per
            SM sub-partition), so `int_util` = executed 255-bit Montgomery multiplications x 247 SASS instructions /
            (time x 148 SMs x 64 lanes x clock) is reported for every group as well.  `traffic` is read from the
            committed ncu capture (profiles/r02_ncu_traffic.json), not hard-coded.
  sweeps    BASELINE configs[3]: Vesta AND Pallas MSM 2^16..2^22 (uniform and witness-like scalars), Fp NTT 2^17..2^23.
  cpu_baseline   the CPU oracle (threaded C++ restatement of the halo2 prover; the Rust reference cannot be built in
            this image) timed on this box's host cores on a bounded sample (1 Compliance + 1 VP proof -> ptx/s).
  --impl reference   times that CPU arm alone, same metric / config (see DESIGN.md "Reference arm").
  --dump-outputs DIR   writes the proofs of the last timed step (rank 0) as DIR/compliance_proofs.npy and DIR/vp_proofs.npy,
            one row of proof bytes per proof in float32, so that two builds can be compared output for output.
Synthetic data: Taiga-shaped circuits with satisfying witnesses (taiga_b200/circuits_taiga.py), a distinct witness per
proof; a sample of the proofs of the last timed step is checked with the oracle's verifier restatement and ALL of them
with the device verifier, outside the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N15 = 1 << 15
SASS_PER_MODMUL = 247          # cuobjdump count of the inlined Montgomery product (profiles/r02_modmul_sass.md)
INT_LANES_PER_SM = 64          # 16 lanes x 4 sub-partitions: one integer warp instruction per 2 cycles per sub-partition (tools/modmul_bench.cu)
PUBLISHED = {"compliance_proof_s": 3.1445, "vp_proof_s": 2.2328, "source": "taiga_halo2/benches/Perfromance.md:3,9 (hardware not stated)"}


def load_srs():
    raw = np.fromfile(os.path.join(ROOT, "tests", "golden", "srs_k15_affine.bin"), dtype=np.uint8).reshape(-1, 64)
    return {"k": 15, "n": N15, "g": raw[:N15], "g_lagrange": raw[N15:2 * N15], "w": raw[2 * N15], "u": raw[2 * N15 + 1]}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        try:
            p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                 stdout=subprocess.PIPE, text=True)
        except Exception:
            return
        self.proc = p
        for line in p.stdout:
            if self.stop_flag:
                break
            self.samples.append([x.strip() for x in line.split(",")])
        p.terminate()

    def summary(self):
        self.stop_flag = True
        if getattr(self, "proc", None):
            self.proc.terminate()
        sm = sorted(int(float(s[0])) for s in self.samples if s and s[0].replace(".", "").isdigit())
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            for i, nme in enumerate(names):
                if len(s) > 3 + i and s[3 + i].lower().startswith("active"):
                    reasons.add(nme)
        mx = [int(float(s[1])) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


class CpuFarm:
    """CPU arm: W oracle prover processes (oracle/cpu_worker.py) of T threads each, W*T = the host's hardware threads, proving
    independent proofs side by side.  One prover on all threads stops scaling at about 8 threads (FFT stages, serial
    transcript phases), so this is how the reference prover would be run for throughput on a many-core host."""
    THREADS = 4
    GB_PER_WORKER = 3.0   # resident set is about 1.2 GB per prover (keys + one proof in flight); headroom for the extended-domain buffers

    @staticmethod
    def host_threads():
        """hardware threads this process may really use: the affinity mask, cut by a cgroup CPU quota when the container has one"""
        hw = len(os.sched_getaffinity(0))
        try:
            quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]   # cgroup v2
            if quota != "max":
                hw = min(hw, max(1, int(float(quota) / float(period))))
        except (OSError, ValueError):
            try:   # cgroup v1
                q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
                p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    hw = min(hw, max(1, q // p))
            except (OSError, ValueError):
                pass
        return hw

    def __init__(self, workers=None, threads=None):
        import subprocess
        hw = self.host_threads()
        self.threads = threads or int(os.environ.get("TB_CPU_THREADS_PER_PROVER", min(self.THREADS, hw)))
        w = workers or int(os.environ.get("TB_CPU_PROVERS", max(1, hw // self.threads)))
        try:
            import psutil
            w = max(1, min(w, int(psutil.virtual_memory().available / 2**30 / self.GB_PER_WORKER)))
        except ImportError:
            pass
        self.workers = w
        env = dict(os.environ, OMP_NUM_THREADS="1", OPENBLAS_NUM_THREADS="1", MKL_NUM_THREADS="1", CUDA_VISIBLE_DEVICES="")
        self.procs = [subprocess.Popen([sys.executable, os.path.join(ROOT, "oracle", "cpu_worker.py"), str(self.threads)], stdin=subprocess.PIPE, stdout=subprocess.PIPE,
                                       text=True, env=env) for _ in range(w)]
        for p in self.procs:
            if p.stdout.readline().strip() != "ready":
                for q in self.procs:
                    q.kill()
                raise RuntimeError("CPU prover worker failed to start")

    def sample(self, provers=None):
        """Every worker (or the first `provers` of them) proves 1 Compliance-shaped + 1 VP-shaped proof at the same time; returns the cpu_baseline object."""
        procs = self.procs[:provers] if provers else self.procs
        t = time.time()
        for p in procs:
            p.stdin.write("go\n")
            p.stdin.flush()
        res = [tuple(float(x) for x in p.stdout.readline().split()) for p in procs]
        wall = time.time() - t
        if any(len(r) != 2 for r in res):
            raise RuntimeError("CPU prover worker died")
        val = sum(1.0 / (2 * c + 4 * v) for c, v in res)   # each prover's serial-loop rate (2C + 4V per ptx, shielded_ptx.rs:107-125), summed
        cs, vs = sorted(c for c, _ in res), sorted(v for _, v in res)
        pub = 2 * PUBLISHED["compliance_proof_s"] + 4 * PUBLISHED["vp_proof_s"]
        return {"value": val, "unit": "ptx/s", "cores": len(procs) * self.threads, "kind": "port",
                "sample": "%d concurrent prover processes x %d threads, each proving 1 Compliance-shaped + 1 VP-shaped proof (k=15) in %.1f s of wall time; "
                          "value = sum over provers of 1/(2C+4V) seconds per ptx" % (len(procs), self.threads, wall),
                "provers": len(procs), "threads_per_prover": self.threads, "sample_wall_s": round(wall, 2),
                "compliance_proof_s": round(cs[len(cs) // 2], 3), "vp_proof_s": round(vs[len(vs) // 2], 3),
                "reference_published": dict(PUBLISHED, ptx_per_s=round(1.0 / pub, 5))}

    def close(self):
        for p in self.procs:
            try:
                p.stdin.write("quit\n")
                p.stdin.close()
            except OSError:
                pass
        for p in self.procs:
            try:
                p.wait(timeout=20)
            except Exception:
                p.kill()


WORKLOAD = "%d shielded partial transaction(s) per GPU per step = %d Compliance-shaped (degree 17, ext 2^19, 4480 B proofs) + %d VP-shaped (degree 9) Halo2/IPA proofs, k=15, Taiga params_15 SRS (BASELINE configs[%d])"


def default_ptx(world):
    return 128 if world >= 8 else 64


def run_reference(args, rank, world):
    """--impl reference: the CPU arm (oracle port; the Rust reference cannot be compiled here: no cargo, un-vendored git deps).
    Every step is the bounded sample of CpuFarm.sample(): all host threads busy with independent provers, one Compliance-shaped and
    one VP-shaped proof each; the value is the summed ptx/s of those provers (proofs are independent, so batch size does not change it)."""
    if rank != 0:
        return
    P = args.ptx or default_ptx(world)
    times = []
    base = None
    farm = CpuFarm()
    try:
        for i in range(args.warmup + args.steps):
            base = farm.sample()
            if i >= args.warmup:
                times.append(1.0 / base["value"])
    finally:
        farm.close()
    sec_per_ptx = sum(times) / len(times)
    val = 1.0 / sec_per_ptx
    line = {"impl": "reference", "metric": "partial-tx proofs/sec", "value": val, "unit": "ptx/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * sec_per_ptx * P * world, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32x8 (255-bit Montgomery integers, Pasta Fp/Fq)", "data": "synthetic",
            "config": {"workload": WORKLOAD % (P, 2 * P, 4 * P, 2 if P > 1 else 1), "ptx_per_gpu": P,
                       "note": "CPU step = bounded sample (every prover process: 1 Compliance + 1 VP proof); ms_per_step is the time the host needs for the %d ptx of the step at that rate" % (P * world)},
            "cpu_baseline": dict(base, value=val), "e2e": {"value": val, "unit": "ptx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def witness_like(rng, n):
    """SURVEY 8d scalar mix of a Compliance advice column: 30 % zero, 30 % one, 20 % < 2^8, 8 % < 2^32, 12 % uniform."""
    s = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    s[:, 31] &= 0x3F
    u = rng.random(n)
    s[u < 0.3] = 0
    o = (u >= 0.3) & (u < 0.6)
    s[o] = 0
    s[o, 0] = 1
    s[(u >= 0.6) & (u < 0.8), 1:] = 0
    s[(u >= 0.8) & (u < 0.88), 4:] = 0
    return s


def sweep(ctx, hbm_peak, quick):
    """BASELINE configs[3]: standalone Vesta / Pallas MSM 2^16-2^22 and Fp NTT 2^17-2^23, device resident, algorithmic GB/s."""
    import torch
    from taiga_b200 import lib
    st = torch.cuda.ExternalStream(ctx.stream)
    out = {"msm": [], "ntt": []}
    rng = np.random.default_rng(0)
    srs = load_srs()
    msm_sizes = [16, 19, 22] if quick else list(range(16, 23))
    ntt_sizes = [17, 20, 23] if quick else list(range(17, 24))
    # 2^16 distinct Pallas points [i] * (-1, 2), made by the library itself (batched 1-term MSMs); the Vesta rows use Taiga's SRS
    # points.  Larger sizes tile the 2^16 points: the (point, digit) pairs stay distinct in all but ~10^-4 of the bucket additions.
    pallas_pts = None
    try:
        P_MOD = 0x40000000000000000000000000000000224698fc094cf91b992d30ed00000001
        G = np.frombuffer((P_MOD - 1).to_bytes(32, "little") + (2).to_bytes(32, "little"), np.uint8)
        halves = []
        for h in range(2):
            sc = np.zeros((1 << 15, 32), np.uint8)
            idx = np.arange(1, (1 << 15) + 1, dtype=np.uint64) + (h << 15)
            for b_ in range(3):
                sc[:, b_] = (idx >> (8 * b_)) & 0xFF
            halves.append(ctx.msm(lib.TB_PALLAS, sc, G[None], batch=1 << 15))
        pallas_pts = np.concatenate(halves)
    except Exception as ex:  # pragma: no cover
        sys.stderr.write("pallas sweep skipped: %r\n" % (ex,))
    for lg in msm_sizes:
        n = 1 << lg
        for curve, cname, pts_src in ((lib.TB_VESTA, "vesta", np.concatenate([srs["g"], srs["g_lagrange"]])), (lib.TB_PALLAS, "pallas", pallas_pts)):
            if pts_src is None:
                continue
            pts = np.concatenate([pts_src] * max(1, -(-n // len(pts_src))))[:n]
            fs, fb = (lib.TB_FP, lib.TB_FQ) if curve == lib.TB_VESTA else (lib.TB_FQ, lib.TB_FP)
            d_pts = torch.from_numpy(np.ascontiguousarray(pts)).cuda()
            ctx.dev_to_mont(fb, d_pts, 2 * n)
            d_out = torch.zeros(64, dtype=torch.uint8, device="cuda")
            for dist in ("uniform", "witness"):
                if dist == "uniform":
                    sc = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
                    sc[:, 31] &= 0x3F
                else:
                    sc = witness_like(rng, n)
                d_sc = torch.from_numpy(sc).cuda()
                ctx.dev_to_mont(fs, d_sc, n)
                for _ in range(2):
                    ctx.dev_msm(curve, n, d_sc, d_pts, d_out)
                ctx.sync()
                reps = 3
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(st)
                for _ in range(reps):
                    ctx.dev_msm(curve, n, d_sc, d_pts, d_out)
                e1.record(st)
                ctx.sync()
                ms = e0.elapsed_time(e1) / reps
                gbs = 96.0 * n / (ms * 1e-3) / 1e9
                out["msm"].append({"curve": cname, "scalars": dist, "log2_n": lg, "ms": round(ms, 3), "gpoints_per_s": round(n / ms / 1e6, 4), "alg_gbs": round(gbs, 2),
                                   "frac_hbm": round(gbs / hbm_peak, 5)})
                del d_sc
            del d_pts
    for lg in ntt_sizes:
        n = 1 << lg
        x = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
        x[:, 31] &= 0x3F
        d_in = torch.from_numpy(x).cuda()
        d_out = torch.empty_like(d_in)
        d_scr = torch.empty_like(d_in)
        ctx.dev_to_mont(lib.TB_FP, d_in, n)
        for name, kw in (("forward", {}), ("inverse", {"inverse": True}), ("coset", {"coset": True})):
            if quick and name != "forward":
                continue
            for _ in range(2):
                ctx.dev_ntt(lib.TB_FP, lg, d_in, d_out, d_scr, **kw)
            ctx.sync()
            reps = 5
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(reps):
                ctx.dev_ntt(lib.TB_FP, lg, d_in, d_out, d_scr, **kw)
            e1.record(st)
            ctx.sync()
            ms = e0.elapsed_time(e1) / reps
            gbs = 64.0 * n / (ms * 1e-3) / 1e9
            out["ntt"].append({"kind": name, "log2_n": lg, "ms": round(ms, 4), "alg_gbs": round(gbs, 1), "frac_hbm": round(gbs / hbm_peak, 4),
                               "int_util": round((n / 2) * lg * SASS_PER_MODMUL / (ms * 1e-3) / (148 * INT_LANES_PER_SM * 1.965e9), 3)})
        del d_in, d_out, d_scr
    return out


# The contract is ONE JSON line on stdout.  Libraries may write to file descriptor 1 behind Python's back (NCCL prints its
# version banner there when the communicator is created), so the real stdout is set aside at import time, everything
# else that targets fd 1 is sent to stderr, and only emit() writes to the real one.
_REAL_STDOUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, records):
    """records: {name: list of equal-length proof byte strings}.  Writes out_dir/<name>.npy, float32 [proofs, bytes] (exact for
    bytes).  Above DUMP_LIMIT_BYTES in all, every array keeps the same share of its rows, a sample fixed by seed 0."""
    arrays = {k: np.frombuffer(b"".join(v), np.uint8).reshape(len(v), -1) for k, v in records.items()}
    total = sum(4 * a.size for a in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_LIMIT_BYTES:
            keep = len(a) * DUMP_LIMIT_BYTES // total
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernels, from the committed ncu capture
    (written by profiles/extract_ncu_traffic.py from the raw page of the .ncu-rep; not a constant in this file)."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    try:
        return json.load(open(p))
    except Exception:
        return {}


ALG_BYTES_NOTE = {
    "ntt": "64*n per size-n transform (read + write once)",
    "msm_accum": "96 B per MSM term (64 B affine base + 32 B scalar); IPA 192*n per proof (SURVEY 8d)",
    "msm_sort": "96 B per MSM term", "msm_reduce": "96 B per MSM term",
    "quotient_gates": "32*(C+1) B per extended row, C = column-cosets read", "quotient_finish": "32*(C+1) B per extended row",
    "ipa_fold": "96 B per folded generator", "transcript": "-", "lookup_sort": "64 B per key", "poly": "64 B per coefficient",
}
KERNEL_OF = {"msm_accum": "msm_ba_fwd_kernel + msm_ba_bwd_kernel (batch-affine rounds)", "quotient_gates": "q_interp_kernel", "ntt": "ntt_pass_kernel",
             "msm_sort": "msm_sort_kernel", "msm_reduce": "msm_linesum_kernel + msm_weighted_kernel", "quotient_finish": "q_finish_kernel"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--ptx", type=int, default=0, help="partial transactions per GPU per step (default 64 = BASELINE configs[2]; 128 at 8 GPUs = configs[4]; 1 = configs[1])")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--full-sweep", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--no-synth-pipeline", action="store_true")
    ap.add_argument("--all-probes", action="store_true", help="multi-GPU runs skip the secondary probes (single-ptx latency, overlapped synthesis) unless this is given")
    ap.add_argument("--serial", action="store_true", help="one stream, no threads (for ncu launch lists; not a benchmark configuration)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the proofs of the last timed step as DIR/<name>.npy (float32 bytes)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's proofs; the reference arm makes none")
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1 and not args.all_probes:   # the scaling runs need value / e2e; the secondary probes cost host cores and minutes on every rank
        args.no_latency = args.no_synth_pipeline = True

    from taiga_b200 import ptx, shard
    # witness-synthesis workers, forked before CUDA / threads exist; the host cores are shared by the ranks of a multi-GPU run.
    # Half of the usable hardware threads: with more, the overlapped pipeline starves the proving threads (16-CPU quota on the
    # B200 box: 14 processes -> 18.0 ptx/s overlapped, 11 -> 18.8, 8 -> 19.9; profiles/r02_bench_synth_pipe_procs8.json)
    spool = ptx.SynthPool(int(os.environ.get("TB_SYNTH_PROCS", 0)) or min(64, max(4, (CpuFarm.host_threads() // 2) // max(1, world))))
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    srs = load_srs()
    P = args.ptx or default_ptx(world)
    nw_lat = 1 if args.serial else 2                      # single ptx: two streams per circuit so latency-bound phases overlap
    nw_batch = 1 if (args.serial or P > 2) else 2         # batches fill the GPU from one stream per circuit
    svc = ptx.ProverService(local, srs, c_workers=int(os.environ.get("TB_C_WORKERS", nw_lat)), v_workers=int(os.environ.get("TB_V_WORKERS", nw_lat)), serial=args.serial)
    ctx = svc.ctx
    t_syn = time.time()
    wit = svc.synthesize_ptx(P, wseed=rank, pool=spool)
    synth_s = time.time() - t_syn
    h2d = wit["c_adv"].nbytes + wit["v_adv"].nbytes + wit["c_inst"].nbytes + wit["v_inst"].nbytes
    d2h = svc.pk_c.proof_len * 2 * P + svc.pk_v.proof_len * 4 * P
    c_pin, v_pin = torch.from_numpy(wit["c_adv"]).pin_memory(), torch.from_numpy(wit["v_adv"]).pin_memory()
    c_dev, v_dev = c_pin.cuda(), v_pin.cuda()
    st = torch.cuda.ExternalStream(ctx.stream)
    seed0 = bytes((rank * 37 + i) & 0xFF for i in range(32))

    def step(i, device_resident, w=wit, cd=None, vd=None, nw=nw_batch):
        seed = bytes((b + i) & 0xFF for b in seed0)
        if cd is None:
            cd, vd = (c_dev, v_dev) if device_resident else (c_pin, v_pin)
        proofs = svc.build_ptx_batch(w, seed, cd, vd, workers_per_circuit=nw)
        if world > 1:  # the only collective on the path: gather the finished proof bytes (fixed-size records) over NCCL
            rec = shard.pack_records(proofs[0], proofs[1], svc.pk_c.proof_len, svc.pk_v.proof_len)
            shard.gather_records(rec, (len(proofs[0]) // 2) * world, device="cuda")
        return proofs

    def timed(device_resident, steps, warmup, **kw):
        for i in range(warmup):
            step(i, device_resident, **kw)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        l0 = svc.launch_count
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record(st)
        last = None
        for i in range(steps):
            last = step(100 + i, device_resident, **kw)
        e1.record(st)
        torch.cuda.synchronize()
        wall = time.time() - t0
        if world > 1:
            dist.barrier()
        ms = max(e0.elapsed_time(e1), 0.0)
        t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), svc.launch_count - l0, last

    sampler = ClockSampler(local)
    sampler.start()
    dev_ms, dev_wall_ms, launches, last = timed(True, args.steps, args.warmup)
    e2e_ms, e2e_wall_ms, _, last_e2e = timed(False, args.steps, args.warmup)
    clocks = sampler.summary()

    # configs[1]: one partial transaction per step, two streams per circuit (latency-bound; secondary figure)
    latency = None
    if not args.no_latency and P > 1:
        w1 = {k_: (v_[:2] if k_.startswith("c_") and k_ != "c_len" else v_[:4] if k_.startswith("v_") and k_ != "v_len" else v_) for k_, v_ in wit.items() if not k_.startswith("_")}
        c1, v1 = c_dev[:2], v_dev[:4]
        lsteps = max(5, args.steps)
        _, lw, ll, _ = timed(True, lsteps, 3, w=w1, cd=c1, vd=v1, nw=nw_lat)
        c1p, v1p = c_pin[:2], v_pin[:4]
        _, lw2, _, _ = timed(False, lsteps, 2, w=w1, cd=c1p, vd=v1p, nw=nw_lat)
        latency = {"workload": "1 partial transaction per step (BASELINE configs[1]), %d CUDA streams per circuit" % nw_lat, "ms_per_ptx": round(lw / lsteps, 3),
                   "value": round(world * 1e3 / (lw / lsteps), 4), "e2e_value": round(world * 1e3 / (lw2 / lsteps), 4), "unit": "ptx/s", "gpu_launches_per_ptx": int(ll / lsteps), "steps": lsteps}

    # host witness synthesis on the clock (SURVEY 8 (f)-1): the stand-in for Rust `synthesize` runs in worker processes WHILE the
    # previous batch is proved; every step's advice comes from pageable shared memory through the C ABI (H2D inside the timed region)
    synth_pipe = None
    if not args.no_synth_pipeline and P > 1:
        rt = torch.cuda.cudart()
        locked = set()

        def page_lock(a, on):
            """cudaHostRegister / Unregister of a witness array; a refusal (e.g. a locked-memory limit) only costs the fast DMA"""
            if on:
                if int(rt.cudaHostRegister(a.ctypes.data, a.nbytes, 0)) == 0:
                    locked.add(a.ctypes.data)
                else:
                    try:   # drop the (per-thread) error so that the library's launch checks do not see it
                        import ctypes
                        ctypes.CDLL("libcudart.so.12").cudaGetLastError()
                    except OSError:
                        pass
            elif a.ctypes.data in locked:
                locked.discard(a.ctypes.data)
                rt.cudaHostUnregister(a.ctypes.data)

        # three stages, each on its own thread, one step apart: synthesis (forked processes) -> page-locking -> proving (+ release)
        import queue
        psteps = 3
        q_synth, q_ready, q_done = queue.Queue(maxsize=1), queue.Queue(maxsize=1), queue.Queue()
        stage_s = {"synthesis": 0.0, "page_lock": 0.0, "prove": 0.0, "release": 0.0}

        import shutil
        set_bytes = wit["c_adv"].nbytes + wit["v_adv"].nbytes
        live = threading.Semaphore(3 if shutil.disk_usage("/dev/shm").free > 3.3 * set_bytes else 2)   # witness sets alive at once (4 GB each at P = 64)

        def stage_synth():
            for i in range(psteps + 1):
                live.acquire()
                t_ = time.time()
                w_ = svc.synthesize_ptx(P, wseed=1000 + 10 * rank + i, pool=spool)
                stage_s["synthesis"] += time.time() - t_
                q_synth.put(w_)

        def stage_lock():
            for i in range(psteps + 1):
                w_ = q_synth.get()
                t_ = time.time()
                for key in ("c_adv", "v_adv"):   # page-lock the shared memory so that the upload is one fast DMA
                    page_lock(w_[key], True)
                stage_s["page_lock"] += time.time() - t_
                q_ready.put(w_)

        def stage_release():
            while True:
                w_ = q_done.get()
                if w_ is None:
                    return
                t_ = time.time()
                for key in ("c_adv", "v_adv"):
                    page_lock(w_[key], False)
                stage_s["release"] += time.time() - t_
                del w_
                live.release()

        ths = [threading.Thread(target=f) for f in (stage_synth, stage_lock, stage_release)]
        for th in ths:
            th.start()
        cur = q_ready.get()   # the first step's witnesses are ready before the clock starts (steady state of a service)
        page_locked_any = len(locked) > 0
        for key in stage_s:
            stage_s[key] = 0.0
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.time()
        for i in range(psteps):
            t_ = time.time()
            step(200 + i, False, w=cur, cd=cur["c_adv"], vd=cur["v_adv"])
            stage_s["prove"] += time.time() - t_
            q_done.put(cur)
            cur = q_ready.get()   # the witnesses of the next step (the last one is synthesised but not proved: steady state)
        torch.cuda.synchronize()
        pw = torch.tensor([(time.time() - t0) * 1e3], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(pw, op=dist.ReduceOp.MAX)
        q_done.put(cur)
        q_done.put(None)
        for th in ths:
            th.join()
        synth_pipe = {"page_locked": bool(page_locked_any), "value": round(P * world / (float(pw[0]) * 1e-3 / psteps), 4), "unit": "ptx/s", "steps": psteps,
                      "stage_seconds_per_step": {k_: round(v_ / psteps, 3) for k_, v_ in stage_s.items()},
                      "note": "fresh witnesses every step; three host stages one step apart: synthesis by forked host processes, page-locking (cudaHostRegister) of the shared-memory advice, "
                              "proving through the C ABI; the slowest stage sets the rate"}

    # one profiled step (CUDA events around every kernel group) for the share-of-step table and the roofline.  It runs the
    # workers one after the other: with the streams overlapped an event pair also times the wait for SMs held by the other
    # streams' kernels, and the shares would not be comparable with the (serialised) ncu launch list in profiles/.
    svc.prof_enable(True)
    svc.work_read()   # reset the multiplication counters
    was_serial, svc.serial = svc.serial, True
    step(999, True)
    svc.serial = was_serial
    prof = svc.prof_read()
    work = svc.work_read()
    svc.prof_enable(False)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"compliance_proofs": last[0], "vp_proofs": last[1]})

    # acceptance (outside the timed region): a sample of the last e2e step under the oracle's verifier restatement (35 ms/proof of
    # CPU each), ALL of its proofs under the library's batched device verifier (tb_verify_batch, SURVEY 8 (f)-3)
    accepted = None
    try:
        from oracle import cpu as oc
        kc, kv = oc.OracleKey(svc.kd_c, srs), oc.OracleKey(svc.kd_v, srs)
        ic = sorted(set([0, len(last_e2e[0]) // 2, len(last_e2e[0]) - 1] + list(range(0, len(last_e2e[0]), 16))))
        iv = sorted(set([0, len(last_e2e[1]) // 2, len(last_e2e[1]) - 1] + list(range(0, len(last_e2e[1]), 32))))
        accepted = all(kc.verify(wit["c_inst"][i], wit["c_len"], last_e2e[0][i]) == 0 for i in ic) and \
            all(kv.verify(wit["v_inst"][i], wit["v_len"], last_e2e[1][i]) == 0 for i in iv)
        accepted = {"all_accepted": bool(accepted), "checked": len(ic) + len(iv), "of": len(last_e2e[0]) + len(last_e2e[1])}
    except Exception as ex:  # pragma: no cover
        accepted = "verifier unavailable: %r" % (ex,)
    try:
        accepted_dev = all(svc.pk_c.verify_batch(wit["c_inst"], wit["c_len"], list(last_e2e[0]))) and \
            all(svc.pk_v.verify_batch(wit["v_inst"], wit["v_len"], list(last_e2e[1]), ctx=svc.v_workers[0][0]))
    except Exception as ex:  # pragma: no cover
        accepted_dev = "device verifier failed: %r" % (ex,)

    hbm_peak, peak_kind = measured_peaks()
    total_ptx = P * world
    dev_step_ms, e2e_step_ms = dev_wall_ms / args.steps, e2e_wall_ms / args.steps
    value = total_ptx / (dev_step_ms * 1e-3)
    e2e_val = total_ptx / (e2e_step_ms * 1e-3)
    tot_prof = sum(v[0] for v in prof.values()) or 1.0
    n = N15
    nproofs_c, nproofs_v = 2 * P, 4 * P
    cs_c, cs_v = svc.kd_c.cs, svc.kd_v.cs
    # algorithmic bytes of one profiled step per category (SURVEY 8d figures x units processed)
    commits_c, commits_v = 33, 26                       # n-term commitments per proof (SURVEY 8a H1)
    msm_bytes = (nproofs_c * commits_c + nproofs_v * commits_v) * 96.0 * n + (nproofs_c + nproofs_v) * 192.0 * n   # + IPA: 192*n per proof
    alg = {
        "msm_accum": msm_bytes, "msm_sort": msm_bytes, "msm_reduce": msm_bytes,
        "ntt": 64.0 * n * (nproofs_c * (14 + 15 * 16 + 16) + nproofs_v * (15 + 16 * 8 + 8)),
        "quotient_gates": 32.0 * (cs_c.num_advice + cs_c.num_fixed + 2) * (1 << 19) * nproofs_c + 32.0 * (cs_v.num_advice + cs_v.num_fixed + 2) * (1 << 18) * nproofs_v,
        "ipa_fold": 96.0 * n * (nproofs_c + nproofs_v),
    }
    clk_hz = (clocks.get("sm_mhz") or 1965) * 1e6
    int_peak = 148 * INT_LANES_PER_SM * clk_hz          # integer lane-instructions per second

    def int_util(cat, ms):
        mm = work.get(cat)
        if not mm or ms <= 0:
            return None, None
        return round(mm / (ms * 1e-3) / 1e9, 2), round(mm * SASS_PER_MODMUL / (ms * 1e-3) / int_peak, 4)

    top_name, (top_ms, top_groups) = max(prof.items(), key=lambda kv_: kv_[1][0])     # dominant GROUP of the step, whatever it is
    top_bytes = alg.get(top_name)
    tr = ncu_traffic()
    roof = {"bound": "hbm", "kernel": top_name, "kernel_name": KERNEL_OF.get(top_name), "achieved": None, "peak": hbm_peak, "unit": "GB/s", "frac": None, "traffic": None,
            "peak_source": peak_kind, "share_of_step": round(top_ms / tot_prof, 3), "launch_groups": top_groups, "avg_group_ms": round(top_ms / max(1, top_groups), 4),
            "algorithmic_bytes_per_step": top_bytes, "bytes_rule": ALG_BYTES_NOTE.get(top_name),
            "note": "255-bit modular arithmetic: every hot kernel is bound by the integer pipe (0.5 warp instructions per cycle per SM sub-partition, measured by tools/modmul_bench.cu: "
                    "72.7 G Montgomery products/s = int_util 0.97), not by HBM; frac is reported against HBM because the metric asks for it, int_util is the binding roofline"}
    if top_bytes:
        roof["achieved"] = round(top_bytes / (top_ms * 1e-3) / 1e9, 2)
        roof["frac"] = round(roof["achieved"] / hbm_peak, 5)
    roof["gmodmul_per_s"], roof["int_util"] = int_util(top_name, top_ms)
    if top_name in tr:
        roof["traffic"] = tr[top_name].get("dram_bytes_per_launch")
        roof["traffic_detail"] = tr[top_name]
    roof["per_kernel"] = {}
    for k_, v_ in prof.items():
        gm, iu = int_util(k_, v_[0])
        roof["per_kernel"][k_] = {"ms": round(v_[0], 3), "groups": v_[1], "achieved_gbs": (round(alg[k_] / (v_[0] * 1e-3) / 1e9, 2) if alg.get(k_) and v_[0] > 0 else None),
                                  "frac": (round(alg[k_] / (v_[0] * 1e-3) / 1e9 / hbm_peak, 5) if alg.get(k_) and v_[0] > 0 else None), "gmodmul_per_s": gm, "int_util": iu}
    line = {
        "metric": "partial-tx proofs/sec", "value": round(value, 4), "unit": "ptx/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(dev_step_ms, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32x8 (255-bit Montgomery integers, Pasta Fp/Fq)", "data": "synthetic",
        "config": {"workload": WORKLOAD % (P, 2 * P, 4 * P, 1 if P == 1 else (4 if world >= 8 and P >= 128 else 2)), "ptx_per_gpu": P,
                   "parallelism": "independent ptx per GPU (no collective inside a proof; NCCL all_gather of proof bytes); %d CUDA stream(s) per circuit, tb_prove_batch chunks of 64 proofs" % nw_batch,
                   "l2": "inputs (60 MiB advice per ptx, %.1f GB per step + 0.9 GB resident key cosets) exceed L2; no explicit flush" % (h2d / 1e9),
                   "hbm_resident_gb": round(torch.cuda.memory_allocated() / 1e9, 1), "proofs_accepted_by_oracle_verifier": accepted, "proofs_accepted_by_device_verifier": accepted_dev},
        "e2e": {"value": round(e2e_val, 4), "unit": "ptx/s", "ms_per_step": round(e2e_step_ms, 3), "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
        "device_event_ms_per_step": round(dev_ms / args.steps, 3),
        "gpu_launches": int(launches), "gpu_launches_per_proof": round(launches / max(1, args.steps * 6 * P), 1), "clocks": clocks,
        "roofline": roof,
        "profile_share": {k: round(v[0] / tot_prof, 4) for k, v in sorted(prof.items(), key=lambda kv_: -kv_[1][0])},
        "profile_ms": {k: round(v[0], 3) for k, v in prof.items()},
        "kernel_time_over_step_time": round(tot_prof / dev_step_ms, 3),
        "latency": latency,
        "witness_synthesis": {"seconds_for_step_inputs": round(synth_s, 2), "ptx_per_s": round(P / synth_s, 2), "procs": "%d forked host processes (ptx.SynthPool)" % spool.procs,
                              "note": "host synthesis of the Taiga-shaped witnesses (the stand-in for Rust Circuit::synthesize, compliance_circuit.rs:174-327); outside value and e2e, "
                                      "reported so that an end-to-end service can be sized: e2e_with_synthesis = 1 / (1/e2e + 1/synthesis) if not overlapped",
                              "e2e_with_synthesis_serial": round(1.0 / (1.0 / e2e_val + synth_s / total_ptx), 4), "e2e_with_synthesis_overlapped": synth_pipe},
    }
    try:
        free_b, total_b = torch.cuda.mem_get_info()
        line["config"]["hbm_used_gb"] = round((total_b - free_b) / 1e9, 1)
    except Exception:
        pass
    if not args.no_sweep and world == 1:
        line["sweeps"] = sweep(ctx, hbm_peak, quick=not args.full_sweep)
    if not args.no_cpu and world == 1:   # the CPU arm is timed on rank 0 of a single-GPU run only
        try:   # a failure of the CPU arm must not cost the GPU line
            farm = CpuFarm()
            try:
                line["cpu_baseline"] = farm.sample()
            finally:
                farm.close()
            line["speedup_e2e_vs_cpu_port"] = round(e2e_val / line["cpu_baseline"]["value"], 2)
            line["speedup_e2e_vs_published_reference"] = round(e2e_val / line["cpu_baseline"]["reference_published"]["ptx_per_s"], 2)
        except Exception as ex:  # pragma: no cover
            line["cpu_baseline"] = {"value": None, "unit": "ptx/s", "kind": "port", "error": repr(ex)}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
