#!/usr/bin/env python
"""bench.py — GG20 offline-signing phases/s on B200 (BASELINE.json metric, configs[4] sharded per GPU).

A "step" is one pass of the hot path over one batch: every rank runs 8 192 two-signer sessions = 16 384 party-phases
("units": one party's OfflineStage Round0..Round6, t = 1, n = 3) over 8 synthetic key sets, builds the 256-byte result
record of every unit and joins the single NCCL all-gather of those records (SURVEY.md section 8d/e, config 5).  Ranks hold
disjoint sessions (weak scaling: the batch per GPU is fixed).

  value  : phases/s, whole job, inputs resident in HBM, CUDA-event timed on the engine's stream, max over ranks.
  e2e    : the same metric through ONE C-ABI call with HOST (pinned) buffers — tecdsa_gg20_offline_records: H2D of the
           randomness records and session descriptors -> seven rounds -> record packing -> NCCL gather -> D2H of the
           gathered records, all inside the timed region.
  roofline: the path is bound by the INT32 multiply-add pipe (IMAD.WIDE.U32), not HBM and not the tensor cores
           (SURVEY.md section 8d).  `achieved` = multiply-accumulates counted by the kernels themselves (tecdsa_ctx_work)
           for the dominant kernel, divided by its launch durations measured with CUDA events around each of its launches
           in this run; `peak` = the on-box IMAD.WIDE.U32 saturation micro-benchmark (MEASURED_PEAKS.json has no integer
           entry).  The reference-operation-list view (W_unit = 2.003e9 MAC32 per unit) and the HBM view are reported beside it.
  parity : inside the run — 256 sampled units (status, R, sigma_i, k_i, transcript digest) bit-compared with the CPU twin
           of the oracle (GMP + OpenSSL), every session signed on the device (online step) and the sampled sessions'
           signatures verified under OpenSSL (`cryptography`), as gg_2020/test.rs:711-748 does with libsecp256k1.
  cpu_baseline / --impl reference: the same protocol executed the way the reference executes it on a CPU (scalar GMP
           mpz_powm / mpz_invert, every redundant verification kept) on all host threads — oracle/gg20_twin.c; the Rust
           reference itself cannot be built in this image (no cargo/rustc, crates not vendored).
Secondary block `modexp`: BASELINE.json configs[1], 65 536 x 2048-bit modexp, ALL outputs compared with GMP.
"""
from __future__ import annotations

import argparse
import ctypes
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SESSIONS_PER_GPU = 8192                 # 16 384 units per GPU: configs[4] (128k units over 8 GPUs)
SEED = 0xB2000005                       # SURVEY.md section 8(d) config 5
METRIC = "GG20 offline-sign phases/sec (batched)"
UNIT = "phases/s"
WORKLOAD = ("batch 128k full GG20 offline-signing phases (t=1,n=3) sharded over 8xB200 with NCCL gather (BASELINE.json configs[4]): "
            "16384 phases (8192 two-signer sessions) per GPU, 8 key sets")
W_UNIT = 2.003e9                        # SURVEY.md section 8(d): MAC32 per unit, reference operation list
BYTES_PER_UNIT = 18 * 1024              # SURVEY.md section 8(d)
REC = 256
# modexp block (configs[1])
MODEXP_BATCH, K, EL, MODEXP_SEED = 65536, 64, 64, 0xB2000002
W_MODEXP = 1.2 * 2048 * (2 * K * K + K)
Q = 0xFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFEBAAEDCE6AF48A03BBFD25E8CD0364141
DUMP_BYTES, DUMP_SEED = 60 << 20, 0xB200D      # --dump-outputs: budget (under 64 MB with the .npy headers) and row-sample seed


def config_dict(world: int) -> dict:
    return {"workload": WORKLOAD, "sessions_per_gpu": SESSIONS_PER_GPU, "units_per_gpu": 2 * SESSIONS_PER_GPU, "keysets": 8, "t": 1, "n": 3,
            "signers": 2, "seed": SEED, "parallelism": f"shard{world}", "record_bytes": REC,
            "cache": "per-step working set (92 MB randomness records + 0.65 GB per-unit arena) exceeds the 126 MB L2"}


def host_threads() -> int:
    """Threads this process may actually run at once: the affinity mask capped by the cgroup CPU quota (a box whose container
    is limited to a few CPUs' worth of time gains nothing from one thread per visible core)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    if quota:
        n = max(1, min(n, int(quota + 0.5)))
    return n


def cpu_model() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.rows, self.proc, self.first = device, [], None, 0

    def mark(self):
        """samples from here on are the ones reported (the poller itself is started before the warm-up: its NVML start-up takes the driver
        lock for a few hundred ms, which would otherwise stall kernel launches inside the timed region)"""
        self.first = len(self.rows)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.device)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm, mx, reasons = [], 0, set()
        for r in self.rows[self.first:]:
            try:
                sm.append(float(r[1])); mx = max(mx, float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        loaded = sorted(x for x in sm if x > 0.5 * mx) or sorted(sm)
        return {"sm_mhz": loaded[len(loaded) // 2] if loaded else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------- workload
def load_keysets():
    from tests.golden import fixtures
    ks = fixtures.load_all_keysets()
    assert len(ks) == 8, "tests/golden/keys_t1n3.json must hold the 8 key sets of config 5"
    return ks


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write every array as out_dir/<name>.npy: bytes as float32 and 32-bit limbs as float64, both exact.  When the set exceeds
    DUMP_BYTES, each array keeps its share of the budget as a fixed, seeded sample of rows whose indices go to <name>_rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: v.astype(np.float32 if v.dtype.itemsize == 1 else np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            keep = max(1, int(DUMP_BYTES * a.nbytes / total) // (a.nbytes // a.shape[0] + 8))
            rows = np.sort(np.random.default_rng(DUMP_SEED).choice(a.shape[0], keep, replace=False))
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def make_batch(keysets, n_sessions: int, rank: int):
    """Sessions and randomness records of this rank's block (oracle-free: mpecdsa_b200.gg20.synthetic_batch)."""
    import __graft_entry__ as entry
    entry.load_package()                      # registers the package; the input generator needs neither the library nor a GPU
    from mpecdsa_b200 import gg20
    return gg20.synthetic_batch(keysets, n_sessions, SEED + 0x1000 * rank)


def message_limbs(n_sessions: int) -> np.ndarray:
    """The message of the reference's tests: Sha256.chain_bigint(from_bytes(b"ZenGo")).result_bigint() (sign.rs:693-696)."""
    m = int.from_bytes(hashlib.sha256(b"ZenGo").digest(), "big")
    row = np.frombuffer(m.to_bytes(32, "little"), dtype="<u4")
    return np.ascontiguousarray(np.tile(row, (n_sessions, 1))), m


# ------------------------------------------------------------------------------------------------- CPU arm (oracle twin)
def cpu_phases(keysets, n_sessions: int, threads: int, seed_rank: int = 1000):
    """Time the oracle's C twin (the reference's scalar GMP path) on `n_sessions` sessions of the same workload."""
    from oracle import twin
    kt = twin.KeyTables(keysets)
    sess, rnd = make_batch(keysets, n_sessions, seed_rank)
    t0 = time.perf_counter()
    res = twin.offline_batch(kt, sess, rnd, threads)
    dt = time.perf_counter() - t0
    if not (res.status == 0).all():
        raise SystemExit("CPU twin: a unit failed on valid inputs")
    return 2 * n_sessions / dt, dt


def cpu_sample_sessions(keysets, threads: int, target_s: float):
    """How many sessions keep `threads` host threads busy for about target_s: sized from a short probe, because the CPU time a
    GPU box gives its container varies from box to box (round 1 saw 5x between two boxes of the same CPU model)."""
    v1, _ = cpu_phases(keysets, 1, 1, seed_rank=900)
    vt, _ = cpu_phases(keysets, max(threads // 2, 2), threads, seed_rank=901)
    return max(int(vt * target_s / 2), 16), v1, vt


def run_reference(args):
    """Reference arm: the reference's CPU implementation of the path (scalar BigInt calls over GMP, secp256k1 on the CPU) on all
    host threads through a persistent thread pool; each step is a bounded sample of the workload."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import twin
    threads = host_threads()
    keysets = load_keysets()
    per_step, _, _ = cpu_sample_sessions(keysets, threads, 3.0)      # sessions per step: about 3 s of wall time on this box (also the warm-up)
    t, units = 0.0, 0
    for i in range(args.steps):
        v, dt = cpu_phases(keysets, per_step, threads, seed_rank=2000 + i)
        t += dt; units += 2 * per_step
    value = units / t
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": config_dict(world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{2 * per_step} phases ({per_step} sessions) per step x {args.steps} steps of the same workload, persistent pool of {threads} threads, "
                                   f"oracle/gg20_twin.c: the reference's scalar call sequence over GMP {twin.lib().oracle_gmp_version().decode()} mpz_powm/mpz_invert + OpenSSL "
                                   f"secp256k1/SHA-256, redundant verifications kept; cpu={cpu_model()}; the Rust reference cannot be built here (no cargo/rustc, crates not vendored)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------- modexp block
def modexp_inputs(count: int, seed: int):
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 2**32, size=(count, K), dtype=np.uint32)
    exp = rng.integers(0, 2**32, size=(count, EL), dtype=np.uint32)
    mod = rng.integers(0, 2**32, size=(count, K), dtype=np.uint32)
    mod[:, 0] |= 1
    mod[:, K - 1] |= 0x80000000
    exp[:, EL - 1] |= 0x80000000
    return base, exp, mod


def bench_modexp(eng, pkg, torch, rank, steps: int, threads: int, check: bool):
    """configs[1]: 65 536 independent 2048-bit modexps with distinct moduli; every output compared with GMP mpz_powm."""
    base, exp, mod = modexp_inputs(MODEXP_BATCH, MODEXP_SEED + rank)
    d_base, d_exp, d_mod = (torch.from_numpy(x.view(np.int32)).cuda() for x in (base, exp, mod))
    d_out = torch.empty((MODEXP_BATCH, K), dtype=torch.int32, device="cuda")
    d_st = torch.empty(MODEXP_BATCH, dtype=torch.uint8, device="cuda")

    def step():
        eng.modexp_raw(2048, EL, d_base, d_exp, d_mod, d_out, d_st, mem=pkg.DEVICE)

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    eng.work(reset=True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        step()
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / steps
    macs = eng.work() / steps
    out = {"metric": "2048-bit modexp/s", "value": MODEXP_BATCH / (ms * 1e-3), "unit": "modexp/s", "batch": MODEXP_BATCH, "steps": steps,
           "ms_per_step": ms, "executed_mac32_per_modexp": macs / MODEXP_BATCH, "reference_mac32_per_modexp": W_MODEXP}
    if check:
        lib = ctypes.CDLL(os.path.join(ROOT, "oracle", "libgg20_ref.so"))
        lib.oracle_modexp_batch.argtypes = [ctypes.c_void_p] * 5 + [ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_int]
        want = np.zeros_like(base)
        t0 = time.perf_counter()
        lib.oracle_modexp_batch(base.ctypes.data, exp.ctypes.data, mod.ctypes.data, None, want.ctypes.data, MODEXP_BATCH, K, EL, threads)
        dt = time.perf_counter() - t0
        got = d_out.cpu().numpy().view(np.uint32)
        out["outputs_compared_with_gmp"] = MODEXP_BATCH
        out["parity_ok"] = bool(np.array_equal(got, want)) and bool((d_st == 0).all().item())
        out["cpu_baseline"] = {"value": MODEXP_BATCH / dt, "unit": "modexp/s", "cores": threads, "kind": "port",
                               "sample": f"all {MODEXP_BATCH} modexps of the batch, GMP mpz_powm on {threads} threads"}
    return out, ms, macs


# ------------------------------------------------------------------------------------------------- main arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--sessions", type=int, default=SESSIONS_PER_GPU, help=argparse.SUPPRESS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-modexp", action="store_true", help="skip the secondary modexp block")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy: rank 0's per-unit status, R, sigma, t_vec, digest "
                         "and every rank's gathered 256-byte records")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    import __graft_entry__ as entry

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    pkg = entry.load_package()
    from mpecdsa_b200 import gg20
    stream = torch.cuda.current_stream()
    eng = pkg.Engine(local_rank, stream.cuda_stream)
    threads = host_threads()

    # ---- the workload: this rank's block of sessions, one pinned host copy, one device-resident copy
    n_sessions = args.sessions
    U = 2 * n_sessions
    keysets = load_keysets()
    ks = gg20.KeySets(eng, keysets)
    sess, rnd = make_batch(keysets, n_sessions, rank)
    h_rnd = torch.from_numpy(rnd.view(np.int32)).pin_memory()
    h_sess = torch.from_numpy(sess.view(np.int32)).pin_memory()
    d_rnd, d_sess = h_rnd.cuda(), h_sess.cuda()
    d_status = torch.empty(U, dtype=torch.uint8, device="cuda")
    d_R = torch.empty((U, 16), dtype=torch.int32, device="cuda")
    d_sigma = torch.empty((U, 8), dtype=torch.int32, device="cuda")
    d_tvec = torch.empty((U, 32), dtype=torch.int32, device="cuda")
    d_digest = torch.empty((U, 8), dtype=torch.int32, device="cuda")
    d_rec = torch.empty((U, REC), dtype=torch.uint8, device="cuda")
    d_all = torch.empty((world, U, REC), dtype=torch.uint8, device="cuda")
    h_all = torch.empty((world, U, REC), dtype=torch.uint8).pin_memory()

    # ---- the communicator of the single gather: id drawn by rank 0, handed round through torch.distributed
    comm = None
    if world > 1:
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.from_numpy(eng.nccl_unique_id()))
        dist.broadcast(idt, 0)
        comm = eng.nccl_comm_create(idt.cpu().numpy(), world, rank)

    def step_device():
        gg20.offline_raw(eng, ks, d_sess, n_sessions, d_rnd, d_status, d_R, d_sigma, d_tvec, d_digest, pkg.DEVICE)
        eng.pack_records(d_status, d_R, d_sigma, d_tvec, d_digest, d_rnd, U, d_rec)
        eng.gather_results(comm, d_rec, U, d_all)                     # the single NCCL all-gather (identity copy on one rank)

    def step_e2e():
        eng.offline_records(ks, comm, h_sess, n_sessions, h_rnd, h_all, pkg.HOST)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- device-resident timing
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step_device()
    barrier()
    sampler.mark()
    eng.work(reset=True)
    launches0 = eng.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        step_device()
    ev1.record(stream)
    barrier()
    dev_ms = ev0.elapsed_time(ev1)
    launches = eng.launch_count() - launches0
    macs_per_step = eng.work() / args.steps
    clocks = sampler.stop() if rank == 0 else None
    dev_records = d_all[rank].cpu().numpy().copy()
    outputs = None
    if args.dump_outputs and rank == 0:
        outputs = {"status": d_status, "R": d_R, "sigma": d_sigma, "t_vec": d_tvec, "digest": d_digest, "records": d_all.reshape(world * U, REC)}
        outputs = {k: v.cpu().numpy().view(np.uint32 if v.dtype == torch.int32 else np.uint8) for k, v in outputs.items()}

    # ---- per-launch durations of the job kernels (CUDA events around every launch, one extra step, single stream)
    prof = eng.profile_step(step_device)

    # ---- end to end: host buffers in, host records out, copies inside the timed region
    step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    t = torch.tensor([dev_ms, e2e_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms = (float(x) for x in t.tolist())
    e2e_records = h_all.numpy()

    # ---- the online step for every session (device), statuses must be OK
    msg, m_int = message_limbs(n_sessions)
    d_k = torch.from_numpy(np.ascontiguousarray(rnd[:, 8:16]).view(np.int32)).cuda()
    sig = gg20.sign_batch(eng, ks, sess, msg, d_R.cpu().numpy().view(np.uint32), d_sigma.cpu().numpy().view(np.uint32),
                          d_k.cpu().numpy().view(np.uint32))
    all_ok = bool((dev_records[:, 0] == 0).all()) and bool((sig["status"] == 0).all())
    paths_agree = bool(np.array_equal(e2e_records[rank], dev_records))
    gather_ok = True
    if world > 1:
        # every rank's block must have arrived identically on every rank: compare a digest of the gathered buffer
        dg = torch.tensor([int.from_bytes(hashlib.sha256(e2e_records.tobytes()).digest()[:7], "big")], dtype=torch.int64, device="cuda")
        lo, hi = dg.clone(), dg.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        gather_ok = bool((lo == hi).item()) and bool((e2e_records[:, :, 0] == 0).all())

    parity = None
    if rank == 0:
        parity = parity_block(keysets, sess, rnd, dev_records, sig, m_int, threads)

    modexp = None
    if not args.no_modexp:
        try:
            modexp, _, _ = bench_modexp(eng, pkg, torch, rank, args.steps, threads, check=(rank == 0))
        except Exception as exc:
            modexp = {"error": f"{type(exc).__name__}: {exc}"}

    if rank != 0:
        if comm is not None:
            eng.nccl_comm_destroy(comm)
        if world > 1:
            dist.destroy_process_group()
        return

    total_units = U * world
    value = total_units * args.steps / (dev_ms * 1e-3)
    e2e_value = total_units * args.steps / (e2e_ms * 1e-3)
    step_ms = dev_ms / args.steps
    # roofline denominator: the issue ceiling of the FMA-heavy pipe, 32 IMAD.WIDE.U32 per clock and SM (one warp instruction per
    # 4 cycles and sub-partition; confirmed by ncu: useful MACs x 4 cycles = the pipe-busy share, profiles/r02_ncu_*_summary.md) at the
    # SM clock sampled during the timed region.  The two on-box saturation micro-benchmarks (carry-free IMAD.WIDE.U32 and the
    # IMAD.WIDE.U32.X carry chains of the Montgomery rows) reach 78-87 % of it — their loops carry register moves on the same pipe
    # (profiles/r02_sass_mix.md) — and are reported beside it; the LARGER figure is the denominator so that `frac` is never flattered.
    peak_free, _ = eng.imad_peak()
    peak_chain, _ = eng.imad_peak(chained=True)
    sm_count = torch.cuda.get_device_properties(local_rank).multi_processor_count
    pipe_ceiling = sm_count * 32 * (clocks["sm_mhz"] or 0) * 1e6 if clocks else None
    peak_mac = max(peak_free, peak_chain, pipe_ceiling or 0.0)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    dom = max(prof.items(), key=lambda kv: kv[1]["ms"]) if prof else None
    roofline = {"bound": "int32-mad", "unit": "TMAC32/s", "peak": peak_mac / 1e12,
                "peak_source": "max(pipe issue ceiling = SMs x 32 IMAD.WIDE.U32 per clock x sampled SM clock, on-box saturation micro-benchmarks "
                               "tecdsa_imad_peak / tecdsa_imad_peak_chained); MEASURED_PEAKS.json has no integer entry",
                "peak_carry_free": peak_free / 1e12, "peak_carry_chained": peak_chain / 1e12,
                "pipe_ceiling": pipe_ceiling / 1e12 if pipe_ceiling else None,
                "pipe_ceiling_source": f"{sm_count} SMs x 32 IMAD.WIDE.U32 per clock x sampled SM clock"}
    if dom:
        name, d = dom
        ach = d["mac32"] / (d["ms"] * 1e-3)
        roofline.update({"kernel": name, "achieved": ach / 1e12, "frac": ach / peak_mac, "kernel_ms_per_step": d["ms"], "launches_per_step": d["launches"],
                         "work_per_step_mac32": d["mac32"], "work_source": "counted by the kernel (tecdsa_ctx_work), CUDA events around each launch",
                         "share_of_step_kernel_time": d["ms"] / sum(x["ms"] for x in prof.values()),
                         "frac_of_measured_microbenchmark": ach / max(peak_free, peak_chain), "traffic": None})
        try:        # dram__bytes_read + dram__bytes_write of this kernel's largest launch, from the committed ncu --set full capture
            t = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
            if t["kernel"].split("<")[0] == name.split("<")[0]:
                roofline["traffic"] = t["dram_bytes_read"] + t["dram_bytes_write"]
                roofline["traffic_note"] = "bytes of ONE launch (" + t["launch"] + "), " + t["source"]
        except Exception:
            pass
    roofline["whole_step"] = {
        "ms_per_step": step_ms, "executed_mac32_per_unit": macs_per_step / U,
        "achieved_executed": macs_per_step / (step_ms * 1e-3) / 1e12, "frac_executed": macs_per_step / (step_ms * 1e-3) / peak_mac,
        "reference_oplist_mac32_per_unit": W_UNIT,
        "achieved_reference_oplist": W_UNIT * U / (step_ms * 1e-3) / 1e12, "frac_reference_oplist": W_UNIT * U / (step_ms * 1e-3) / peak_mac,
        "note": "reference-oplist figures exceed the executed ones because of the declared value-preserving shortcuts (DESIGN.md section 4)"}
    roofline["hbm"] = {"achieved": BYTES_PER_UNIT * U / (step_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                       "frac": BYTES_PER_UNIT * U / (step_ms * 1e-3) / 1e9 / hbm_peak,
                       "peak_source": "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback"}
    roofline["kernels"] = prof

    cpu = None
    if not args.no_cpu_baseline:
        from oracle import twin
        n_cpu, v1, _ = cpu_sample_sessions(keysets, threads, 12.0)      # about 12 s of wall time on this box
        v, dt = cpu_phases(keysets, n_cpu, threads)
        cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{2 * n_cpu} phases ({n_cpu} sessions) of the same workload in {dt:.1f} s on a persistent pool of {threads} threads (oracle/gg20_twin.c: the "
                         f"reference's scalar call sequence, GMP {twin.lib().oracle_gmp_version().decode()} + OpenSSL, {cpu_model()}); single thread: {v1:.2f} phases/s"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": config_dict(world),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(rnd.nbytes + sess.nbytes), "d2h_bytes_per_step": int(world * U * REC),
                "ms_per_step": e2e_ms / args.steps, "call": "tecdsa_gg20_offline_records(TECDSA_HOST)"},
        "gpu_launches": int(launches),
        "sessions_per_s": value / 2,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "clocks": clocks,
        "parity": {"all_units_ok": all_ok, "host_and_device_paths_agree": paths_agree, "gather_consistent": gather_ok, **(parity or {})},
        "modexp": modexp,
    }
    print(json.dumps(line), flush=True)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if comm is not None:
        eng.nccl_comm_destroy(comm)
    if world > 1:
        dist.destroy_process_group()
    p = line["parity"]
    if not (p["all_units_ok"] and p["host_and_device_paths_agree"] and p["gather_consistent"] and p.get("units_match_cpu_twin") and p.get("signatures_verify")):
        raise SystemExit("parity check FAILED: " + json.dumps(p))
    if modexp is not None and ("error" in modexp or not modexp.get("parity_ok", True)):
        raise SystemExit("modexp block failed: " + json.dumps(modexp))


def parity_block(keysets, sess, rnd, records, sig, m_int, threads):
    """256 units (128 sessions spread over the batch) against the oracle's C twin, and their signatures against OpenSSL."""
    from cryptography.hazmat.primitives import hashes
    from cryptography.hazmat.primitives.asymmetric import ec, utils
    from oracle import gg20_oracle as o
    from oracle import twin
    n_sessions = sess.shape[0]
    pick = np.unique(np.linspace(0, n_sessions - 1, min(128, n_sessions)).astype(np.int64))
    units = np.stack([2 * pick, 2 * pick + 1], axis=1).reshape(-1)
    res = twin.offline_batch(twin.KeyTables(keysets), sess[pick], rnd[units], threads)

    def be(limbs):            # [n][8] little-endian limbs -> [n][32] big-endian bytes
        return np.ascontiguousarray(limbs[:, ::-1]).astype(">u4").view(np.uint8).reshape(limbs.shape[0], 32)

    got = records[units]
    ok = bool((res.status == 0).all()) and bool((got[:, 0] == 0).all())
    ok = ok and np.array_equal(got[:, 164:196], be(res.digest))
    ok = ok and np.array_equal(got[:, 34:66], be(res.sigma)) and np.array_equal(got[:, 66:98], be(res.k))
    ok = ok and np.array_equal(got[:, 2:34], be(res.R[:, :8])) and np.array_equal(got[:, 1], 2 + (res.R[:, 8] & 1).astype(np.uint8))
    ok = ok and np.array_equal(got[:, 99:131], be(res.t_vec[:, :8])) and np.array_equal(got[:, 132:164], be(res.t_vec[:, 16:24]))
    # signatures: (r, s) of every sampled session verifies under OpenSSL against the key set's public key y
    sig_ok = True
    digest = m_int.to_bytes(32, "big")
    for s in pick:
        y = keysets[int(sess[s, 0])][0].y_sum_s
        pub = ec.EllipticCurvePublicNumbers(y[0], y[1], ec.SECP256K1()).public_key()
        r = int.from_bytes(sig["r"][s].tobytes(), "little"); sv = int.from_bytes(sig["s"][s].tobytes(), "little")
        try:
            pub.verify(utils.encode_dss_signature(r, sv), digest, ec.ECDSA(utils.Prehashed(hashes.SHA256())))
        except Exception:
            sig_ok = False
        sig_ok = sig_ok and o.ecdsa_verify(r, sv, y, m_int) and sv <= Q - sv
    return {"units_compared_with_cpu_twin": int(len(units)), "units_match_cpu_twin": bool(ok), "signatures_checked": int(len(pick)),
            "signatures_verify": bool(sig_ok), "checker": "oracle/gg20_twin.c (GMP + OpenSSL) bit-compare of status, R, sigma_i, k_i, t_vec, transcript digest; "
                                                          "ECDSA verify under OpenSSL (`cryptography`) and the oracle's in-tree `verify`"}


if __name__ == "__main__":
    main()
