#!/usr/bin/env python3
"""bench.py — headline benchmark of the B200 validation hot path.

Workload (BASELINE.json configs[1]): batch-verify 1 Mi standalone BIP-340 Schnorr (pubkey, msg, sig)
triples per GPU; ~98 % valid, ~1 % single-bit corruptions, ~1 % adversarial encodings
(rusty_kaspa_b200/workload.py).  One "step" = one pass of the verify kernel over the rank's batch,
followed (N > 1) by the NCCL all-gather of the per-shard validity bitmaps.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--n ITEMS] [--dump-outputs DIR]

N > 1 is launched by torchrun, one rank per GPU; shards are independent (weak scaling: every rank
verifies its own 1 Mi triples), the only collective is the bitmap all-gather.

Timing rules followed: W >= 3 warm-ups; L2 flushed (256 MiB write) before every timed step and the
inputs (128 MiB) exceed the 126 MB L2 anyway; CUDA events on the stream the kernels are launched
on, per step, summed; max over ranks; barrier + synchronize on both sides; clocks sampled with
nvidia-smi during the timed region.

--impl reference times the CPU path instead: the reference's own implementation cannot be built
here (no Rust toolchain, libsecp256k1 not vendored; DESIGN.md), so this arm runs the C restatement
of it (oracle/, kind "port") on all host threads over a bounded sample per step.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_DEFAULT = 1 << 20
ALG_BYTES_PER_VERIFY = 129  # 32 pk + 32 msg + 64 sig read, 1 status byte written (SURVEY.md §8d)
METRIC = "schnorr_sig_verifies_per_sec"
UNIT = "verifies/s"
DUMP_MAX_BYTES = 60 << 20  # --dump-outputs: under 64 MB in all with the .npy headers


def dump_outputs(out_dir, arrays):
    """--dump-outputs: writes each array as out_dir/<name>.npy in float32, so that two builds run with the same arguments (hence the
    same seeded inputs) can be compared output for output.  Beyond DUMP_MAX_BYTES in all, every array is cut to the same fixed,
    seeded sample of its elements (sorted indices from default_rng(0)), so the files stay comparable between runs."""
    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.size for a in arrays.values())
    for name, a in arrays.items():
        a = a.reshape(-1)
        k = min(a.size, a.size * (DUMP_MAX_BYTES // 4) // total)
        if k < a.size:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, k, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


# ------------------------------------------------------------------------------------------------
def load_oracle():
    """CPU oracle — used ONLY by the cpu_baseline leg and --impl reference (never on the GPU path)."""
    path = os.path.join(ROOT, "oracle", "libkaspa_oracle.so")
    if not os.path.exists(path):
        subprocess.run(["make", "-C", os.path.join(ROOT, "oracle")], check=True, capture_output=True)
    lib = ctypes.CDLL(path)
    lib.ok_secp_init()
    return lib


def oracle_verify(lib, pk, msg, sig, threads):
    n = len(pk)
    st = np.zeros(n, dtype=np.uint8)
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    t0 = time.perf_counter()
    # the speed-oriented port (oracle/ok_secp_fast.c: GLV + wNAF + effective-affine tables; verdicts identical to the plain checker's)
    lib.ok_schnorr_verify_batch_fast(vp(pk), vp(msg), vp(sig), ctypes.c_size_t(n), vp(st), int(threads))
    return time.perf_counter() - t0, st


def cpu_quota():
    """(logical CPUs this process may run on, cgroup CPU quota in CPUs or None)"""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    q = None
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            q = int(quota) / int(period)
    except Exception:
        pass
    return n, q


def host_threads():
    """Threads for the CPU arm: all CPUs this process may run on, but no more than twice the container's CPU quota
    (cgroup cpu.max).  On the GPU boxes (128 logical CPUs, quota 16) 32 threads give 111 k verifies/s while 128 threads
    spend their time being throttled (87 k/s) — tools/cpu_threads.py."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(round(2 * int(quota) / int(period)))))
    except Exception:
        pass
    return n


class ClockSampler:
    """SM clock / power / throttle reasons of ONE GPU during the timed region (B200_PROFILING.md's clocks line).

    Sampled in-process through NVML (nvidia_ml_py), attached to this rank's GPU only and initialised in prepare() BEFORE the warm-up: spawning
    `nvidia-smi -lms` per rank at the start of the timed region - the round-1 form - makes eight NVML initialisations enumerate every GPU of
    the node while the steps run, which stalled rank 0's GPU by ~12 ms per step and WAS the N=8 scaling cliff (measured: 197.8 -> 277.3 M
    verifies/s at N=8 with nothing else changed, profiles/r02_scaling_n8.md).  nvidia-smi remains the fallback when NVML cannot be loaded;
    it is then started in prepare() as well and only rows that fall inside the timed region are kept."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, uuid=None, period_s=0.025):
        self.index, self.uuid, self.period = index, uuid, period_s
        self.rows = []          # (t, sm, max_sm, power_w, reasons-set)
        self.nvml = self.handle = self.proc = self.thread = None
        self.t_start = self.t_stop = None
        self.active = False
        self.how = None

    def prepare(self):
        """everything slow (NVML init / process start) happens here, outside the timed region"""
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if self.uuid:
                for cand in ("GPU-" + self.uuid, self.uuid):
                    try:
                        h = pynvml.nvmlDeviceGetHandleByUUID(cand)
                        break
                    except Exception:
                        h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)  # fail here rather than in the thread
            self.nvml, self.handle, self.how = pynvml, h, "nvml"
        except Exception:
            self.nvml = None
            try:
                self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                self.how = "nvidia-smi"
            except Exception:
                self.proc = None
        if self.nvml or self.proc:
            self.thread = threading.Thread(target=self._pump_nvml if self.nvml else self._pump_smi, daemon=True)
            self.alive = True
            self.thread.start()

    def start(self):
        if self.thread is None:
            self.prepare()
        self.t_start = time.perf_counter()
        self.active = True

    def _sample_nvml(self):
        n, h = self.nvml, self.handle
        sm = float(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM))
        mx = float(n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM))
        try:
            pw = n.nvmlDeviceGetPowerUsage(h) / 1000.0
        except Exception:
            pw = None
        try:
            mask = n.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        names = (("hw_slowdown", n.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", n.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", n.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", n.nvmlClocksEventReasonSwPowerCap))
        return sm, mx, pw, {k for k, bit in names if mask & bit}

    def _pump_nvml(self):
        while self.alive:
            if self.active:
                try:
                    self.rows.append((time.perf_counter(),) + self._sample_nvml())
                except Exception:
                    pass
            time.sleep(self.period)

    def _pump_smi(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(",")]
            if not self.active or len(f) < 7:
                continue
            try:
                row = (time.perf_counter(), float(f[0]), float(f[1]), float(f[2]))
            except ValueError:
                continue
            self.rows.append(row + ({name for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7])
                                     if v.lower().startswith("active")},))

    def stop(self):
        self.t_stop = time.perf_counter()
        if self.nvml and self.active and not self.rows:  # a timed region shorter than one period: one sample at its end
            try:
                self.rows.append((self.t_stop,) + self._sample_nvml())
            except Exception:
                pass
        self.active = False
        self.alive = False
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["neither NVML nor nvidia-smi available"]}
        rows = [r for r in self.rows if self.t_start is None or self.t_start <= r[0] <= self.t_stop]
        sm = [r[1] for r in rows]
        power = [r[3] for r in rows if r[3] is not None]
        reasons = set().union(*[r[4] for r in rows]) if rows else set()
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(r[2] for r in rows) if rows else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons), "sampler": self.how}


def measured_peak_hbm():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """CPU arm: the reference's path restated for the CPU (oracle/ok_secp_fast.c, kind "port": the reference itself is Rust + the C
    libsecp256k1 and cannot be built here) on all host threads, over the SAME workload as the GPU arm: every step verifies the full
    batch of args.n triples (same generator, same seed as rank 0 of the GPU arm)."""
    if rank != 0:
        return
    from rusty_kaspa_b200 import workload as W
    lib = load_oracle()
    threads = host_threads()
    logical, quota = cpu_quota()
    n = args.n
    pk, msg, sig, kind = W.schnorr_triples(n, seed=0x6B61737061)
    for _ in range(min(args.warmup, 1)):
        oracle_verify(lib, pk[:n // 16], msg[:n // 16], sig[:n // 16], threads)
    total = 0.0
    for _ in range(args.steps):
        dt, st = oracle_verify(lib, pk, msg, sig, threads)
        total += dt
    assert int((st == 1).sum()) == int((kind == 0).sum())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"status": st})
    value = n * args.steps / total
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64 limbs (256-bit modular integer)",
            "data": "synthetic", "config": {"workload": "1Mi standalone BIP-340 Schnorr triples per GPU, batch-verify (BASELINE configs[1]); "
                                                        "98% valid / 1% bit-flips / 1% adversarial; CPU arm: the full batch per step",
                                            "items_per_gpu_per_step": n, "items_per_step": n},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "logical_cpus": logical, "cgroup_cpu_quota": quota,
                             "per_quota_cpu": value / (quota or logical),
                             "sample": f"the full {n} triples per step x {args.steps} steps, oracle/ok_secp_fast.c (GLV + wNAF-5 + effective-affine tables + 8-bit generator comb, "
                                       f"4x64 limbs), {threads} pthreads with static chunks on {logical} logical CPUs under a cgroup quota of {quota} CPUs"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit_json_line(line)


# Issue cycles per Schnorr verify per SM sub-partition for the shipping kernel's instruction stream (DESIGN.md §4):
# 1.355e5 IMAD.WIDE x 4.3 cycles + 2.772e5 other instructions x 1 cycle, per warp of 32 verifies (ncu: 412.7 k thread instructions per verify
# in the final round-2 build, profiles/r02_schnorr_verify_ncu_summary.json - the multiply count is that of the unchanged field arithmetic,
# profiles/r01_schnorr_verify_ncu_summary.json; per-instruction costs, profiles/r01_pipe_microbench.txt).
ISSUE_CYCLES_PER_WARP_VERIFY = 1.355e5 * 4.3 + 2.772e5 * 1.0
SCHEDULERS = 148 * 4


def integer_issue_roofline(n_items, kernel_ms, clocks):
    mhz = (clocks or {}).get("sm_mhz") or 1965.0
    peak = SCHEDULERS * mhz * 1e6 * 32.0 / ISSUE_CYCLES_PER_WARP_VERIFY
    achieved = n_items / (kernel_ms * 1e-3)
    return {"bound": "integer issue (IMAD.WIDE 4.3 cyc, other 1 cyc per warp instruction per scheduler, measured)", "achieved": achieved,
            "peak": peak, "unit": "verifies/s", "frac": achieved / peak, "sm_mhz": mhz}


def measure_tx_validation(ctx, dev, n_txs, steps, mix=(1.0, 0.0, 0.0, 0.0), label="config 3"):
    """Secondary metric of BASELINE.json ("txs-validated/sec"): config-3-shaped window of independent
    1-in/2-out and 2-in/2-out P2PK Schnorr transactions validated against the GPU UTXO table by ONE
    kgv_validate_txs call (populate + context rules + sighash + verify + resolve), device-resident batch,
    then end to end with host arrays; followed by kgv_utxo_apply_accepted."""
    import ctypes as C
    import torch
    from rusty_kaspa_b200 import GpuUtxoSet, Params, TransactionValidator, simgen
    from rusty_kaspa_b200.txbatch import build_batch
    from rusty_kaspa_b200.validator import RESULT_DTYPE
    from rusty_kaspa_b200.verifier import _KgvTxBatch
    t0 = time.perf_counter()
    fkeys, fentries, txs = simgen.funded_window(n_txs, mix=mix)
    b = build_batch(txs)
    earr, earena = simgen.entries_to_arrays(fentries)
    gen_s = time.perf_counter() - t0
    n_sigs = int(b.n_inputs)
    us = GpuUtxoSet(ctx, 4 * len(fkeys))
    us.apply_diff(add_keys36=fkeys, add_entries=earr, add_bytes=earena)
    tv = TransactionValidator(ctx, Params(coinbase_maturity=100, storage_mass_parameter=simgen.DEFAULT_STORAGE_MASS_PARAMETER))
    res = tv.validate_transactions_in_parallel(us, b, 10)  # warm-up + correctness guard
    assert (res["status"] == 0).all(), "funded window must validate completely"
    # device-resident batch
    dt = [torch.from_numpy(a.view(np.uint8).reshape(-1)).to(dev) for a in (b.txs, b.inputs, b.outputs, b.arena)]
    dres = torch.empty(len(b.txs) * RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    cb = _KgvTxBatch(dt[0].data_ptr(), len(b.txs), dt[1].data_ptr(), len(b.inputs), dt[2].data_ptr(), len(b.outputs), None, dt[3].data_ptr(), len(b.arena))
    lib, h = ctx._lib, ctx._h
    stream = torch.cuda.current_stream(dev)
    call = lambda: ctx._check(lib.kgv_validate_txs(h, us._h, C.byref(cb), 10, 0, C.byref(tv.params), dres.data_ptr()))
    call(); stream.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        call()
    e1.record(stream)
    stream.synchronize()
    dev_s = e0.elapsed_time(e1) * 1e-3 / steps
    st = np.frombuffer(dres.cpu().numpy().tobytes(), dtype=RESULT_DTYPE)
    assert (st["status"] == 0).all()
    # K8: the MuHash half of validate_transactions_with_muhash_in_parallel for the same window (all accepted)
    dacc = torch.ones(len(b.txs), dtype=torch.uint8, device=dev)
    dmu = torch.zeros(768, dtype=torch.uint8, device=dev)
    mu_call = lambda: ctx._check(lib.kgv_muhash_txs(h, us._h, C.byref(cb), dacc.data_ptr(), 10, dmu.data_ptr(), dmu.data_ptr() + 384))
    mu_call(); stream.synchronize()
    m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    m0.record(stream)
    for _ in range(steps):
        mu_call()
    m1.record(stream)
    stream.synchronize()
    mu_s = m0.elapsed_time(m1) * 1e-3 / steps
    mu_dev = dmu.cpu().numpy().tobytes()
    from rusty_kaspa_b200 import MuHash
    mu_host = MuHash.from_transactions(ctx, b, np.ones(len(b.txs), dtype=np.uint8), 10, utxo_set=us)
    assert mu_dev[:384] == mu_host.numerator and mu_dev[384:] == mu_host.denominator and mu_host.numerator != (1).to_bytes(384, "little")
    # end to end from host memory: the batch arrays are page-locked first (what a host integration would allocate them as)
    cudart = torch.cuda.cudart()
    pinned = []
    for a in (b.txs, b.inputs, b.outputs, b.arena):
        if a.nbytes and int(cudart.cudaHostRegister(a.ctypes.data, a.nbytes, 0)) == 0:
            pinned.append(a)
    for _ in range(2):
        tv.validate_transactions_in_parallel(us, b, 10)
    t0 = time.perf_counter()
    for _ in range(steps):
        tv.validate_transactions_in_parallel(us, b, 10)
    e2e_s = (time.perf_counter() - t0) / steps
    for a in pinned:
        cudart.cudaHostUnregister(a.ctypes.data)
    t0 = time.perf_counter()
    us.add_transactions(b, np.ones(len(txs), dtype=np.uint8), 10)
    n_after = us.count()
    apply_s = time.perf_counter() - t0
    assert n_after == 2 * len(txs)
    us.close()
    return {"workload": label + ": window of independent txs (50% 1-in/2-out, 50% 2-in/2-out), spent-output mix (P2PK Schnorr, P2PK ECDSA, P2SH 2-of-3 Schnorr, P2SH 2-of-3 ECDSA) = "
                        + str(tuple(mix)) + ", vs GPU UTXO table, one kgv_validate_txs call",
            "n_txs": len(txs), "n_sig_checks": n_sigs, "txs_per_s": len(txs) / dev_s, "sig_checks_per_s": n_sigs / dev_s,
            "e2e_txs_per_s": len(txs) / e2e_s, "e2e_h2d_bytes": int(b.txs.nbytes + b.inputs.nbytes + b.outputs.nbytes + b.arena.nbytes),
            "apply_accepted_ms": apply_s * 1e3, "ms_per_call": dev_s * 1e3,
            "muhash": {"what": "kgv_muhash_txs: MuHash::from_transaction of every tx of the window, combined (K8)", "elements": int(b.n_inputs + len(b.outputs)),
                       "ms_per_call": mu_s * 1e3, "u3072_mults_per_s": (int(b.n_inputs + len(b.outputs)) - 2) / mu_s,
                       "txs_per_s_validate_plus_muhash": len(txs) / (dev_s + mu_s)},
            "generation_s": round(gen_s, 1)}


def measure_dag_replay(ctx, dev, n_blocks, tpb, window, cpu_budget_s, mix=(1.0, 0.0, 0.0, 0.0), label="config 3", seed=0x6B61737061, frac_invalid=0.01):
    """BASELINE.json's second headline, txs-validated/s ON A DAG (configs[2]): a generated simpa-shaped chain of n_blocks blocks
    (<= tpb transactions each, 50 % 1-in/2-out + 50 % 2-in/2-out, coinbase maturity 200 as in simpa/src/main.rs:204, ~1 % deliberately
    invalid transactions) replayed IN ORDER against the GPU UTXO table (2^24 slots) by kgv_replay_window, `window` blocks per call:
    what calculate_utxo_state does block by block (utxo_validation.rs:110-173) and simpa times (simpa/src/main.rs:454-460).
    Reported: device-resident batches (CUDA events around all calls), end to end from page-locked host arrays (H2D of every window,
    D2H of every verdict inside the wall-clock region), and the CPU path (oracle/ok_state_replay: the restated rayon path with a
    persistent thread pool) on a time-bounded prefix of the SAME blocks, whose verdicts must equal the GPU's."""
    import ctypes as C
    import torch
    from rusty_kaspa_b200 import GpuUtxoSet, Params, simgen
    from rusty_kaspa_b200.replay import REPLAY_BLOCK_DTYPE, ReplayStats
    from rusty_kaspa_b200.validator import RESULT_DTYPE
    from rusty_kaspa_b200.verifier import _KgvTxBatch
    t0 = time.perf_counter()
    gen = simgen.FastDag(seed=seed, n_keys=1024, n_nonces=4096, mix=mix, frac_two_inputs=0.5, frac_invalid=frac_invalid, coinbase_outputs=16)
    wins = []
    done = 0
    while done < n_blocks:
        k = min(window, n_blocks - done)
        gen.generate(k, tpb)
        b, first, pov = gen.take()
        arr = np.zeros(k, dtype=REPLAY_BLOCK_DTYPE)
        arr["first_tx"], arr["n_txs"], arr["pov_daa_score"], arr["flags"] = first[:-1], np.diff(first), pov, 1
        wins.append((b, arr, first, pov))
        done += k
    cnt = gen.counts()
    n_txs = sum(len(w[0].txs) for w in wins)
    n_user = n_txs - n_blocks
    n_sigs_gen = cnt["n_signatures"]
    gen_s = time.perf_counter() - t0
    prm = Params(coinbase_maturity=gen.maturity, storage_mass_parameter=gen.C)
    lib, h = ctx._lib, ctx._h
    stream = torch.cuda.current_stream(dev)

    def c_batch(ptrs, b):
        return _KgvTxBatch(ptrs[0], len(b.txs), ptrs[1], len(b.inputs), ptrs[2], len(b.outputs), None, ptrs[3], len(b.arena))

    # ---- device-resident windows
    us = GpuUtxoSet(ctx, 1 << 24)
    dwins = []
    for b, arr, _, _ in wins:
        ts = [torch.from_numpy(a.view(np.uint8).reshape(-1)).to(dev) for a in (b.txs, b.inputs, b.outputs, b.arena)]
        dres = torch.empty(len(b.txs) * 16, dtype=torch.uint8, device=dev)
        dwins.append((ts, dres, c_batch([t.data_ptr() for t in ts], b)))
    # warm-up: the whole chain once against a scratch table (untimed) - it sizes every per-call buffer of the context (the first windows of a
    # cold context would otherwise pay cudaMalloc inside the timed region: +-25 % on a leg of only 3-4 windows)
    scratch = GpuUtxoSet(ctx, 1 << 24)
    for (b, arr, _, _), (ts, dres, cb) in zip(wins, dwins):
        ctx._check(lib.kgv_replay_window(h, scratch._h, C.byref(cb), arr.ctypes.data, len(arr), C.byref(prm), dres.data_ptr(), None, None))
    ctx.synchronize()
    scratch.close()
    stream.synchronize()
    l0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for (b, arr, _, _), (ts, dres, cb) in zip(wins, dwins):
        ctx._check(lib.kgv_replay_window(h, us._h, C.byref(cb), arr.ctypes.data, len(arr), C.byref(prm), dres.data_ptr(), None, None))
    e1.record(stream)
    stream.synchronize()
    dev_s = e0.elapsed_time(e1) * 1e-3
    launches = ctx.launch_count - l0
    dev_status = [np.frombuffer(d[1].cpu().numpy().tobytes(), dtype=RESULT_DTYPE)["status"].copy() for d in dwins]
    n_table = us.count()
    assert n_table == cnt["n_utxos"], (n_table, cnt["n_utxos"])
    us.close()
    del dwins
    # ---- end to end from page-locked host arrays
    cudart = torch.cuda.cudart()
    # page-locked copies of the windows (cudaHostAlloc through torch: pinning the generator's arrays in place with cudaHostRegister ran into the
    # box's locked-memory limit beyond a few hundred MB, and an array that silently stays pageable uploads at a fraction of the PCIe rate)
    pinned, n_pin_failed = [], 0
    hbufs = []
    for b, arr, _, _ in wins:
        row = []
        for a in (b.txs, b.inputs, b.outputs, b.arena):
            src = torch.from_numpy(a.view(np.uint8).reshape(-1))
            try:
                t = src.pin_memory() if a.nbytes else src
            except Exception:
                t, n_pin_failed = src, n_pin_failed + 1
            row.append(t)
        hbufs.append(row)
    us = GpuUtxoSet(ctx, 1 << 24)
    hres_t = []
    for w in wins:
        t = torch.zeros(len(w[0].txs) * RESULT_DTYPE.itemsize, dtype=torch.uint8)
        try:
            t = t.pin_memory()
        except Exception:
            n_pin_failed += 1
        hres_t.append(t)
    hres = [t.numpy().view(RESULT_DTYPE) for t in hres_t]
    st = ReplayStats()
    n_acc = n_sig = 0
    h2d = 0
    t0 = time.perf_counter()
    cbs = [c_batch([t.data_ptr() for t in row], w[0]) for row, w in zip(hbufs, wins)]
    for wi, ((b, arr, _, _), r) in enumerate(zip(wins, hres)):
        cb = cbs[wi]
        if wi + 1 < len(wins):  # the next window's upload rides on a side stream under this window's compute (kgv_batch_prefetch)
            ctx._check(lib.kgv_batch_prefetch(h, C.byref(cbs[wi + 1])))
        ctx._check(lib.kgv_replay_window(h, us._h, C.byref(cb), arr.ctypes.data, len(arr), C.byref(prm), r.ctypes.data, None, C.byref(st)))
        n_acc += int(st.n_accepted); n_sig += int(st.n_sig_checks)
        h2d += b.txs.nbytes + b.inputs.nbytes + b.outputs.nbytes + b.arena.nbytes
    e2e_s = time.perf_counter() - t0
    for a in pinned:
        cudart.cudaHostUnregister(a.ctypes.data)
    assert n_acc == n_user - cnt["n_invalid"], (n_acc, n_user, cnt["n_invalid"])
    assert us.count() == cnt["n_utxos"]
    for a, r in zip(dev_status, hres):
        assert (a == r["status"]).all()
    us.close()
    # ---- the CPU path beside it: same blocks, time-bounded prefix, verdicts must be identical
    cpu = None
    if cpu_budget_s > 0:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_tx
        ora = load_oracle()
        ora.ok_use_fast_verify(1)  # baseline mode: signature checks through the fast port (identical verdicts)
        threads = host_threads()
        ost = oracle_tx.State(ora)
        op = oracle_tx.params(coinbase_maturity=gen.maturity, storage_mass_parameter=gen.C)
        c_txs = c_blocks = 0
        c_s = 0.0
        for (b, arr, first, pov), r in zip(wins, hres):
            t0 = time.perf_counter()
            cres, _ = oracle_tx.state_replay(ost, b, first, pov, op, threads=threads)
            c_s += time.perf_counter() - t0
            assert (cres["status"] == r["status"]).all() and (cres["script_err"] == r["script_err"]).all(), "CPU path and GPU replay disagree"
            c_txs += len(b.txs) - len(pov); c_blocks += len(pov)
            if c_s > cpu_budget_s:
                break
        ost.close()
        ora.ok_use_fast_verify(0)
        cpu = {"value": c_txs / c_s, "unit": "txs/s", "cores": threads, "kind": "port",
               "sample": f"first {c_blocks} blocks ({c_txs} non-coinbase txs) of the same chain, oracle/ok_state_replay (validate in parallel on a persistent pool of {threads} "
                         f"pthreads, accept, commit, block after block); verdicts identical to the GPU's", "seconds": round(c_s, 2)}
    gen.close()
    return {"workload": f"{label}: generated chain of {n_blocks} blocks, <= {tpb} txs/block (50% 1-in/2-out, 50% 2-in/2-out), spent-output mix (P2PK Schnorr, P2PK ECDSA, "
                        f"P2SH 2-of-3 Schnorr, P2SH 2-of-3 ECDSA) = {tuple(mix)}, ~{frac_invalid:.0%} invalid, replayed in order against a 2^24-slot GPU UTXO table, "
                        f"kgv_replay_window over {window} blocks per call",
            "n_blocks": n_blocks, "n_txs": n_user, "n_sig_checks": n_sig, "n_accepted": n_acc, "window_blocks": window,
            "txs_per_s": n_user / dev_s, "blocks_per_s": n_blocks / dev_s, "sig_checks_per_s": n_sig / dev_s, "ms_total": dev_s * 1e3, "gpu_launches": int(launches),
            "e2e_txs_per_s": n_user / e2e_s, "e2e_sig_checks_per_s": n_sig / e2e_s, "e2e_h2d_bytes": int(h2d), "e2e_d2h_bytes": int(16 * n_txs), "e2e_arrays_not_page_locked": n_pin_failed,
            "e2e_how": "per window: kgv_batch_prefetch of the NEXT window (checks + upload on a worker thread / side stream), kgv_replay_window of this one from page-locked host arrays, verdicts to host memory",
            "cpu_baseline": cpu, "generation_s": round(gen_s, 1), "generator_signatures": n_sigs_gen}


def measure_ecdsa(ctx, dev, stream, n, steps):
    """Secondary: kgv_ecdsa_verify (33-byte compressed keys, low-S rule, tri-state verdicts), device-resident triples."""
    import torch
    from rusty_kaspa_b200 import workload as W
    t0 = time.perf_counter()
    pk, msg, sig, kind = W.ecdsa_triples(1 << 14, seed=0x45434453, n_keys=4096, n_nonces=4096)
    pk, msg, sig, kind = W.tile_triples(pk, msg, sig, kind, n)
    gen_s = time.perf_counter() - t0
    dpk, dmsg, dsig = (torch.from_numpy(a).to(dev) for a in (pk, msg, sig))
    dst = torch.empty(n, dtype=torch.uint8, device=dev)
    for _ in range(2):
        ctx.verify_ecdsa_batch(dpk, dmsg, dsig, n=n, status=dst)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        ctx.verify_ecdsa_batch(dpk, dmsg, dsig, n=n, status=dst)
    e1.record(stream)
    stream.synchronize()
    s = e0.elapsed_time(e1) * 1e-3 / steps
    st = dst.cpu().numpy()
    assert int((st == 1).sum()) == int((kind == 0).sum()) and not (st[kind != 0] == 1).any()
    return {"what": "kgv_ecdsa_verify, device-resident", "n": n, "verifies_per_s": n / s, "ms_per_call": s * 1e3, "generation_s": round(gen_s, 1)}


def measure_utxo_table(ctx, dev, stream, peak_gbs):
    """K5: the GPU UTXO table on its own: 4 Mi entries in a 16 Mi-slot (2 GiB) table; every timed call looks up a DIFFERENT random
    permutation of all 4 Mi entries (occupied slots = 512 MiB, four times L2), keys and results device-resident; then erase / re-insert of 1 Mi
    entries per call (kgv_utxo_apply_diff, device arrays).  Algorithmic bytes per lookup (SURVEY §8d): 36 B key + one 128 B slot = 164 B
    (+ 33 B of results written).  The probe itself reads only the first 64 bytes of a slot (two LDG.256), so DRAM moves LESS than that."""
    import torch
    from rusty_kaspa_b200 import GpuUtxoSet
    from rusty_kaspa_b200.txbatch import ENTRY_DTYPE
    n_ent = 1 << 22
    n = n_ent
    rng = np.random.default_rng(7)
    keys = rng.integers(0, 256, size=(n_ent, 36), dtype=np.uint8)
    ent = np.zeros(n_ent, dtype=ENTRY_DTYPE)
    ent["amount"] = rng.integers(1, 1 << 40, size=n_ent)
    ent["script_off"] = (np.arange(n_ent, dtype=np.uint64) * 34 % (1 << 20)).astype(np.uint32)
    ent["script_len"] = 34
    arena = rng.integers(0, 256, size=(1 << 20) + 64, dtype=np.uint8)
    us = GpuUtxoSet(ctx, 4 * n_ent)
    t0 = time.perf_counter()
    us.apply_diff(add_keys36=keys, add_entries=ent, add_bytes=arena)
    ctx.synchronize()
    ins_s = time.perf_counter() - t0
    assert us.count() == n_ent
    reps = 4
    dkeys = torch.from_numpy(keys).to(dev)
    dks = [dkeys[torch.randperm(n_ent, device=dev)].contiguous() for _ in range(reps + 1)]
    de = torch.empty(n * ENTRY_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    df = torch.empty(n, dtype=torch.uint8, device=dev)
    call = lambda dk: ctx._check(ctx._lib.kgv_utxo_lookup(ctx._h, us._h, dk.data_ptr(), n, de.data_ptr(), None, 0, df.data_ptr()))
    call(dks[reps]); stream.synchronize()
    assert int(df.sum().item()) == n
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for r in range(reps):
        call(dks[r])
    e1.record(stream)
    stream.synchronize()
    s = e0.elapsed_time(e1) * 1e-3 / reps
    # erase + re-insert 1 Mi entries per call, device arrays
    m = 1 << 20
    sel = torch.randperm(n_ent, device=dev)[:m]
    dk1 = dkeys[sel].contiguous()
    dent = torch.from_numpy(ent.view(np.uint8).reshape(-1, ENTRY_DTYPE.itemsize)).to(dev)[sel].contiguous()
    darena = torch.from_numpy(arena).to(dev)
    drs, das = torch.empty(m, dtype=torch.uint8, device=dev), torch.empty(m, dtype=torch.uint8, device=dev)
    lib, h = ctx._lib, ctx._h
    erase = lambda: ctx._check(lib.kgv_utxo_apply_diff(h, us._h, dk1.data_ptr(), m, drs.data_ptr(), None, None, None, 0, 0, None))
    insert = lambda: ctx._check(lib.kgv_utxo_apply_diff(h, us._h, None, 0, None, dk1.data_ptr(), dent.data_ptr(), darena.data_ptr(), len(arena), m, das.data_ptr()))
    erase(); insert(); stream.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    t_er = t_in = 0.0
    for _ in range(3):
        ev[0].record(stream); erase(); ev[1].record(stream); insert(); ev[2].record(stream); stream.synchronize()
        t_er += ev[0].elapsed_time(ev[1]) * 1e-3 / 3; t_in += ev[1].elapsed_time(ev[2]) * 1e-3 / 3
    assert int(drs.sum().item()) == m and us.count() == n_ent
    us.close()
    gbs = n * 164 / s * 1e-9
    return {"what": "k_utxo_lookup, 4 Mi random hits per call (every entry of a 2 GiB table, new order every call; device-resident keys/results)",
            "lookups_per_s": n / s, "ms_per_call": s * 1e3, "insert_4Mi_entries_host_arrays_ms": ins_s * 1e3,
            "erase_per_s": m / t_er, "insert_per_s": m / t_in,
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak_gbs, "unit": "GB/s", "frac": gbs / peak_gbs if peak_gbs else None,
                         "bytes_per_lookup": 164, "note": "SURVEY §8d bytes (36 B key + one 128 B slot); 33 more bytes per lookup are written (entry + found flag); "
                                                          "the probe reads 64 of the slot's 128 bytes"},
            "roofline_erase": {"achieved": m * 164 / t_er * 1e-9, "peak": peak_gbs, "unit": "GB/s", "frac": m * 164 / t_er * 1e-9 / peak_gbs if peak_gbs else None,
                               "bytes_per_op": 164},
            "roofline_insert": {"achieved": m * (36 + 32 + 34 + 128) / t_in * 1e-9, "peak": peak_gbs, "unit": "GB/s",
                                "frac": m * (36 + 32 + 34 + 128) / t_in * 1e-9 / peak_gbs if peak_gbs else None, "bytes_per_op": 230}}


def measure_small_batches(ctx):
    """Mempool-shaped use (SURVEY §8f-3): latency of ONE kgv_validate_txs call on small host-resident batches
    (upload + populate + context rules + scripts + verdict download), median of 20 calls."""
    from rusty_kaspa_b200 import GpuUtxoSet, Params, TransactionValidator, simgen
    from rusty_kaspa_b200.txbatch import build_batch
    fkeys, fentries, txs = simgen.funded_window(256, n_keys=64, n_nonces=64)
    earr, earena = simgen.entries_to_arrays(fentries)
    us = GpuUtxoSet(ctx, 4096)
    us.apply_diff(add_keys36=fkeys, add_entries=earr, add_bytes=earena)
    tv = TransactionValidator(ctx, Params(coinbase_maturity=100, storage_mass_parameter=simgen.DEFAULT_STORAGE_MASS_PARAMETER))
    out = {}
    for n in (1, 16, 256):
        b = build_batch(txs[:n])
        ts = []
        for _ in range(23):
            t0 = time.perf_counter()
            res = tv.validate_transactions_in_parallel(us, b, 10)
            ts.append(time.perf_counter() - t0)
        assert (res["status"] == 0).all()
        out[str(n)] = round(sorted(ts[3:])[10] * 1e3, 3)
    us.close()
    return {"what": "median wall-clock ms of one kgv_validate_txs call, host arrays in, verdicts out", "ms_by_batch_size": out}


def merge_clocks(per_rank):
    """clocks of every rank -> one record: the LOWEST median SM clock, the union of throttle reasons"""
    rows = [c for c in per_rank if c]
    if not rows:
        return None
    sm = [c["sm_mhz"] for c in rows if c.get("sm_mhz")]
    out = dict(rows[0])
    out["sm_mhz"] = min(sm) if sm else None
    out["sm_mhz_per_rank"] = [c.get("sm_mhz") for c in rows]
    if any("kernel_ms" in c for c in rows):
        out["kernel_ms_per_rank"] = [c.get("kernel_ms") for c in rows]
        out["step_ms_per_rank"] = [c.get("step_ms") for c in rows]
        out.pop("kernel_ms", None); out.pop("step_ms", None); out.pop("timeline", None)
        if any(c.get("timeline") for c in rows):
            out["timeline_per_rank"] = [c.get("timeline") for c in rows]
    out["power_w_max_per_rank"] = [c.get("power_w_max") for c in rows]
    out["reasons"] = sorted(set(r for c in rows for r in (c.get("reasons") or [])))
    out["ranks_sampled"] = len(rows)
    return out


def measure_dag_replay_sharded(ctx, dev, comm, rank, world, n_blocks, tpb, window):
    """BASELINE configs[4]: the IBD-shaped replay with the signature batches sharded over the GPUs.  Every rank generates the SAME chain (same
    seed) window by window (streaming: bounded memory; generation is outside the timed region), replays each window against its own replica
    of the UTXO table with kgv_set_sharding on - each rank verifies 1/N of the candidate (signature, key) pairs, the verdict bytes are
    exchanged through the communicator, scripts are resolved and the in-order pass runs identically everywhere.  Time = sum over windows of
    the slowest rank's wall clock per window (a barrier before each window)."""
    import ctypes as C
    import torch
    import torch.distributed as dist
    from rusty_kaspa_b200 import GpuUtxoSet, Params, simgen
    from rusty_kaspa_b200.replay import REPLAY_BLOCK_DTYPE, ReplayStats
    from rusty_kaspa_b200.validator import RESULT_DTYPE
    from rusty_kaspa_b200.verifier import _KgvTxBatch
    gen = simgen.FastDag(seed=0x6B61737061, n_keys=1024, n_nonces=4096, frac_two_inputs=0.5, frac_invalid=0.01, coinbase_outputs=16)
    prm = Params(coinbase_maturity=gen.maturity, storage_mass_parameter=gen.C)
    us = GpuUtxoSet(ctx, 1 << 25)
    comm.shard_validation(True)
    lib, h = ctx._lib, ctx._h
    cudart = torch.cuda.cudart()
    st = ReplayStats()
    total_s = gen_s = pre_ms = ord_ms = 0.0
    n_txs = n_sig = n_acc = done = 0
    try:
        def make_window(k):
            """generate + page-lock one window (outside the timed region)"""
            nonlocal gen_s
            t0 = time.perf_counter()
            gen.generate(k, tpb)
            b, first, pov = gen.take()
            gen_s += time.perf_counter() - t0
            arr = np.zeros(k, dtype=REPLAY_BLOCK_DTYPE)
            arr["first_tx"], arr["n_txs"], arr["pov_daa_score"], arr["flags"] = first[:-1], np.diff(first), pov, 1
            res = np.zeros(len(b.txs), dtype=RESULT_DTYPE)
            pinned = [a for a in (b.txs, b.inputs, b.outputs, b.arena, res) if a.nbytes and int(cudart.cudaHostRegister(a.ctypes.data, a.nbytes, 0)) == 0]
            cb = _KgvTxBatch(b.txs.ctypes.data, len(b.txs), b.inputs.ctypes.data, len(b.inputs), b.outputs.ctypes.data, len(b.outputs), None, b.arena.ctypes.data, len(b.arena))
            return b, arr, res, pinned, cb, k

        cur = make_window(min(window, n_blocks))
        while cur is not None:
            b, arr, res, pinned, cb, k = cur
            nxt = make_window(min(window, n_blocks - done - k)) if done + k < n_blocks else None
            dist.barrier()
            t0 = time.perf_counter()
            if nxt is not None:  # the next window's upload overlaps this window's compute
                ctx._check(lib.kgv_batch_prefetch(h, C.byref(nxt[4])))
            ctx._check(lib.kgv_replay_window(h, us._h, C.byref(cb), arr.ctypes.data, k, C.byref(prm), res.ctypes.data, None, C.byref(st)))
            dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            total_s += float(dt.item())
            for a in pinned:
                cudart.cudaHostUnregister(a.ctypes.data)
            n_txs += len(b.txs) - k; n_sig += int(st.n_sig_checks); n_acc += int(st.n_accepted)
            pre_ms += float(st.pre_check_ms); ord_ms += float(st.in_order_ms)
            done += k
            cur = nxt
        cnt = gen.counts()
        assert n_acc == n_txs - cnt["n_invalid"] and us.count() == cnt["n_utxos"], (n_acc, n_txs, cnt)
        dig = torch.frombuffer(bytearray(us.digest()), dtype=torch.uint8).to(dev)
        alld = torch.zeros(32 * world, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(alld, dig)
        assert all(torch.equal(alld[:32], alld[32 * r:32 * r + 32]) for r in range(world)), "table replicas diverged"
    finally:
        comm.shard_validation(False)
        us.close(); gen.close()
    return {"workload": f"config 5 shape: generated chain of {n_blocks} blocks (<= {tpb} txs/block, mixed 1-/2-input P2PK Schnorr, ~1% invalid) replayed in order on every rank "
                        f"against its own 2^25-slot table replica, signature checks sharded over {world} GPUs (kgv_set_sharding), verdict bytes exchanged through the "
                        f"library communicator, kgv_replay_window over {window} blocks per call from page-locked host arrays, the next window's upload prefetched (kgv_batch_prefetch) inside the timed region",
            "n_blocks": n_blocks, "n_txs": n_txs, "n_sig_checks": n_sig, "n_gpus": world, "txs_per_s": n_txs / total_s, "blocks_per_s": n_blocks / total_s,
            "sig_checks_per_s": n_sig / total_s, "seconds": total_s,
            "device_ms_rank0": {"pre_check_sharded": round(pre_ms, 2), "in_order_replicated": round(ord_ms, 2),
                                "note": "device time of the two phases on rank 0 (kgv_replay_stats): the pre-check holds the sharded signature work, the in-order part is replicated; every replica still uploads the whole window (prefetched under the previous window's compute, kgv_batch_prefetch)"},
            "generation_s": round(gen_s, 1), "replicas_identical": True}


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import rusty_kaspa_b200 as rk
    from rusty_kaspa_b200 import workload as W

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — this benchmark has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    n = args.n
    # every rank owns its own shard of the global batch (weak scaling): different seed per rank
    t_gen = time.perf_counter()
    pk, msg, sig, kind = W.schnorr_triples(n, seed=0x6B61737061 + rank)
    gen_s = time.perf_counter() - t_gen
    expected_valid = int((kind == 0).sum())

    ctx = rk.GpuContext(local_rank)  # raises if libkgv.so / device is missing
    stream = torch.cuda.Stream(device=dev)
    ctx.use_stream(stream.cuda_stream)
    comm = None
    with torch.cuda.stream(stream):
        if world > 1:
            from rusty_kaspa_b200.comm import ShardComm
            # torch.distributed is the bootstrap only (NCCL id / peer handles); the data path is libkgv's own exchange
            comm = ShardComm.from_torch_distributed(ctx, slice_capacity=max(1 << 22, (n + 7) // 8 + 4096), nccl=args.collective == "nccl", peer=args.collective == "peer")
        dpk, dmsg, dsig = (torch.from_numpy(a).to(dev) for a in (pk, msg, sig))
        dst = torch.empty(n, dtype=torch.uint8, device=dev)
        nbm = 4 * ((n + 31) // 32)
        dbm = torch.empty(nbm, dtype=torch.uint8, device=dev)
        gathered = torch.empty(nbm * world, dtype=torch.uint8, device=dev) if world > 1 else None
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

        def exchange(mid=None):
            """every rank ends up with every shard's validity bitmap"""
            if world == 1:
                ctx.status_to_bitmap(dst, n=n, bitmap=dbm)
            elif args.collective == "peer":   # the bitmap kernel writes straight into every peer over NVLink, consumers wait on local flags
                e = comm.publish_bitmap(dst.data_ptr(), n)
                if mid is not None:
                    mid.record(stream)
                comm.wait(e, nbm, gathered.data_ptr())
            elif args.collective == "nccl":   # ncclAllGather called from the library
                ctx.status_to_bitmap(dst, n=n, bitmap=dbm)
                comm.allgather(dbm.data_ptr(), nbm, gathered.data_ptr())
            else:                             # torch.distributed (round-1 form, kept for comparison)
                ctx.status_to_bitmap(dst, n=n, bitmap=dbm)
                dist.all_gather_into_tensor(gathered, dbm)

        def step():
            ctx.verify_schnorr_batch(dpk, dmsg, dsig, n=n, status=dst)
            exchange()

        try:
            dev_uuid = str(torch.cuda.get_device_properties(dev).uuid)
        except Exception:
            dev_uuid = None
        sampler = ClockSampler(local_rank, dev_uuid)
        if not os.environ.get("KGV_BENCH_NO_SAMPLER"):  # (diagnosis only: the contract wants the clocks)
            sampler.prepare()                            # NVML attach happens here, before the warm-up
        for _ in range(max(args.warmup, 3)):
            step()
        stream.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if not os.environ.get("KGV_BENCH_NO_SAMPLER"):
            sampler.start()
        launches0 = ctx.launch_count
        evs = []
        for _ in range(args.steps):
            flush.fill_(1)  # L2 flush, outside the timed events
            e0, ek, ep, e1 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
            e0.record(stream)
            ctx.verify_schnorr_batch(dpk, dmsg, dsig, n=n, status=dst)
            ek.record(stream)
            exchange(ep)
            e1.record(stream)
            evs.append((e0, ek, e1, ep))
        stream.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        launches = ctx.launch_count - launches0
        clocks = sampler.stop()
        step_ms = [a.elapsed_time(c) for a, _, c, _ in evs]
        kern_ms = [a.elapsed_time(b) for a, b, _, _ in evs]
        # where a step's time goes on THIS rank: publish (own stores to every peer), wait (for the slowest peer), and the gap to the next step (L2 flush)
        timeline = None
        if world > 1 and args.collective == "peer":
            timeline = {"publish_ms": round(float(np.mean([b.elapsed_time(p) for _, b, _, p in evs])), 3),
                        "wait_collect_ms": round(float(np.mean([p.elapsed_time(c) for _, _, c, p in evs])), 3),
                        "gap_to_next_step_ms": round(float(np.mean([evs[i][2].elapsed_time(evs[i + 1][0]) for i in range(len(evs) - 1)])), 3) if len(evs) > 1 else None}
        total_ms = float(sum(step_ms))
        # correctness guard inside the bench: verdict counts must match the generator's ground truth
        st = dst.cpu().numpy()
        assert int((st == 1).sum()) == expected_valid, "GPU verdicts disagree with the generator's ground truth"
        assert not (st[kind != 0] == 1).any()
        if args.dump_outputs and rank == 0:  # the last timed step's verdicts and the bitmap every rank ends up with
            dump_outputs(args.dump_outputs, {"status": st, "bitmap": (gathered if world > 1 else dbm).cpu().numpy()})
        mine = np.zeros(nbm, dtype=np.uint8)
        pb = np.packbits((st == 1).astype(np.uint8), bitorder="little")
        mine[:len(pb)] = pb
        if world > 1:
            bm_all = gathered.cpu().numpy()
            assert (bm_all[rank * nbm:(rank + 1) * nbm] == mine).all()
            chk = torch.tensor([int(bm_all.astype(np.uint64).sum())], dtype=torch.int64, device=dev)
            lo, hi = chk.clone(), chk.clone()
            dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
            assert int(lo.item()) == int(hi.item()), "ranks hold different gathered bitmaps"

        # ---- end to end: HOST (pinned) buffers in, verdicts / gathered bitmap out, every step
        hpk, hmsg, hsig = (torch.from_numpy(a).pin_memory() for a in (pk, msg, sig))
        hst = torch.empty(n, dtype=torch.uint8).pin_memory()
        hall = torch.empty(nbm * world, dtype=torch.uint8).pin_memory() if world > 1 else None
        e2e_steps = max(2, min(args.steps, 5))

        def e2e_step():
            if world == 1:  # kgv_schnorr_verify with host pointers: chunked H2D overlapped with the verification, D2H of the verdicts
                ctx.verify_schnorr_batch(hpk.numpy(), hmsg.numpy(), hsig.numpy(), n=n, status=hst.numpy())
            else:           # device-pointer form with the caller's copies, so that the exchange sits inside the step: H2D, verify, exchange, D2H of the gathered bitmap
                dpk.copy_(hpk, non_blocking=True); dmsg.copy_(hmsg, non_blocking=True); dsig.copy_(hsig, non_blocking=True)
                ctx.verify_schnorr_batch(dpk, dmsg, dsig, n=n, status=dst)
                exchange()
                hall.copy_(gathered, non_blocking=True)
                stream.synchronize()
        for _ in range(2):
            e2e_step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        e2e_s = time.perf_counter() - t0
        if world == 1:
            assert int((hst.numpy() == 1).sum()) == expected_valid
        else:
            assert (hall.numpy()[rank * nbm:(rank + 1) * nbm] == mine).all()

        # ---- config 5: the DAG replay with the signature checks sharded over the ranks (kgv_set_sharding), table replicas
        rep5 = None
        if world > 1 and args.replay_blocks_multi > 0:
            rep5 = measure_dag_replay_sharded(ctx, dev, comm, rank, world, args.replay_blocks_multi, 150, args.replay_window)

    # max over ranks
    if isinstance(clocks, dict):  # per-rank device times next to the clocks they ran at (a slow GPU shows up here, not in the max)
        clocks = dict(clocks, kernel_ms=round(float(np.mean(kern_ms)), 3), step_ms=round(float(np.mean(step_ms)), 3), timeline=timeline)
    cl_all = [clocks]
    if world > 1:
        cl_all = [None] * world
        dist.all_gather_object(cl_all, clocks)
    if world > 1:
        t = torch.tensor([total_ms, e2e_s, float(sum(kern_ms))], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_s, kern_total_ms = (float(x) for x in t.tolist())
    else:
        kern_total_ms = float(sum(kern_ms))
    if comm is not None:
        comm.close()
    if rank != 0:
        return

    value = n * world * args.steps / (total_ms * 1e-3)
    e2e_value = n * world * e2e_steps / e2e_s
    kern_ms_avg = kern_total_ms / args.steps
    peak, peak_src = measured_peak_hbm()
    achieved = ALG_BYTES_PER_VERIFY * n / (kern_ms_avg * 1e-3) / 1e9
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "r02_schnorr_verify_ncu_summary.json")) as f:  # one `ncu --set full` capture at the bench size (1 Mi triples per launch)
            traffic = int(json.load(f).get("dram_bytes_per_launch"))
    except Exception:
        pass

    # ---- CPU baseline beside it: the oracle port on the host cores, bounded sample (rank 0, N=1 only)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        lib = load_oracle()
        threads = host_threads()
        sample = max(4096, min(n, 8192 * threads))
        oracle_verify(lib, pk[:sample // 8], msg[:sample // 8], sig[:sample // 8], threads)
        dt, cst = oracle_verify(lib, pk[:sample], msg[:sample], sig[:sample], threads)
        assert (cst == st[:sample]).all(), "CPU oracle and GPU verdicts differ"
        logical, quota = cpu_quota()
        cpu = {"value": sample / dt, "unit": UNIT, "cores": threads, "kind": "port", "logical_cpus": logical, "cgroup_cpu_quota": quota,
               "per_quota_cpu": sample / dt / (quota or logical),
               "sample": f"first {sample} triples of the same batch, oracle/ok_secp_fast.c (GLV + wNAF CPU port of the reference path), {threads} pthreads; verdicts identical to the GPU's"}

    txv = ecd = small = utx = rep = rep4 = None
    if world == 1 and args.replay_blocks > 0:
        with torch.cuda.stream(stream):
            rep = measure_dag_replay(ctx, dev, args.replay_blocks, 150, args.replay_window, 0 if args.no_cpu_baseline else 12.0)
            # BASELINE configs[3]: ECDSA + P2SH 2-of-3 multisig, 500 k transactions: 50 % P2PK-ECDSA, 25 % P2SH Schnorr 2-of-3, 25 % P2SH ECDSA 2-of-3,
            # ~1 % invalid of every class (wrong order => NullFail, corrupted => EvalFalse, high S, bad hash type, ...), as a chain replayed in order
            rep4 = measure_dag_replay(ctx, dev, max(64, int(args.replay_blocks * 0.35)), 150, args.replay_window, 0 if args.no_cpu_baseline else 8.0,
                                      mix=(0.0, 0.5, 0.25, 0.25), label="config 4", seed=0x4B475634)
    if world == 1 and args.tx_window > 0:
        with torch.cuda.stream(stream):
            txv = measure_tx_validation(ctx, dev, args.tx_window, max(2, min(args.steps, 5)))
            ecd = measure_ecdsa(ctx, dev, stream, min(n, 1 << 19), 3)
            small = measure_small_batches(ctx)
            utx = measure_utxo_table(ctx, dev, stream, peak)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32 limbs (256-bit modular integer)", "data": "synthetic",
            "config": {"workload": "1Mi standalone BIP-340 Schnorr triples per GPU, batch-verify (BASELINE configs[1]); "
                                   "98% valid / 1% bit-flips / 1% adversarial; bitmap pack" + (f" + exchange of the shard bitmaps ({args.collective})" if world > 1 else ""),
                       "collective": None if world == 1 else {"peer": "kgv_shard_publish_bitmap / kgv_shard_wait: peer stores over NVLink + epoch flags (libkgv)",
                                                              "nccl": "kgv_shard_allgather: ncclAllGather called from libkgv", "torch": "torch.distributed all_gather_into_tensor"}[args.collective],
                       "items_per_gpu_per_step": n, "input_bytes_per_gpu": 128 * n, "l2": "256 MiB flush write before every timed step; inputs 128 MiB > L2",
                       "parallelism": f"{world} independent shard(s), one process per GPU", "generation_s": round(gen_s, 1)},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "peak_source": peak_src, "kernel": "k_schnorr_verify", "kernel_ms": kern_ms_avg,
                         "note": "integer-issue bound by construction: 129 algorithmic bytes per verify vs 4.1e5 integer instructions; the binding roofline is integer_issue",
                         "integer_issue": integer_issue_roofline(n, kern_ms_avg, merge_clocks(cl_all))},
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 128 * n * world, "d2h_bytes_per_step": (n if world == 1 else nbm * world) * world,
                    "steps": e2e_steps,
                    "how": ("kgv_schnorr_verify through the C ABI with pinned host buffers: H2D + kernel + D2H + sync inside the timed region (host clock)" if world == 1 else
                            "per rank and step: H2D of the rank's triples from pinned memory, kgv_schnorr_verify (device pointers), the bitmap exchange, D2H of the gathered bitmap, sync "
                            "(host clock, max over ranks)")},
            "dag_replay": rep, "dag_replay_ecdsa_multisig": rep4, "dag_replay_sharded": rep5, "tx_validation": txv, "ecdsa": ecd, "small_batches": small,
            "utxo_table": utx, "gpu_launches": int(launches), "clocks": merge_clocks(cl_all)}
    emit_json_line(line)


_REAL_STDOUT = None


def _quiet_stdout():
    """Libraries (NCCL's version banner, torchrun notices) write to fd 1; the contract is ONE JSON line on stdout.
    Everything else is sent to stderr: fd 1 is pointed at fd 2 for the duration of the run and the JSON line is
    written to the saved descriptor at the end."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit_json_line(line):
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=N_DEFAULT, help="triples per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--collective", default="peer", choices=["peer", "nccl", "torch"], help="N > 1: how the shard bitmaps are exchanged")
    ap.add_argument("--replay-blocks-multi", type=int, default=100000, help="N > 1: blocks of the sharded DAG-replay leg (BASELINE configs[4]: 100k blocks; 0 = skip)")
    ap.add_argument("--replay-blocks", type=int, default=10000, help="blocks of the DAG-replay leg (BASELINE configs[2]: 10k blocks; 0 = skip)")
    ap.add_argument("--replay-window", type=int, default=1024, help="blocks per kgv_replay_window call")
    ap.add_argument("--tx-window", type=int, default=32768, help="transactions in the secondary txs-validated/s measurement (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs (per-triple verdicts, validity bitmap) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    _quiet_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
