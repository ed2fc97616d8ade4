#!/usr/bin/env python
"""bench.py -- ciphertexts/sec (encrypt + decrypt) of the batched NTRU engine, N=509 q=2048.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line on
rank 0.  A step = one pass of the hot path over one batch of synthetic input per GPU:
encrypt `rows` messages under one public key (full VerifyEncrypt witness), then decrypt those
ciphertexts under the private key (full VerifyDecrypt witness).

  value        whole-job ciphertexts/s with inputs resident in HBM (device-pointer C ABI)
  e2e          the same metric through the host-buffer C ABI (pinned host memory, H2D + D2H inside the timing)
  roofline     dominant kernel: algorithmic bytes / its CUDA-event time vs the measured HBM peak
  cpu_baseline the C restatement of the reference's algorithm (oracle/) on this box's host cores

  extras.configs  the other four BASELINE configs, each with its own CUDA-event time, roofline fraction and check:
               1 (N=167 same key), 3 (N=677 distinct valid keys), 4 (N=821, 2^20 rows SHARDED over the ranks: strong
               scaling), 5 (N=701, sum of 10 M rows sharded: peer-memory exchange inside the sum kernel and the NCCL
               all-reduce path, both checked against int64 column sums)

`--impl reference` times that CPU restatement alone (node does not exist in this image, so the
reference's own JavaScript cannot run; see DESIGN.md).

`--dump-outputs DIR` writes the arrays the last timed step returned (a seeded sample of 4096 rows of each) to
DIR/<name>.npy, so that two builds of the engine can be compared on identical inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

CONFIG = "hps509"
WORKLOAD = "NTRU-HPS N=509 q=2048 p=3, {rows} ciphertexts under one key per GPU, encrypt+decrypt, full witness"


def load_key():
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", f"{CONFIG}.npz")))
    return g


DUMP_ROWS = 4096     # rows of each output written by --dump-outputs: 6 arrays x (6 N + 4) float32 columns = 50 MB at N = 509


def dump_outputs(dirname, arrays):
    """Writes the same seeded sample of rows of every array in `arrays` (name -> device tensor of shape (B, width)) to
    dirname/<name>.npy as float32 (exact: every value is below 2^16).  The sample depends on B alone, and the bench's
    inputs are seeded, so two builds run with the same arguments can be compared output for output."""
    import torch
    B = next(iter(arrays.values())).shape[0]
    rows = np.sort(np.random.default_rng(0).choice(B, size=min(B, DUMP_ROWS), replace=False))
    os.makedirs(dirname, exist_ok=True)
    for name, t in arrays.items():
        x = t.index_select(0, torch.from_numpy(rows).to(t.device)).cpu().numpy()
        if x.dtype == np.int16:
            x = x.view(np.uint16)      # the ABI's uint16 coefficients travel in int16 tensors
        np.save(os.path.join(dirname, f"{name}.npy"), x.astype(np.float32))
    return {"dir": dirname, "rows": len(rows),
            "row_sample": "numpy default_rng(0).choice(rows_per_gpu, min(rows_per_gpu, 4096), replace=False), sorted; rank 0"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), "measured"
    return 6650.0, 1590.0, "fallback"


# ------------------------------------------------------------------------------------------------
# CPU baseline / reference arm (oracle = checker; here it is only timed, never part of the product)
# ------------------------------------------------------------------------------------------------
def cpu_sample(rows: int, g, threads: int = 0, seed: int = 1):
    """Times encrypt+decrypt of `rows` ciphertexts with the C restatement; returns (seconds, threads)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import c_oracle
    import ntru_oracle as o
    N, q, p, dr = int(g["N"]), int(g["q"]), int(g["p"]), int(g["dr"])
    rng = np.random.default_rng(seed)
    r = o.sample_ternary_rows(rows, N, dr, dr, rng)
    m = rng.integers(0, 2, size=(rows, N))
    nthreads = threads or c_oracle.num_threads()
    t0 = time.perf_counter()
    enc = c_oracle.encrypt_batch(g["h"], r, m, q, nthreads=nthreads)
    dec = c_oracle.decrypt_batch(g["f"], g["fp"], enc["value"], q, p, nthreads=nthreads)
    dt = time.perf_counter() - t0
    assert np.array_equal(dec["value"], m)
    return dt, nthreads


def cpu_baseline(g, target_s: float = 12.0):
    dt, nthreads = cpu_sample(64, g)
    rows = int(max(64, min(20000, 64 * target_s / max(dt, 1e-3))))
    rows = (rows // nthreads) * nthreads or nthreads
    dt, nthreads = cpu_sample(rows, g, seed=2)
    return {"value": rows / dt, "unit": "ciphertexts/s", "cores": nthreads, "kind": "port",
            "sample": f"{rows} ciphertexts encrypt+decrypt with witness, N=509 q=2048, "
                      f"C restatement of index.js (float64 FFT + long division), {nthreads} pthreads, {dt:.1f}s"}


def run_reference(args, rank):
    if rank != 0:
        return
    g = load_key()
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import c_oracle
    nthreads = c_oracle.num_threads()
    dt, _ = cpu_sample(max(nthreads, 32), g)
    per = max(nthreads, int(max(nthreads, 32) * 4.0 / max(dt, 1e-3)))      # ~4 s per step
    per = min(per, 20000)
    for _ in range(min(args.warmup, 1)):
        cpu_sample(per, g)
    t0 = time.perf_counter()
    for s in range(args.steps):
        cpu_sample(per, g, seed=10 + s)
    dt = time.perf_counter() - t0
    val = per * args.steps / dt
    line = {
        "impl": "reference", "metric": "ciphertexts/sec (encrypt+decrypt) N=509 q=2048", "value": val,
        "unit": "ciphertexts/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD.format(rows=per) + " (bounded CPU sample per step)", "rows_per_step": per},
        "cpu_baseline": {"value": val, "unit": "ciphertexts/s", "cores": nthreads, "kind": "port",
                         "sample": f"{per} ciphertexts per step x {args.steps} steps; node is absent from this image, "
                                   "so this is the C restatement of the reference's algorithm (oracle/ntru_ref_port.c)"},
        "e2e": {"value": val, "unit": "ciphertexts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0=None, t1=None):
        if self.proc:
            self.proc.terminate()
        sm, smax, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            if t0 is not None and not (t0 - 0.15 <= ts <= t1 + 0.15):
                continue
            parts = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(parts[0]))
                smax = max(smax, float(parts[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa_node(index: int):
    """Best effort: restrict this rank to the CPUs NVML reports as local to its GPU, so that the pinned e2e buffers
    (first touch) and the copy-issuing thread sit on the GPU's NUMA node.  Returns the CPU list or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1]
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return f"{allowed[0]}-{allowed[-1]} ({len(allowed)} CPUs)"
    except Exception:
        pass
    return None


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def other_configs(rank, world, local_rank, hbm_gbs, which):
    """BASELINE configs 1, 3, 4, 5 (the headline is config 2).  Device-resident, CUDA events on the launch stream,
    barrier + synchronize on both sides, max over ranks; every rank takes part, rank 0 gets the dict."""
    import torch
    import torch.distributed as dist
    import ntru_circom_b200 as nb
    from ntru_circom_b200 import sharding

    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.current_stream(dev)
    l2_flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)        # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    def timed(fn, iters, warm=3, flush=False):
        """ms per call: events around every call (the L2 flush between calls is outside them), summed."""
        for _ in range(warm):
            fn()
        barrier()
        pairs = []
        for _ in range(iters):
            if flush:
                l2_flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            pairs.append((e0, e1))
        barrier()
        return max_over_ranks(sum(a.elapsed_time(b) for a, b in pairs) / iters)

    def engine(cfg):
        g = dict(np.load(os.path.join(ROOT, "tests", "golden", f"{cfg}.npz")))
        N, q, p = int(g["N"]), int(g["q"]), int(g["p"])
        eng = nb.Engine(N, p, q, local_rank)
        eng.set_public_key(g["h"])
        eng.set_private_key(g["f"], g["fp"])
        eng.set_stream(stream.cuda_stream)
        return g, eng, N, q, int(g["dr"])

    def kernel_times(eng, fn, iters=3):
        eng.set_timing(True)
        eng.timing_reset()
        for _ in range(iters):
            fn()
        kt = {k: round(v[0] / v[1], 4) for k, v in eng.timing_read().items() if v[1] and k != "other"}
        eng.set_timing(False)
        return kt

    def buffers(B, P):
        val = torch.empty((B, P), dtype=torch.int16, device=dev)
        return (val, torch.empty_like(val), torch.empty_like(val), torch.empty_like(val),
                torch.empty((B, P), dtype=torch.uint8, device=dev), torch.empty((B, P), dtype=torch.uint8, device=dev))

    out = {}

    # ---- config 1: N=167 q=128, 2^16 ciphertexts per GPU under one key (weak) ----
    if "c1" in which:
        g, eng, N, q, dr = engine("default167")
        B, P = 1 << 16, eng.pitch
        r = torch.zeros((B, P), dtype=torch.uint8, device=dev)
        eng.sample_r_dev(B, dr, rank * B, r, seed=167)
        m = torch.zeros((B, P), dtype=torch.uint8, device=dev)
        m[:, :N] = torch.randint(0, 2, (B, N), generator=torch.Generator(device=dev).manual_seed(167 + rank), device=dev, dtype=torch.uint8)
        val, quo, q1, r1, pv, q2 = buffers(B, P)

        def step1():
            eng.encrypt_dev(B, r, m, value=val, quotientE=quo)
            eng.decrypt_dev(B, val, value=pv, quotient1=q1, remainder1=r1, quotient2=q2)

        ms = timed(step1, 20, flush=True)
        kt = kernel_times(eng, step1)
        # check: the register-fragment schedule on a prefix, bit for bit (oracle parity is tests/); decryption failures
        # are part of the reference at these parameters (~1 row in 3000), so the round trip is reported as a fraction
        nchk = 4096
        eng.set_path(nb.PATH_IMMA)
        val2, quo2, q12, r12, pv2, q22 = buffers(nchk, P)
        eng.encrypt_dev(nchk, r[:nchk], m[:nchk], value=val2, quotientE=quo2)
        eng.decrypt_dev(nchk, val2, value=pv2, quotient1=q12, remainder1=r12, quotient2=q22)
        torch.cuda.synchronize(dev)
        same = all(torch.equal(a[:nchk], b) for a, b in ((val, val2), (quo, quo2), (q1, q12), (r1, r12), (pv, pv2), (q2, q22)))
        rt = float((pv[:, :N] == m[:, :N]).all(dim=1).float().mean().item())
        out["config1"] = {"workload": f"N=167 q=128 same key, {B} ciphertexts per GPU, encrypt+decrypt, full witness", "scaling": "weak",
                          "rows_per_gpu": B, "ms": ms, "ct_per_s": world * B / (ms * 1e-3), "kernel_ms": kt,
                          "GBps_14N_per_gpu": 14 * N * B / (ms * 1e-3) / 1e9, "frac_hbm": 14 * N * B / (ms * 1e-3) / 1e9 / hbm_gbs,
                          "l2": "flushed between timed iterations (153 MB per step is close to the 126 MB L2)", "collective": "none",
                          "matches_imma_schedule_bit_for_bit": bool(same), "roundtrip_fraction": rt}
        eng.close()

    # ---- config 3: N=677 q=2048, a DISTINCT valid key per row, full witness ----
    if "c3" in which:
        g, eng, N, q, dr = engine("hps677")
        B, P, nkeys = 1 << 18, eng.pitch, 4096
        rng = np.random.default_rng(677)
        df, dg = int(g["df"]), int(g["dg"])

        def ternary(n, ones, negs):
            base = np.zeros(N, dtype=np.int8)
            base[:ones] = 1
            base[ones:ones + negs] = -1
            return rng.permuted(np.tile(base, (n, 1)), axis=1)

        t0 = time.perf_counter()
        fk, gk = ternary(nkeys + nkeys // 2, df, df - 1), ternary(nkeys + nkeys // 2, dg, dg)     # index.js:57, 68
        ks = eng.keygen_batch(fk, gk)
        ok = np.flatnonzero(ks["valid"])[:nkeys]
        keygen_s = time.perf_counter() - t0
        reps = (B + len(ok) - 1) // len(ok)
        h = torch.zeros((B, P), dtype=torch.int16, device=dev)
        f = torch.zeros((B, P), dtype=torch.int8, device=dev)
        fp = torch.zeros((B, P), dtype=torch.uint8, device=dev)
        h[:, :N] = torch.from_numpy(np.tile(ks["h"][ok].astype(np.int16), (reps, 1))[:B]).to(dev)
        f[:, :N] = torch.from_numpy(np.tile(fk[ok], (reps, 1))[:B]).to(dev)
        fp[:, :N] = torch.from_numpy(np.tile(ks["fp"][ok], (reps, 1))[:B]).to(dev)
        r = torch.zeros((B, P), dtype=torch.uint8, device=dev)
        eng.sample_r_dev(B, dr, rank * B, r, seed=677)
        m = torch.zeros((B, P), dtype=torch.uint8, device=dev)
        m[:, :N] = torch.randint(0, 2, (B, N), generator=torch.Generator(device=dev).manual_seed(677 + rank), device=dev, dtype=torch.uint8)
        val, quo, q1, r1, pv, q2 = buffers(B, P)

        def step3():
            eng.encrypt_dev(B, r, m, value=val, quotientE=quo, h_rows=h)
            eng.decrypt_dev(B, val, value=pv, quotient1=q1, remainder1=r1, quotient2=q2, f_rows=f, fp_rows=fp)

        ms = timed(step3, 5, warm=2)
        kt = kernel_times(eng, step3, 2)
        nchk = 2048
        eng.set_path(nb.PATH_CUDA_CORE)
        val2, quo2, q12, r12, pv2, q22 = buffers(nchk, P)
        eng.encrypt_dev(nchk, r[:nchk], m[:nchk], value=val2, quotientE=quo2, h_rows=h[:nchk])
        eng.decrypt_dev(nchk, val2, value=pv2, quotient1=q12, remainder1=r12, quotient2=q22, f_rows=f[:nchk], fp_rows=fp[:nchk])
        torch.cuda.synchronize(dev)
        same = all(torch.equal(a[:nchk], b) for a, b in ((val, val2), (quo, quo2), (q1, q12), (r1, r12), (pv, pv2), (q2, q22)))
        macs = 3 * N * N * B / (ms * 1e-3) / 1e12
        out["config3"] = {"workload": f"N=677 q=2048, distinct key per row ({len(ok)} valid key pairs from ntru_keygen_batch, tiled), "
                                      f"{B} ciphertexts per GPU, encrypt+decrypt, full witness", "scaling": "weak",
                          "rows_per_gpu": B, "ms": ms, "ct_per_s": world * B / (ms * 1e-3), "kernel_ms": kt, "keygen_s": keygen_s,
                          "GBps_18N_per_gpu": 18 * N * B / (ms * 1e-3) / 1e9, "frac_hbm": 18 * N * B / (ms * 1e-3) / 1e9 / hbm_gbs,
                          "TMAC_per_s_3N2": macs, "frac_of_imma_peak_570_TMACs": macs / 570.0,
                          # byte-limb products the IMMA schedule has to execute: 2 (r*h) + 2 (f*e) + 1 (fp*b) per ciphertext
                          "byte_TMAC_per_s_5N2": macs * 5 / 3, "frac_of_imma_peak_on_byte_macs": macs * 5 / 3 / 570.0,
                          "bound": "instruction issue of the schedulers: 8.4 cycles per IMMA.16832 + ~1.2 per other instruction "
                                   "(DESIGN.md 3.3, profiles/r2_imma_merged.txt)", "collective": "none",
                          "matches_cuda_core_schedule_bit_for_bit": bool(same),
                          "roundtrip_equals_message": bool(torch.equal(pv[:, :N], m[:, :N]))}
        eng.close()

    # ---- config 4: N=821 q=4096, 2^20 ciphertexts under one key, SHARDED over the ranks (strong scaling) ----
    if "c4" in which:
        g, eng, N, q, dr = engine("hps821")
        total = 1 << 20
        lo, hi = sharding.shard_bounds(total, world, rank)
        B, P = hi - lo, eng.pitch
        r = torch.zeros((B, P), dtype=torch.uint8, device=dev)
        eng.sample_r_dev(B, dr, lo, r, seed=821)                      # row-numbered generator: the same rows at every world size
        m = torch.zeros((B, P), dtype=torch.uint8, device=dev)
        blk = 1 << 16                                                 # message rows from per-block generators: world-size independent
        for b0 in range((lo // blk) * blk, hi, blk):
            rows = torch.randint(0, 2, (blk, N), generator=torch.Generator(device=dev).manual_seed(821_000 + b0 // blk), device=dev, dtype=torch.uint8)
            s0, s1 = max(b0, lo), min(b0 + blk, hi)
            m[s0 - lo:s1 - lo, :N] = rows[s0 - b0:s1 - b0]
        val, quo, q1, r1, pv, q2 = buffers(B, P)

        def step4():
            eng.encrypt_dev(B, r, m, value=val, quotientE=quo)
            eng.decrypt_dev(B, val, value=pv, quotient1=q1, remainder1=r1, quotient2=q2)

        ms = timed(step4, 5)
        kt = kernel_times(eng, step4, 2)
        # checksum of checksums, identical at every world size (q = 4096: decrypt != message by the reference's lift)
        chk = torch.stack([(val[:, :N].to(torch.int64) & 0xFFFF).sum(), (quo[:, :N].to(torch.int64) & 0xFFFF).sum(),
                           (r1[:, :N].to(torch.int64) & 0xFFFF).sum(), pv[:, :N].to(torch.int64).sum(), q2[:, :N].to(torch.int64).sum()])
        if world > 1:
            dist.all_reduce(chk, op=dist.ReduceOp.SUM)
        out["config4"] = {"workload": f"N=821 q=4096 same key, 2^20 ciphertexts sharded over {world} GPU(s), encrypt+decrypt, full witness",
                          "scaling": "strong", "rows_per_gpu": B, "ms": ms, "ct_per_s": total / (ms * 1e-3), "kernel_ms": kt,
                          "GBps_14N_per_gpu": 14 * N * B / (ms * 1e-3) / 1e9, "frac_hbm": 14 * N * B / (ms * 1e-3) / 1e9 / hbm_gbs,
                          "int8_TOPs_10N2_per_gpu": 10 * N * N * B / (ms * 1e-3) / 1e12, "collective": "none",
                          "checksum": [int(x) for x in chk.tolist()]}
        eng.close()

    # ---- config 5: N=701 q=8192, homomorphic sum of 10 M ciphertext rows sharded over the ranks ----
    if "c5" in which:
        g, eng, N, q, dr = engine("hrss701")
        total = 10_000_000
        lo, hi = sharding.shard_bounds(total, world, rank)
        B, P = hi - lo, eng.pitch
        blk = 250_000                                                 # rows from per-block generators: world-size independent
        e = torch.empty((B, P), dtype=torch.int16, device=dev)
        for b0 in range((lo // blk) * blk, hi, blk):
            rows = torch.randint(0, q, (blk, P), generator=torch.Generator(device=dev).manual_seed(7_000_000 + b0 // blk), device=dev, dtype=torch.int16)
            s0, s1 = max(b0, lo), min(b0 + blk, hi)
            e[s0 - lo:s1 - lo] = rows[s0 - b0:s1 - b0]
        e[:, N:] = 0
        want = torch.zeros(N, dtype=torch.int64, device=dev)
        for b0 in range(0, B, 500_000):
            want += e[b0:b0 + 500_000, :N].to(torch.int64).sum(dim=0)
        if world > 1:
            dist.all_reduce(want, op=dist.ReduceOp.SUM)
        want %= q
        # (a) the product path: column sums fused with the exchange over NVLink peer memory, one kernel per call
        sharding.connect_exchange(eng)
        res = torch.empty(P, dtype=torch.int16, device=dev)
        ms_x = timed(lambda: eng.sum_allreduce_dev(B, e, res), 10)
        eng.sync()                                                    # raises if a peer timed out inside the kernel
        ok_x = bool(torch.equal(res[:N].to(torch.int64) & 0xFFFF, want)) and not bool(res[N:].any())
        # (b) the same local kernel + one ncclAllReduce of N int32 (baseline for the exchange)
        partial = torch.zeros(P, dtype=torch.int32, device=dev)
        loc = torch.empty(P, dtype=torch.int16, device=dev)
        red = torch.empty(P, dtype=torch.int32, device=dev)

        def nccl_path():
            partial.zero_()
            eng.sum_partial_dev(B, e, partial)
            eng.sum_finalize_dev(partial, loc)
            red.copy_(loc)
            red.bitwise_and_(0xFFFF)
            if world > 1:
                dist.all_reduce(red, op=dist.ReduceOp.SUM)
            red.bitwise_and_(q - 1)

        ms_n = timed(nccl_path, 10)
        ok_n = bool(torch.equal(red[:N].to(torch.int64), want))

        def local_only():
            partial.zero_()
            eng.sum_partial_dev(B, e, partial)

        ms_l = timed(local_only, 10)
        sharding.disconnect_exchange(eng)
        out["config5"] = {"workload": f"N=701 q=8192, homomorphic sum of 10 000 000 ciphertext rows sharded over {world} GPU(s)",
                          "scaling": "strong", "rows_per_gpu": B, "ms": ms_x, "ct_per_s": total / (ms_x * 1e-3),
                          "GBps_2N_per_gpu": 2 * N * B / (ms_x * 1e-3) / 1e9, "frac_hbm": 2 * N * B / (ms_x * 1e-3) / 1e9 / hbm_gbs,
                          "collective": ("stores into every peer's exchange window over NVLink inside the sum kernel (ntru_sum_allreduce_dev), "
                                         "no collective library on the data path") if world > 1 else "none (one rank)",
                          "matches_int64_column_sums": ok_x,
                          "nccl_allreduce_path": {"ms": ms_n, "collective": "ncclAllReduce of N int32 after the local column sums" if world > 1 else "none",
                                                  "matches_int64_column_sums": ok_n},
                          "local_column_sums_only_ms": ms_l, "checksum": int(want.sum().item())}
        eng.close()
    del l2_flush
    return out


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import ntru_circom_b200 as nb

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None     # pinned host buffers land next to this rank's GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    g = load_key()
    N, q, p, dr = int(g["N"]), int(g["q"]), int(g["p"]), int(g["dr"])
    eng = nb.Engine(N, p, q, local_rank)
    eng.set_public_key(g["h"])
    eng.set_private_key(g["f"], g["fp"])
    if args.path:
        eng.set_path(args.path)
    stream = torch.cuda.current_stream(dev)
    eng.set_stream(stream.cuda_stream)
    P, B = eng.pitch, args.rows

    # ---- synthetic inputs, resident in HBM: r from the device sampler, m = random bits ----
    r = torch.zeros((B, P), dtype=torch.uint8, device=dev)
    eng.sample_r_dev(B, dr, rank * B, r, seed=2026)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    m = torch.zeros((B, P), dtype=torch.uint8, device=dev)
    m[:, :N] = torch.randint(0, 2, (B, N), generator=gen, device=dev, dtype=torch.uint8)
    value = torch.empty((B, P), dtype=torch.int16, device=dev)
    quo = torch.empty((B, P), dtype=torch.int16, device=dev)
    out = torch.empty((B, P), dtype=torch.uint8, device=dev)
    q1 = torch.empty((B, P), dtype=torch.int16, device=dev)
    r1 = torch.empty((B, P), dtype=torch.int16, device=dev)
    q2 = torch.empty((B, P), dtype=torch.uint8, device=dev)

    def step():
        # remainderE == value and remainder2 == plaintext value: written once (SURVEY 8d)
        eng.encrypt_dev(B, r, m, value=value, quotientE=quo)
        eng.decrypt_dev(B, value, value=out, quotient1=q1, remainder1=r1, quotient2=q2)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize(dev)
    assert torch.equal(out[:, :N], m[:, :N]), "decrypt(encrypt(m)) != m"

    eng.set_timing(True)
    eng.timing_reset()
    launches0 = eng.launch_count
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    barrier()
    t_wall1 = time.perf_counter()
    ms = ev0.elapsed_time(ev1)
    launches = eng.launch_count - launches0
    kt = eng.timing_read()
    eng.set_timing(False)
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value_cts = world * B * args.steps / (ms * 1e-3)
    # what the last timed step computed, as the host-buffer ABI returns it (remainderE == value, remainder2 == plaintext)
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = dump_outputs(args.dump_outputs, {
            "value": value[:, :N], "quotientE": quo[:, :N + 1], "plaintext": out[:, :N],
            "quotient1": q1[:, :N + 1], "remainder1": r1[:, :N + 1], "quotient2": q2[:, :N + 1]})

    # ---- secondary figures (outside the timed region above): value-only mode, encrypt-only, decrypt-only ----
    def timed_ms(fn, iters=5):
        fn()
        torch.cuda.synchronize(dev)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(stream)
        for _ in range(iters):
            fn()
        a1.record(stream)
        torch.cuda.synchronize(dev)
        return a0.elapsed_time(a1) / iters

    t_enc = timed_ms(lambda: eng.encrypt_dev(B, r, m, value=value, quotientE=quo))
    t_dec = timed_ms(lambda: eng.decrypt_dev(B, value, value=out, quotient1=q1, remainder1=r1, quotient2=q2))
    t_enc_v = timed_ms(lambda: eng.encrypt_dev(B, r, m, value=value))
    t_dec_v = timed_ms(lambda: eng.decrypt_dev(B, value, value=out))
    extras = {"encrypt_only_ct_per_s": B / (t_enc * 1e-3), "decrypt_only_ct_per_s": B / (t_dec * 1e-3),
              "value_only_ct_per_s": B / ((t_enc_v + t_dec_v) * 1e-3), "value_only_ms": {"enc": t_enc_v, "dec": t_dec_v},
              "value_only_GBps_7N": 7 * N * B / ((t_enc_v + t_dec_v) * 1e-3) / 1e9, "note": "per GPU, measured after the timed region"}

    # ---- end to end through the host-buffer ABI (pinned host memory, copies inside the timing) ----
    # Two wire formats of the same two calls: "field_elements" -- every array as packOutput(maxVal, width, row).expected
    # (index.js:572-596, the form CombineArray / UnpackArray take; bits packed and unpacked on the device) -- and
    # "plain_arrays" (uint16 / uint8 coefficient rows).  Same rows, same results (checked below after unpacking).
    # rows per end-to-end step: the whole batch when the host can pin it (both wire formats are measured one after the
    # other, ~20 KB of host buffers per row at the peak), else a half or a quarter of it -- longer steps amortise the fill and
    # drain of the copy pipeline (0.92 / 0.95 / 0.96 of the PCIe roof at 2^18 / 2^19 / 10^6 rows)
    if args.e2e_rows:
        Be = min(args.e2e_rows, B)
    else:
        try:
            import psutil
            per_rank_gb = psutil.virtual_memory().total / world / 2 ** 30
        except Exception:
            per_rank_gb = 0.0
        Be = min(B, 1_000_000 if per_rank_gb >= 64 else (524_288 if per_rank_gb >= 32 else 262_144))
    eng2 = nb.Engine(N, p, q, local_rank)
    eng2.set_public_key(g["h"])
    eng2.set_private_key(g["f"], g["fp"])
    if args.path:
        eng2.set_path(args.path)
    pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()   # noqa: E731
    lib, ctx = eng2.lib, eng2._h
    r_host, m_host = r[:Be, :N].cpu().numpy(), m[:Be, :N].cpu().numpy()

    def wall(fn, n):
        fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(n):
            fn()
        torch.cuda.synchronize(dev)
        d = (time.perf_counter() - t0) / n
        if world > 1:
            t = torch.tensor([d], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            d = float(t.item())
        return d

    def e2e_measure(fe: bool):
        if fe:
            el = lambda mod_q, width: (Be, eng2.packed_elems(mod_q, width), 8)   # noqa: E731
            h_r, h_m = pin(el(False, N), torch.int32), pin(el(False, N), torch.int32)
            h_r.numpy()[:] = nb.wire.pack_rows(p - 1, r_host).view(np.int32)
            h_m.numpy()[:] = nb.wire.pack_rows(p - 1, m_host).view(np.int32)
            h_val, h_quo = pin(el(True, N), torch.int32), pin(el(True, N + 1), torch.int32)
            h_out, h_q1, h_r1 = pin(el(False, N), torch.int32), pin(el(True, N + 1), torch.int32), pin(el(True, N + 1), torch.int32)
            h_q2 = pin(el(False, N + 1), torch.int32)
            f_enc, f_dec = lib.ntru_encrypt_batch_packed, lib.ntru_decrypt_batch_packed
        else:
            h_r, h_m = pin((Be, N), torch.uint8), pin((Be, N), torch.uint8)
            h_r.numpy()[:] = r_host
            h_m.numpy()[:] = m_host
            h_val, h_quo = pin((Be, N), torch.int16), pin((Be, N + 1), torch.int16)
            h_out, h_q1, h_r1 = pin((Be, N), torch.uint8), pin((Be, N + 1), torch.int16), pin((Be, N + 1), torch.int16)
            h_q2 = pin((Be, N + 1), torch.uint8)
            f_enc, f_dec = lib.ntru_encrypt_batch, lib.ntru_decrypt_batch

        def e2e_step():
            rc = f_enc(ctx, Be, h_r.data_ptr(), h_m.data_ptr(), h_val.data_ptr(), h_quo.data_ptr(), None, None)
            assert rc == 0, eng2.lib.ntru_last_error(ctx)
            rc = f_dec(ctx, Be, h_val.data_ptr(), h_out.data_ptr(), h_q1.data_ptr(), h_r1.data_ptr(), h_q2.data_ptr(), None)
            assert rc == 0, eng2.lib.ntru_last_error(ctx)

        dt = wall(e2e_step, args.e2e_steps)
        nbytes = lambda *ts: int(sum(t.numel() * t.element_size() for t in ts))   # noqa: E731
        res = {"value": world * Be / dt, "unit": "ciphertexts/s",
               "h2d_bytes_per_step": nbytes(h_r, h_m, h_val), "d2h_bytes_per_step": nbytes(h_val, h_quo, h_out, h_q1, h_r1, h_q2),
               "rows_per_step": Be, "steps": args.e2e_steps, "timer": "host wall clock around the synchronous C-ABI calls"}
        # PCIe roof of exactly these transfers: one plain cudaMemcpyAsync per array of a step (no kernels), host -> device
        # on one stream and device -> host on another, every rank at the same time; same wall-clock timer
        h_in, h_outs = (h_r, h_m, h_val), (pin(tuple(h_val.shape), h_val.dtype), h_quo, h_out, h_q1, h_r1, h_q2)   # value lands in its own rows
        d_in = [torch.empty(t.shape, dtype=t.dtype, device=dev) for t in h_in]
        d_out = [torch.zeros(t.shape, dtype=t.dtype, device=dev) for t in h_outs]
        s_up, s_down = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        keep = {k: v.clone() for k, v in (("value", h_val), ("quotientE", h_quo), ("plain", h_out), ("quotient1", h_q1),
                                          ("remainder1", h_r1), ("quotient2", h_q2))}     # results, before the roof copies overwrite them

        def pcie_step(up=True, down=True):
            if up:
                with torch.cuda.stream(s_up):
                    for d, h in zip(d_in, h_in):
                        d.copy_(h, non_blocking=True)
            if down:
                with torch.cuda.stream(s_down):
                    for h, d in zip(h_outs, d_out):             # h_val itself is being read by the upload at the same time
                        h.copy_(d, non_blocking=True)

        t_both, t_up, t_down = wall(pcie_step, 3), wall(lambda: pcie_step(True, False), 3), wall(lambda: pcie_step(False, True), 3)
        res["pcie_roof"] = {"s_per_step_both_directions": t_both, "ct_per_s": world * Be / t_both,
                            "h2d_GBps_per_gpu_alone": res["h2d_bytes_per_step"] / t_up / 1e9,
                            "d2h_GBps_per_gpu_alone": res["d2h_bytes_per_step"] / t_down / 1e9,
                            "how": "plain cudaMemcpyAsync of the step's arrays from/to the same pinned buffers, two streams, no kernels"}
        res["frac_of_pcie"] = t_both / dt
        return res, keep

    e2e_plain, keep_plain = e2e_measure(False)
    e2e, keep_fe = e2e_measure(True)
    # both wire formats carry the same results: unpack the field elements on the host and compare every array
    assert np.array_equal(keep_plain["plain"].numpy(), m_host), "decrypt(encrypt(m)) != m (plain arrays)"
    for k, mod_q, width in (("value", True, N), ("quotientE", True, N + 1), ("plain", False, N), ("quotient1", True, N + 1),
                            ("remainder1", True, N + 1), ("quotient2", False, N + 1)):
        got = nb.wire.unpack_rows(q - 1 if mod_q else p - 1, width, keep_fe[k].numpy().view(np.uint32), np.uint16 if mod_q else np.uint8)
        want = keep_plain[k].numpy()
        assert np.array_equal(got, want.view(np.uint16) if mod_q else want), f"field-element wire format differs from the plain arrays in {k}"
    e2e["wire"] = ("BN254 field elements, packOutput(maxVal, width, row).expected per row (index.js:572-596): maxVal = q - 1 for value / "
                   "quotientE / quotient1 / remainder1, p - 1 for r / m / plaintext / quotient2; ntru_encrypt_batch_packed + ntru_decrypt_batch_packed")
    e2e["equals_plain_arrays_after_unpack"] = True
    e2e_plain["wire"] = "uint16 / uint8 coefficient rows; ntru_encrypt_batch + ntru_decrypt_batch"
    e2e["plain_arrays"] = e2e_plain
    e2e["cpu_affinity"] = numa
    del keep_plain, keep_fe

    # ---- the other BASELINE configs (every rank takes part: configs 4 and 5 are sharded over the ranks) ----
    hbm_gbs, bf16_tf, peak_src = peaks()
    for t in (r, m, value, quo, out, q1, r1, q2):
        t.untyped_storage().resize_(0)                 # the headline's 7 GB of device rows are done
    eng.close()
    eng2.close()
    configs = other_configs(rank, world, local_rank, hbm_gbs, [c for c in args.configs.split(",") if c]) if args.configs else {}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (CUDA events on the launch stream, inside the timed region) ----
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "r2_dram_traffic.json")))     # written by scripts/ncu_traffic.py
        prof["int8_peak_tops"] = json.load(open(os.path.join(ROOT, "profiles", "r1_dram_traffic.json"))).get("int8_peak_tops")
    except OSError:
        prof = {"bytes_per_ciphertext": {}, "int8_peak_tops": None}
    alg_bytes = {"enc_tensor": 6 * N, "dec1_tensor": 6 * N, "dec2_tensor": 2 * N, "enc_core": 6 * N, "dec_core": 8 * N,
                 "enc_imma": 6 * N, "dec_imma": 8 * N}
    limbs = 2 if q > 256 else 1
    alg_ops = {"enc_tensor": 2 * N * N * limbs, "dec1_tensor": 2 * N * N * limbs, "dec2_tensor": 2 * N * N,
               "enc_core": 2 * N * N, "dec_core": 4 * N * N, "enc_imma": 2 * N * N * limbs, "dec_imma": 2 * N * N * (limbs + 1)}
    kernels = {}
    for name, (tot, n) in kt.items():
        if name not in alg_bytes:
            continue
        avg = tot / n
        kernels[name] = {"avg_ms": avg, "launches": n, "share_of_step": tot / ms,
                         "GB/s": alg_bytes[name] * B / (avg * 1e-3) / 1e9,
                         "TOP/s": alg_ops[name] * B / (avg * 1e-3) / 1e12}
    dom = max(kernels, key=lambda k: kernels[k]["avg_ms"])
    roofline = {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["GB/s"], "peak": hbm_gbs, "unit": "GB/s",
                "frac": kernels[dom]["GB/s"] / hbm_gbs,
                "traffic": (prof["bytes_per_ciphertext"].get(dom) or 0) * B or None,
                "traffic_source": "ncu --set full at 1 000 000 rows per launch: dram__bytes_read.sum + dram__bytes_write.sum per ciphertext "
                                  "(profiles/r2_dram_traffic.json, written by scripts/ncu_traffic.py) x rows per launch",
                "traffic_over_algorithmic": (prof["bytes_per_ciphertext"].get(dom) or 0) / alg_bytes[dom] or None,
                "peak_source": peak_src,
                "algorithmic_bytes_per_ciphertext": alg_bytes[dom],
                "int8_tensor": {"achieved_TOPs": kernels[dom]["TOP/s"], "peak_TOPs": prof.get("int8_peak_tops") or 2 * bf16_tf,
                                "frac": kernels[dom]["TOP/s"] / (prof.get("int8_peak_tops") or 2 * bf16_tf),
                                "peak_source": "measured MMA-loop-only probe (scripts/mma_peak.cu)" if prof.get("int8_peak_tops") else "2 x measured bf16",
                                "frac_of_2x_measured_bf16": kernels[dom]["TOP/s"] / (2 * bf16_tf)},
                "whole_step": {"GB/s": 14 * N * B * args.steps / (ms * 1e-3) / 1e9,
                               "frac": 14 * N * B * args.steps / (ms * 1e-3) / 1e9 / hbm_gbs},
                "kernels": kernels}
    line = {
        "metric": "ciphertexts/sec (encrypt+decrypt) N=509 q=2048", "value": value_cts, "unit": "ciphertexts/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int8 x int8 -> int32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD.format(rows=B), "rows_per_gpu": B, "parallelism": f"batch-sharded x{world}, no collective",
                   "l2": "inputs+outputs per step (7 GB at 1M rows) exceed the 126 MB L2; no flush needed",
                   "schedule": {0: "auto", 1: "cuda-core", 2: "tcgen05", 3: "imma"}[args.path], "key": "tests/golden/hps509.npz"},
        "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "extras": extras,
    }
    extras["configs"] = configs
    if dumped:
        line["dump_outputs"] = dumped
    if not args.no_cpu and world == 1:                  # the CPU leg runs at N = 1 only (rank 0's host cores)
        line["cpu_baseline"] = cpu_baseline(g)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=1_000_000, help="ciphertexts per GPU per step")
    ap.add_argument("--e2e-rows", type=int, default=0, help="rows per end-to-end step; 0 = by host memory per rank (10^6, 2^19 or 2^18)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--path", type=int, default=0, help="0 auto, 1 fp32 CUDA-core schedule, 2 tcgen05 schedule, 3 register-fragment IMMA schedule")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--configs", default="c1,c3,c4,c5", help="other BASELINE configs to run after the headline (extras.configs); '' for none")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write a seeded sample of 4096 rows of every output of the last step to DIR/<name>.npy "
                         "(float32, 50 MB; rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch with torchrun for --gpus > 1 (one process per GPU)")
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
