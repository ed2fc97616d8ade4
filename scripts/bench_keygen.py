"""Key-generation measurements (recurring):  python scripts/bench_keygen.py [--ab OTHER_LIB.so]

1. ntru_keygen_batch (host buffers) on the inputs and sizes of the round-2 record: keys/s, GPU kernel time, and with
   --ab an A/B against another build of the library (for example the parent commit's), alternated, median of 5, outputs
   compared bit for bit.  Raw ctypes on the one entry point both builds have, so that an older build loads.
2. ntru_generate_keys_dev at B = 2^18 keys (draws, inversions, redraws, lifting, h all on the device): keys/s, and the
   device time split into inverse / muldiv / other by NTRU_OPT_TIMING in a separate run.
3. bench.py's config 3 (N = 677, encrypt + decrypt with full witness, 2^18 rows) with a distinct device-generated key on
   every row instead of 4096 tiled keys.
Prints the GPU's name and power limit first."""
import argparse
import ctypes
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle")]
import ntru_circom_b200 as nb  # noqa: E402
import ntru_oracle as o  # noqa: E402

R2_SIZES = (("default167", 4096), ("hps509", 2048), ("hps677", 2048), ("hps821", 1024))


def r2_inputs(cfg, B):
    """the inputs of the round-2 record (seeded permutations of the exact-weight arrays)"""
    c = o.CONFIGS[cfg]
    N = c["N"]
    rng = np.random.default_rng(0)
    f = np.stack([rng.permutation(np.array([1] * c["df"] + [-1] * (c["df"] - 1) + [0] * (N - 2 * c["df"] + 1), dtype=np.int8)) for _ in range(B)])
    g = np.stack([rng.permutation(np.array([1] * c["dg"] + [-1] * c["dg"] + [0] * (N - 2 * c["dg"]), dtype=np.int8)) for _ in range(B)])
    return f, g


class RawLib:
    """ntru_keygen_batch of one build through raw ctypes"""

    def __init__(self, path, cfg):
        c = o.CONFIGS[cfg]
        V = ctypes.c_void_p
        self.lib = lib = ctypes.CDLL(path)
        lib.ntru_create.argtypes = [ctypes.POINTER(V), ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int]
        lib.ntru_keygen_batch.argtypes = [V, ctypes.c_size_t] + [V] * 6
        lib.ntru_destroy.argtypes = [V]
        self.h = V()
        assert lib.ntru_create(ctypes.byref(self.h), c["N"], c["p"], c["q"], 0) == 0
        self.N = c["N"]

    def keygen(self, f, g):
        B, N = f.shape
        out = {"fq": np.empty((B, N), np.uint16), "fp": np.empty((B, N), np.uint8), "h": np.empty((B, N), np.uint16),
               "valid": np.empty(B, np.uint8)}
        rc = self.lib.ntru_keygen_batch(self.h, B, f.ctypes.data, g.ctypes.data, out["fq"].ctypes.data, out["fp"].ctypes.data,
                                        out["h"].ctypes.data, out["valid"].ctypes.data)
        assert rc == 0, rc
        return out

    def close(self):
        self.lib.ntru_destroy(self.h)


def part_keygen_batch(libs):
    print("## ntru_keygen_batch, host buffers (inputs and sizes of profiles/r2_bench_keygen.txt); wall time of the call, "
          "median of 5, libraries alternated", flush=True)
    for cfg, B in R2_SIZES:
        f, g = r2_inputs(cfg, B)
        runs = {name: RawLib(path, cfg) for name, path in libs}
        outs, times = {}, {name: [] for name in runs}
        for name, r in runs.items():
            r.keygen(f[:64], g[:64])
        for _ in range(5):
            for name, r in runs.items():
                t0 = time.perf_counter()
                outs[name] = r.keygen(f, g)
                times[name].append(time.perf_counter() - t0)
        ref = outs[libs[0][0]]
        for name, r in runs.items():
            same = all(np.array_equal(outs[name][k], ref[k]) for k in ref)
            ms = statistics.median(times[name]) * 1e3
            print(f"{cfg}: {name}: {B} keys in {ms:.2f} ms = {B / ms * 1e3:.0f} keys/s (valid {int(outs[name]['valid'].sum())})"
                  f"{'' if name == libs[0][0] else f', outputs identical to {libs[0][0]}: {same}'}", flush=True)
            r.close()
        eng = nb.Engine(o.CONFIGS[cfg]["N"], 3, o.CONFIGS[cfg]["q"], 0)
        eng.keygen_batch(f[:64], g[:64])
        eng.set_timing(True)
        eng.timing_reset()
        eng.keygen_batch(f, g)
        kt = eng.timing_read()
        print(f"{cfg}: this build, kernels (ms, launches): " + ", ".join(f"{k} {v[0]:.3f} / {v[1]}" for k, v in kt.items()), flush=True)
        eng.close()


def part_generate(torch):
    B = 1 << 18
    print(f"## ntru_generate_keys_dev, B = {B} keys per call: wall time to a synchronised stream, median of 5; then one "
          "run with NTRU_OPT_TIMING", flush=True)
    for cfg in ("default167", "hps509", "hps677", "hps821"):
        c = o.CONFIGS[cfg]
        eng = nb.Engine(c["N"], c["p"], c["q"], 0)
        eng.set_stream(torch.cuda.current_stream().cuda_stream)
        P = eng.pitch
        f = torch.empty((B, P), dtype=torch.int8, device="cuda")
        g = torch.empty((B, P), dtype=torch.int8, device="cuda")
        fq = torch.empty((B, P), dtype=torch.int16, device="cuda")
        fp = torch.empty((B, P), dtype=torch.uint8, device="cuda")
        h = torch.empty((B, P), dtype=torch.int16, device="cuda")
        eng.set_rng_key(nb.seed_key(c["N"]), 0)
        eng.generate_keys_dev(1024, c["df"], c["dg"], f, g, fq, fp, h)
        eng.sync()
        ts = []
        for _ in range(5):
            row = eng.rng_next_row
            t0 = time.perf_counter()
            eng.generate_keys_dev(B, c["df"], c["dg"], f, g, fq, fp, h)
            eng.sync()
            ts.append(time.perf_counter() - t0)
            rounds = (eng.rng_next_row - row) // B - 1
        ms = statistics.median(ts) * 1e3
        eng.set_timing(True)
        eng.timing_reset()
        eng.generate_keys_dev(B, c["df"], c["dg"], f, g, fq, fp, h)
        kt = eng.timing_read()
        eng.set_timing(False)
        tot = sum(v[0] for v in kt.values())
        split = ", ".join(f"{k} {v[0]:.2f} ms ({v[1]} launches)" for k, v in kt.items())
        print(f"{cfg}: {B} keys in {ms:.2f} ms = {B / ms * 1e3 / 1e6:.3f} M keys/s (rounds of draws: {rounds}); "
              f"device time {tot:.2f} ms: {split}", flush=True)
        eng.close()


def part_config3(torch):
    c = o.CONFIGS["hps677"]
    N, q, p, dr = c["N"], c["q"], c["p"], c["dr"]
    B = 1 << 18
    kk = nb.NTRU(dict(c))
    eng = kk.engine()
    eng.set_stream(torch.cuda.current_stream().cuda_stream)
    eng.set_rng_key(nb.seed_key(677), 0)
    t0 = time.perf_counter()
    keys = kk.generateKeysDevice(B)
    keygen_ms = (time.perf_counter() - t0) * 1e3
    P = eng.pitch
    r = torch.zeros((B, P), dtype=torch.uint8, device="cuda")
    eng.sample_r_dev(B, dr, 1 << 40, r)
    m = torch.zeros((B, P), dtype=torch.uint8, device="cuda")
    m[:, :N] = torch.randint(0, 2, (B, N), generator=torch.Generator(device="cuda").manual_seed(677), device="cuda", dtype=torch.uint8)
    val, quo, q1, r1 = (torch.empty((B, P), dtype=torch.int16, device="cuda") for _ in range(4))
    pv, q2 = (torch.empty((B, P), dtype=torch.uint8, device="cuda") for _ in range(2))

    def step():
        eng.encrypt_dev(B, r, m, value=val, quotientE=quo, h_rows=keys["h"])
        eng.decrypt_dev(B, val, value=pv, quotient1=q1, remainder1=r1, quotient2=q2, f_rows=keys["f"], fp_rows=keys["fp"])

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(5):
        step()
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / 5
    ok = torch.equal(pv[:, :N], m[:, :N])
    print(f"## config 3 with a distinct device-generated key per row: N=677 q=2048, {B} rows, encrypt+decrypt with full witness: "
          f"{ms:.3f} ms per step = {B / ms * 1e3 / 1e6:.1f} M ct/s (decryptions equal the messages: {ok}); the {B} key pairs took "
          f"{keygen_ms:.1f} ms (generateKeysDevice)", flush=True)
    eng.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ab", default=None, help="another build of libntru_b200.so to compare ntru_keygen_batch with")
    args = ap.parse_args()
    import torch
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(f"# GPU: {smi}", flush=True)
    libs = [("this build", nb._lib.LIB_PATH)]
    if args.ab:
        libs.append((os.path.basename(args.ab), args.ab))
    part_keygen_batch(libs)
    part_generate(torch)
    part_config3(torch)


if __name__ == "__main__":
    main()
