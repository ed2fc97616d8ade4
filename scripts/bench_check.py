"""Witness-check throughput on device-resident rows (ntru_check_*_dev), against the IMMA encrypt / decrypt kernels.

At each BASELINE N: 2^18 rows with a distinct key per row and 2^18 rows under one key (key_stride 0), honest witnesses
made by the engine.  Kernel times come from NTRU_OPT_TIMING events (device time of the launches only); every check must
return SATISFIED | CANONICAL for every row.  Prints the GPU name and power limit with the results.

    python scripts/bench_check.py [--rows 262144] [--reps 5]
"""
import argparse
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = [(167, 128), (509, 2048), (677, 2048), (701, 8192), (821, 4096)]


def gpu_info(torch):
    name = torch.cuda.get_device_name(0)
    try:
        res = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30)
        power = res.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def timed(eng, kind, reps, fn):
    fn()                                           # warm-up: module load, occupancy query
    eng.sync()
    eng.timing_reset()
    for _ in range(reps):
        fn()
    t = eng.timing_read()
    ms, n = t[kind]
    return ms / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1 << 18)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch
    import ntru_circom_b200 as nb
    name, power = gpu_info(torch)
    print(f"GPU: {name}, power limit {power}; {args.rows} rows per batch, mean of {args.reps} launches after one warm-up")
    print(f"{'N':>4} {'q':>5} {'keys':>9} | {'enc_imma ms':>11} {'chk_enc ms':>10} {'Mrow/s':>7} | {'dec_imma ms':>11} "
          f"{'chk_dec ms':>10} {'Mrow/s':>7} | {'chk_inv_q ms':>12} {'chk_inv_p ms':>12}")
    B = args.rows
    for N, q in SHAPES:
        eng = nb.Engine(N, 3, q, 0)
        rng = np.random.default_rng(N)
        h, f, fp = rng.integers(0, q, N), rng.integers(-1, 2, N), rng.integers(0, 3, N)
        eng.set_public_key(h.astype(np.uint16))
        eng.set_private_key(f.astype(np.int8), fp.astype(np.uint8))
        eng.set_path(nb.PATH_IMMA)
        eng.set_timing(True)
        P = eng.pitch
        gen = torch.Generator(device="cuda").manual_seed(N)

        def rows(lo, hi, dtype):
            t = torch.zeros((B, P), dtype=dtype, device="cuda")
            t[:, :N] = torch.randint(lo, hi, (B, N), generator=gen, device="cuda", dtype=dtype)
            return t

        r, m = rows(0, 3, torch.uint8), rows(0, 2, torch.uint8)
        m16 = m.to(torch.int16)
        h_rows, f_rows, fp_rows = rows(0, q, torch.int16), rows(-1, 2, torch.int8), rows(0, 3, torch.uint8)
        f16_rows = torch.where(f_rows < 0, f_rows.to(torch.int32) + q, f_rows.to(torch.int32)).to(torch.int16)
        h_one = torch.zeros(P, dtype=torch.int16, device="cuda")
        h_one[:N] = torch.from_numpy(h.astype(np.int16)).cuda()
        f_one = torch.zeros(P, dtype=torch.int16, device="cuda")
        f_one[:N] = torch.from_numpy(np.where(f < 0, q - 1, f).astype(np.int16)).cuda()
        fp_one = torch.zeros(P, dtype=torch.uint8, device="cuda")
        fp_one[:N] = torch.from_numpy(fp.astype(np.uint8)).cuda()
        e = {k: torch.empty((B, P), dtype=torch.int16, device="cuda") for k in ("value", "quotientE", "remainderE")}
        d = {"value": torch.empty((B, P), dtype=torch.uint8, device="cuda"),
             "quotient1": torch.empty((B, P), dtype=torch.int16, device="cuda"),
             "remainder1": torch.empty((B, P), dtype=torch.int16, device="cuda"),
             "quotient2": torch.empty((B, P), dtype=torch.uint8, device="cuda"),
             "remainder2": torch.empty((B, P), dtype=torch.uint8, device="cuda")}
        v = torch.empty(B, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        for label, distinct in (("distinct", True), ("one", False)):
            hk = {"h_rows": h_rows} if distinct else {}
            fk = {"f_rows": f_rows, "fp_rows": fp_rows} if distinct else {}
            t_enc = timed(eng, "enc_imma", args.reps, lambda: eng.encrypt_dev(B, r, m, **e, **hk))
            t_dec = timed(eng, "dec_imma", args.reps, lambda: eng.decrypt_dev(B, e["value"], **d, **fk))
            key_h, key_f, key_fp, stride = (h_rows, f16_rows, fp_rows, P) if distinct else (h_one, f_one, fp_one, 0)
            t_ce = timed(eng, "check", args.reps,
                         lambda: eng.check_encrypt_dev(B, key_h, stride, r, m16, e["quotientE"], e["remainderE"], v))
            assert bool((v == 3).all()), "encrypt check failed on honest rows"
            t_cd = timed(eng, "check", args.reps,
                         lambda: eng.check_decrypt_dev(B, key_f, key_fp, stride, e["value"], d["quotient1"], d["remainder1"],
                                                       d["quotient2"], d["remainder2"], v))
            assert bool((v == 3).all()), "decrypt check failed on honest rows"
            if distinct:     # VerifyInverse: per-row x and y only (the fq and fp cases of verify_keys)
                eng.muldiv_dev(B, f_rows, h_rows, False, d["quotient1"], d["remainder1"])
                t_iq = timed(eng, "check", args.reps,
                             lambda: eng.check_inverse_dev(B, False, f16_rows, h_rows, d["quotient1"], d["remainder1"], v))
                assert bool((v == 3).all()), "inverse (mod q) check failed on honest rows"
                f2_rows = torch.where(f_rows < 0, 2, f_rows.to(torch.int32)).to(torch.int16)
                eng.muldiv_dev(B, f_rows, fp_rows, True, d["quotient2"], d["remainder2"])
                t_ip = timed(eng, "check", args.reps,
                             lambda: eng.check_inverse_dev(B, True, f2_rows, fp_rows, d["quotient2"], d["remainder2"], v))
                assert bool((v == 3).all()), "inverse (mod p) check failed on honest rows"
                inv = f"{t_iq:12.3f} {t_ip:12.3f}"
            else:
                inv = f"{'-':>12} {'-':>12}"
            print(f"{N:>4} {q:>5} {label:>9} | {t_enc:11.3f} {t_ce:10.3f} {B / t_ce / 1e3:7.1f} | {t_dec:11.3f} {t_cd:10.3f} "
                  f"{B / t_cd / 1e3:7.1f} | {inv}", flush=True)
        eng.close()


if __name__ == "__main__":
    main()
