"""Every schedule at the bounds of its exactness argument: worst-case keys and operands, lift boundaries, full-range
multiply-divide inputs.

Each schedule agrees with the reference bit for bit only because of a range argument written next to its code:
- CUDA-core (csrc/generic_kernels.cu): every fp32 partial sum is an integer of magnitude <= N 2 (q - 1) < 2^24 (at
  N = 1024, q = 8192 that is 2048 below 2^24); the message, up to q - 1 for wide messages, is added after the
  conversion to int.
- IMMA (csrc/imma_kernels.cu): encrypt and decrypt merge the limbs of y = y0 + 256 y1 (y1 < 64) into one accumulator
  through the staged bytes 4 y1 and 64 x.  k_muldiv_imma takes any uint16 y and x in [-1, 2], keeps one accumulator per
  limb, and corrects its mod-p products in (-2N, 4N) through 65536 = 1 (mod 3).
- tcgen05 (csrc/umma_kernels.cu): encrypt recombines h = h0 + 256 h1 from two accumulator column groups as
  acc0 + (acc1 << 8); the first decrypt product stages A = [e0 | e1 << 2] against B = [f | f << 6] or, at
  256 < q <= 2048, reads e as fp16 and recovers the integer from acc + 0.75.
- every schedule lifts b = (r1 + [r1 > q/2]) mod 3 with a strict > (index.js:117).

Uniformly random operands keep the accumulators near sqrt(N) q, far below these bounds, and leave the lift boundary to
chance.  So the rows here are built to reach the bounds: constant rows that hit a bound exactly, and top-of-range random
rows that come close while still telling positions apart.  Each crafted row sits three times in a device-resident
batch of three full 256-row tiles and a partial one: in the first tile, across the boundary of the second and third,
and in the last partial tile.  Every crafted row is compared with the oracle's integer closed forms, pad columns
included, and the whole batch is compared across schedules bit for bit.
"""
import itertools

import numpy as np
import pytest

import ntru_oracle as o

pytestmark = pytest.mark.gpu

AUTO, CORE, TCGEN05, IMMA = 0, 1, 2, 3         # ntru_circom_b200.PATH_*
B = 3 * 256 + 77                               # three full tcgen05 tiles (256 rows of a CTA pair) and 77 rows
S16, S8 = 0x5A5A, 0xA5                         # sentinels of 16-bit and byte outputs: pad columns must be written
ENC_OUT = {"value": 2, "quotientE": 2, "remainderE": 2}
DEC_OUT = {"value": 1, "quotient1": 2, "remainder1": 2, "quotient2": 1, "remainder2": 1}

# (N, q) and why each is here.  The first seven are one tcgen05 geometry branch each (tests/test_output_subsets.py).
SHAPES = [
    (167, 128, "dec1_one_limb"),                          # q <= 256: one K limb, m = 255 is above q
    (509, 2048, "dec1f_one_group"),                       # fp16 first decrypt product at its bound, resident A
    (512, 2048, "pad_memset"),                            # the pad columns are zeroed by memsets
    (677, 2048, "enc_one_unit_dec1f_streamed"),           # ENC message from global memory, fp16 DEC1 with A streamed
    (701, 8192, "dec1_two_limb_one_group"),               # two K limbs, e1 << 2 = 124 at e = q - 1
    (821, 4096, "dec1_two_limb_two_groups_tma_a"),        # two K limbs, A streamed by TMA, even log2 q lift
    (1024, 8192, "fp32_bound_no_imma"),                   # N 2 (q - 1) = 2^24 - 2048: the CUDA-core bound is tightest
    (509, 8192, "largest_limbs_resident_a"),              # h1 = 31, e1 << 2 = 124 with a resident A operand
    (832, 8192, "largest_limbs_top_imma_bucket"),         # largest limbs in the top IMMA bucket (13 column blocks)
    (8, 4, "smallest_q"),                                 # q/2 = 2: the lift boundary values overlap
    (17, 32, "q_half_16"),                                # q/2 = 16, N = 1 mod 16
]
SHAPE_PARAMS = [pytest.param(n, q, id=f"N{n}q{q}-{why}") for n, q, why in SHAPES]


@pytest.fixture(scope="module")
def nb():
    import ntru_circom_b200 as nb
    return nb


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


@pytest.fixture(scope="module")
def engines(nb):
    made = {}

    def get(N, q):
        if (N, q) not in made:
            made[N, q] = nb.Engine(N, 3, q, 0)
        return made[N, q]
    yield get
    for eng in made.values():
        eng.close()


# ---- crafted keys and rows ------------------------------------------------------------------------------------------

def _full(N, v):
    return np.full(N, v, dtype=np.int64)


def _mono(N, k, v):
    a = np.zeros(N, dtype=np.int64)
    a[k] = v
    return a


def _top(q):
    """lowest value of a top-of-range random coefficient: q - q/8 (q - 1 at q = 4)"""
    return q - max(q // 8, 1)


def public_keys(N, q, rng):
    return {"h_all_q_minus_1": _full(N, q - 1), "h_top_random": rng.integers(_top(q), q, N),
            "h_q_minus_1_x0": _mono(N, 0, q - 1), "h_q_minus_1_xN1": _mono(N, N - 1, q - 1),
            "h_random": rng.integers(0, q, N)}


def private_keys(N, rng):
    """(f, fp) pairs.  The engine takes any f in {-1, 0, 1} and fp in [0, p): none of these is a valid NTRU key."""
    one, x0, two_x0 = _full(N, 1), _mono(N, 0, 1), _mono(N, 0, 2)
    return {"f_plus_1_fp_2": (one, 2 * one), "f_minus_1_fp_2": (-one, 2 * one), "f_x0_fp_2": (x0, 2 * one),
            "f_x0_fp_2x0": (x0, two_x0), "f_minus_xN1_fp_2x0": (-_mono(N, N - 1, 1), two_x0),
            "f_random": (rng.integers(-1, 2, N), rng.integers(0, 3, N))}


def encrypt_rows(N, rng):
    """(r, m) byte rows"""
    return {"r_2_m_255": (_full(N, 2), _full(N, 255)), "r_1_m_255": (_full(N, 1), _full(N, 255)),
            "r_random_1_2_m_255": (rng.integers(1, 3, N), _full(N, 255)), "r_0_m_255": (_full(N, 0), _full(N, 255)),
            "r_2_m_random": (_full(N, 2), rng.integers(0, 256, N))}


def decrypt_rows(N, q, rng):
    """e rows.  Under f = x^0 remainder1 equals e, so the lift rows put q/2 - 1, q/2, q/2 + 1 and q - 1 at every
    position (one row per rotation) and decide both sides of the strict > on every schedule; "e_lift_to_2" lifts to
    b = 2 everywhere, which drives the second product under fp = 2 everywhere to its maximum, 4N."""
    j = np.arange(N)
    lift = np.array([q // 2 - 1, q // 2, q // 2 + 1, q - 1])
    to_2 = np.nonzero(o.lift_mod_p(np.arange(q), q) == 2)[0]
    rows = {"e_all_q_minus_1": _full(N, q - 1), "e_q_minus_1_even_0_odd": np.where(j % 2 == 0, q - 1, 0),
            "e_top_random": rng.integers(_top(q), q, N)}
    rows.update({f"e_lift_rotation_{s}": lift[(j + s) % 4] for s in range(4)})
    rows.update({"e_lift_to_2": rng.choice(to_2, N), "e_zero": _full(N, 0)})
    return rows


def _place(n):
    """Batch rows of n crafted rows: the first tile, across the boundary of the second and third tiles, the last tile."""
    assert n <= B - 3 * 256
    j = np.arange(n)
    return np.concatenate([j, 512 - n // 2 + j, B - n + j])


def _copies(a):
    return np.concatenate([a, a, a])


def _device(torch, rows, P, dtype):
    """(n, N) integers -> (n, P) CUDA tensor, zero pad columns (uint16 as int16)"""
    a = np.zeros((rows.shape[0], P), dtype=dtype)
    a[:, :rows.shape[1]] = rows
    return torch.from_numpy(a.view(np.int16) if dtype == np.uint16 else a).cuda()


def _host(t):
    a = t.cpu().numpy()
    return a.view(np.uint16) if a.dtype == np.int16 else a


# ---- calls and checks -----------------------------------------------------------------------------------------------

def same_key_schedules(N, q, op):
    """(name, path, (setter, value, default) or None) of every schedule and tcgen05 variant the shape supports"""
    runs = [("tcgen05", TCGEN05, None), ("tcgen05_cyc_hi", TCGEN05, ("set_schedule", True, False))]
    if op == "decrypt" and 256 < q <= 2048:
        runs += [("tcgen05_dec1_bytes", TCGEN05, ("set_dec1_form", 1, 0)),
                 ("tcgen05_dec1_fp16", TCGEN05, ("set_dec1_form", 2, 0))]
    if N <= 832:                                   # csrc/imma_kernels.cu: imma_supported
        runs.append(("imma", IMMA, None))
    return runs + [("cuda_core", CORE, None)]


def distinct_key_schedules(N):
    return ([("imma", IMMA, None)] if N <= 832 else []) + [("cuda_core", CORE, None)]


def call(eng, torch, op, x, path, option):
    """One device-resident call with every output, into buffers filled with a sentinel."""
    outs = ENC_OUT if op == "encrypt" else DEC_OUT
    out = {k: torch.full((B, eng.pitch), S16 if w == 2 else S8, dtype=torch.int16 if w == 2 else torch.uint8,
                         device="cuda") for k, w in outs.items()}
    eng.set_path(path)
    if option:
        getattr(eng, option[0])(option[1])
    try:
        torch.cuda.synchronize()                   # the engine runs on its own non-blocking stream
        if op == "encrypt":
            eng.encrypt_dev(B, x["r"], x["m"], h_rows=x.get("h_rows"), **out)
        else:
            eng.decrypt_dev(B, x["e"], f_rows=x.get("f_rows"), fp_rows=x.get("fp_rows"), **out)
        eng.sync()
        assert eng.last_path == path, (op, path)
    finally:
        if option:
            getattr(eng, option[0])(option[2])
        eng.set_path(AUTO)
    return out


def expect_rows(got, want, names, what):
    """got: host rows (n, pitch); want: oracle rows (n, w).  Columns [0, w) equal, pad columns [w, pitch) zero."""
    w = want.shape[1]
    diff = np.concatenate([got[:, :w] != want, got[:, w:] != 0], axis=1)
    if diff.any():
        i, c = np.argwhere(diff)[0]
        rows = sorted({names[k] for k in np.nonzero(diff.any(axis=1))[0]})
        pytest.fail(f"{what}: row {names[i]} column {c}: got {got[i, c]}, want {want[i, c] if c < w else 0} "
                    f"({diff.sum()} coefficients differ, rows {rows})")


def check_call(torch, got, want, at, names, what, ref):
    """The crafted rows against the oracle and, if ref is given, the whole batch against ref bit for bit."""
    idx = torch.from_numpy(at).cuda()
    for k, w in want.items():
        expect_rows(_host(got[k][idx]).astype(np.int64), w, names, (what, k))
        if ref is not None:
            assert torch.equal(got[k], ref[1][k]), (what, k, "differs from", ref[0])


def _row_names(names, at):
    return [f"{names[i % len(names)]}@{at[i]}" for i in range(len(at))]


# ---- 1. same key: every schedule, every crafted key ------------------------------------------------------------------

@pytest.mark.parametrize("N,q", SHAPE_PARAMS)
def test_same_key_encrypt_extremes(N, q, engines, torch):
    """Crafted public keys (q - 1 everywhere, top-of-range random, the monomials (q - 1) x^0 and (q - 1) x^(N-1), a
    random control) under r = 2, 1, random {1, 2}, 0 with m = 255: the largest cyclic sums of every schedule and of both
    tcgen05 accumulator column groups."""
    eng = engines(N, q)
    P = eng.pitch
    rng = np.random.default_rng(10 * N + q)
    crafted = encrypt_rows(N, rng)
    at = _place(len(crafted))
    names = _row_names(list(crafted), at)
    r, m = rng.integers(0, 3, (B, N)), rng.integers(0, 256, (B, N))
    r[at] = _copies(np.stack([v[0] for v in crafted.values()]))
    m[at] = _copies(np.stack([v[1] for v in crafted.values()]))
    x = {"r": _device(torch, r, P, np.uint8), "m": _device(torch, m, P, np.uint8)}
    for hname, h in public_keys(N, q, rng).items():
        eng.set_public_key(h.astype(np.uint16))
        want = o.encrypt_batch(h, r[at], m[at], q)
        ref = None
        for sched, path, option in same_key_schedules(N, q, "encrypt"):
            got = call(eng, torch, "encrypt", x, path, option)
            check_call(torch, got, want, at, names, (hname, sched), ref)
            ref = ref or (sched, got)


@pytest.mark.parametrize("N,q", SHAPE_PARAMS)
def test_same_key_decrypt_extremes(N, q, engines, torch):
    """Crafted private keys (f = +1, -1, x^0, -x^(N-1) under fp = 2 everywhere or 2 x^0, a random control) on e rows of
    q - 1, alternating q - 1 / 0, top-of-range random, the lift boundary and rows that lift to b = 2: the first product
    at N (q - 1) in both tcgen05 forms, both sides of the lift on every schedule, the second product at 4N."""
    eng = engines(N, q)
    P = eng.pitch
    rng = np.random.default_rng(20 * N + q)
    crafted = decrypt_rows(N, q, rng)
    at = _place(len(crafted))
    names = _row_names(list(crafted), at)
    e = rng.integers(0, q, (B, N))
    e[at] = _copies(np.stack(list(crafted.values())))
    x = {"e": _device(torch, e, P, np.uint16)}
    for kname, (f, fp) in private_keys(N, rng).items():
        eng.set_private_key(f.astype(np.int8), fp.astype(np.uint8))
        want = o.decrypt_batch(f, fp, e[at], q)
        ref = None
        for sched, path, option in same_key_schedules(N, q, "decrypt"):
            got = call(eng, torch, "decrypt", x, path, option)
            check_call(torch, got, want, at, names, (kname, sched), ref)
            ref = ref or (sched, got)


# ---- 2. distinct keys: the crafted keys as per-row keys --------------------------------------------------------------

@pytest.mark.parametrize("N,q", SHAPE_PARAMS)
def test_distinct_keys_encrypt_extremes(N, q, engines, torch):
    """Every crafted public key with every crafted (r, m) row as h_rows, on the IMMA and CUDA-core schedules."""
    eng = engines(N, q)
    P = eng.pitch
    rng = np.random.default_rng(30 * N + q)
    keys, rows = public_keys(N, q, rng), encrypt_rows(N, rng)
    pairs = list(itertools.product(keys, rows))
    at = _place(len(pairs))
    names = _row_names([f"{k}/{v}" for k, v in pairs], at)
    h, r, m = rng.integers(0, q, (B, N)), rng.integers(0, 3, (B, N)), rng.integers(0, 256, (B, N))
    h[at] = _copies(np.stack([keys[k] for k, _ in pairs]))
    r[at] = _copies(np.stack([rows[v][0] for _, v in pairs]))
    m[at] = _copies(np.stack([rows[v][1] for _, v in pairs]))
    x = {"h_rows": _device(torch, h, P, np.uint16), "r": _device(torch, r, P, np.uint8),
         "m": _device(torch, m, P, np.uint8)}
    want = o.encrypt_batch(h[at], r[at], m[at], q)
    ref = None
    for sched, path, option in distinct_key_schedules(N):
        got = call(eng, torch, "encrypt", x, path, option)
        check_call(torch, got, want, at, names, ("h_rows", sched), ref)
        ref = ref or (sched, got)


@pytest.mark.parametrize("N,q", SHAPE_PARAMS)
def test_distinct_keys_decrypt_extremes(N, q, engines, torch):
    """Every crafted private key with every crafted e row as f_rows / fp_rows, on the IMMA and CUDA-core schedules."""
    eng = engines(N, q)
    P = eng.pitch
    rng = np.random.default_rng(40 * N + q)
    keys, rows = private_keys(N, rng), decrypt_rows(N, q, rng)
    pairs = list(itertools.product(keys, rows))
    at = _place(len(pairs))
    names = _row_names([f"{k}/{v}" for k, v in pairs], at)
    f, fp, e = rng.integers(-1, 2, (B, N)), rng.integers(0, 3, (B, N)), rng.integers(0, q, (B, N))
    f[at] = _copies(np.stack([keys[k][0] for k, _ in pairs]))
    fp[at] = _copies(np.stack([keys[k][1] for k, _ in pairs]))
    e[at] = _copies(np.stack([rows[v] for _, v in pairs]))
    x = {"f_rows": _device(torch, f, P, np.int8), "fp_rows": _device(torch, fp, P, np.uint8),
         "e": _device(torch, e, P, np.uint16)}
    want = o.decrypt_batch(f[at], fp[at], e[at], q)
    ref = None
    for sched, path, option in distinct_key_schedules(N):
        got = call(eng, torch, "decrypt", x, path, option)
        check_call(torch, got, want, at, names, ("f_rows", sched), ref)
        ref = ref or (sched, got)


# ---- 3. wide messages at the fp32 bound ------------------------------------------------------------------------------

@pytest.mark.parametrize("N,q", [pytest.param(1024, 8192, id="N1024q8192-fp32_bound"),
                                 pytest.param(701, 8192, id="N701q8192-hrss701")])
def test_wide_messages_at_the_fp32_bound(N, q, engines, torch):
    """ntru_encrypt_batch_wide (Engine.encrypt_batch with uint16 m, some m > 255) under every crafted public key, with
    m = q - 1 and top-of-range random m: at N = 1024, q = 8192 with r = 2 and h = q - 1 the cyclic sum is 2^24 - 2048
    and the message brings it past 2^24, so it must be added after the fp32 accumulation.  Wide messages always take
    the CUDA-core schedule.  Crafted rows against the oracle; the whole batch against the tcgen05 encryption of m = 0
    plus m modulo q."""
    eng = engines(N, q)
    rng = np.random.default_rng(50 * N + q)
    rs = {"r_2": _full(N, 2), "r_1": _full(N, 1), "r_random_1_2": rng.integers(1, 3, N), "r_0": _full(N, 0)}
    ms = {"m_q_minus_1": _full(N, q - 1), "m_top_random": rng.integers(_top(q), q, N)}
    pairs = list(itertools.product(rs, ms))
    at = _place(len(pairs))
    names = _row_names([f"{a}/{b}" for a, b in pairs], at)
    r, m = rng.integers(0, 3, (B, N)), rng.integers(0, q, (B, N))
    r[at] = _copies(np.stack([rs[a] for a, _ in pairs]))
    m[at] = _copies(np.stack([ms[b] for _, b in pairs]))
    r8, m16 = r.astype(np.uint8), m.astype(np.uint16)
    for hname, h in public_keys(N, q, rng).items():
        eng.set_public_key(h.astype(np.uint16))
        enc = eng.encrypt_batch(r8, m16)
        assert eng.last_path == CORE, hname
        want = o.encrypt_batch(h, r[at], m[at], q)
        for k, w in want.items():
            expect_rows(enc[k][at].astype(np.int64), w, names, (hname, "wide", k))
        eng.set_path(TCGEN05)
        try:
            base = eng.encrypt_batch(r8, np.zeros((B, N), dtype=np.uint8))
        finally:
            eng.set_path(AUTO)
        shifted = (base["value"].astype(np.int64) + m) % q
        assert np.array_equal(enc["value"], shifted), (hname, "value")
        assert np.array_equal(enc["remainderE"][:, :N], shifted) and not enc["remainderE"][:, N:].any(), (hname, "remainderE")
        assert np.array_equal(enc["quotientE"], base["quotientE"]), (hname, "quotientE")


# ---- 4. ntru_muldiv_dev over its whole documented input range -------------------------------------------------------

MULDIV_SHAPES = [pytest.param(n, q, id=f"N{n}q{q}") for n in (191, 192, 193, 512, 513, 704, 705, 832) for q in (2048, 8192)]
MULDIV_SHAPES.append(pytest.param(167, 128, id="N167q128-q_le_256"))


def muldiv(eng, torch, x, y, mod_p, pad):
    """ntru_muldiv_dev on the rows x (int8) and y (uint16, or bytes in mod-p mode); pad: the input pad columns hold
    0xFF bytes instead of zeros.  Returns the host quotient and remainder rows, pad columns included."""
    N, P, n = eng.N, eng.pitch, x.shape[0]
    ydt = np.uint8 if mod_p else np.uint16
    xs, ys = np.zeros((n, P), dtype=np.int8), np.zeros((n, P), dtype=ydt)
    xs[:, :N], ys[:, :N] = x, y
    if pad:
        xs[:, N:], ys[:, N:] = -1, np.iinfo(ydt).max
    xd = torch.from_numpy(xs).cuda()
    yd = torch.from_numpy(ys if mod_p else ys.view(np.int16)).cuda()
    odt, s = (torch.uint8, S8) if mod_p else (torch.int16, S16)
    quo, rem = (torch.full((n, P), s, dtype=odt, device="cuda") for _ in range(2))
    torch.cuda.synchronize()
    eng.muldiv_dev(n, xd, yd, mod_p, quotient=quo, remainder=rem)
    eng.sync()
    return _host(quo).astype(np.int64), _host(rem).astype(np.int64)


def muldiv_want(x, y, N, mod):
    """multiplyPolynomials(x, y, mod) then dividePolynomials(., 1 - x^N, mod) with the literal x (2, or -1)"""
    quo, rem = np.zeros((x.shape[0], N), dtype=np.int64), np.zeros((x.shape[0], N), dtype=np.int64)
    for i in range(x.shape[0]):
        d = o.divide_by_I_closed(o.multiply_polynomials_exact(x[i].tolist(), y[i].tolist(), mod), N, mod)
        quo[i, :len(d["quotient"])] = d["quotient"]
        rem[i, :len(d["remainder"])] = d["remainder"]
    return quo, rem


def _x_rows(N, rng):
    j = np.arange(N)
    return {"x_2": _full(N, 2), "x_minus_1": _full(N, -1), "x_2_minus_1_alternating": np.where(j % 2 == 0, 2, -1),
            "x_random": rng.integers(-1, 3, N)}


def _check_muldiv(eng, torch, x, y, names, mod_p, what):
    N = eng.N
    want_q, want_r = muldiv_want(x, y, N, 3 if mod_p else eng.q)
    quo, rem = muldiv(eng, torch, x, y, mod_p, pad=False)
    expect_rows(quo, want_q, names, (what, "quotient"))
    expect_rows(rem, want_r, names, (what, "remainder"))
    quo2, rem2 = muldiv(eng, torch, x, y, mod_p, pad=True)
    assert np.array_equal(quo2, quo) and np.array_equal(rem2, rem), (what, "input pad columns of 0xFF bytes count")


@pytest.mark.parametrize("N,q", MULDIV_SHAPES)
def test_muldiv_mod_q_full_uint16_range(N, q, engines, torch):
    """Mod-q mode, y anywhere in [0, 2^16): 65535, 0x8000, 0x7FFF, 0xFF00, 0x00FF and random 16-bit rows under x = 2,
    -1, alternating 2 / -1 and random in [-1, 2], at the N edges of the IMMA buckets.  Quotient and remainder against
    the oracle, pad columns zero, and the same results with the input pad columns full of 0xFF bytes."""
    eng = engines(N, q)
    rng = np.random.default_rng(60 * N + q)
    xs = _x_rows(N, rng)
    ys = {"y_ffff": _full(N, 0xFFFF), "y_8000": _full(N, 0x8000), "y_7fff": _full(N, 0x7FFF), "y_ff00": _full(N, 0xFF00),
          "y_00ff": _full(N, 0x00FF), "y_random": rng.integers(0, 1 << 16, N)}
    pairs = list(itertools.product(xs, ys))
    x = np.concatenate([np.stack([xs[a] for a, _ in pairs]), rng.integers(-1, 3, (8, N))])     # and 8 random rows
    y = np.concatenate([np.stack([ys[b] for _, b in pairs]), rng.integers(0, 1 << 16, (8, N))])
    names = [f"{a}/{b}" for a, b in pairs] + [f"random_{i}" for i in range(8)]
    _check_muldiv(eng, torch, x, y, names, False, "mod q")


@pytest.mark.parametrize("N,q", MULDIV_SHAPES)
def test_muldiv_mod_p_both_ends(N, q, engines, torch):
    """Mod-p mode, y bytes in [0, p): x = 2 against y = 2 gives products up to 4N, x = -1 against y = 2 down to -2N,
    which the kernel corrects through 65536 = 1 (mod 3).  Against the oracle modulo 3, pad columns zero, and the same
    results with the input pad columns full of 0xFF bytes."""
    eng = engines(N, q)
    rng = np.random.default_rng(70 * N + q)
    xs = _x_rows(N, rng)
    ys = {"y_2": _full(N, 2), "y_random": rng.integers(0, 3, N)}
    pairs = list(itertools.product(xs, ys))
    x = np.stack([xs[a] for a, _ in pairs])
    y = np.stack([ys[b] for _, b in pairs])
    _check_muldiv(eng, torch, x, y, [f"{a}/{b}" for a, b in pairs], True, "mod p")
