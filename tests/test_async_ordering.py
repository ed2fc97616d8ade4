"""Device-resident calls with work still in flight: key uploads, option changes and stream switches while kernels are
queued, host-buffer calls right after queued device work, and two contexts on one device.

Every context here runs on a non-blocking stream: the one ntru_create makes, or torch streams.  Nothing then orders a
host-side change of the context against kernels already queued except the library itself (include/ntru_b200.h:
setters apply to calls made after them, queued calls keep what they were queued with, ntru_set_stream orders the new
stream after the work queued on the old one).  torch writes the inputs on its own stream; torch.cuda.synchronize()
orders them before the engine's first call, and eng.sync() orders the engine's outputs before torch reads them.

The first call of each sequence runs for milliseconds, far longer than a key upload or a stream switch takes on the
host.  Every result is checked twice: the whole batch, pad columns included, bit for bit against the same call on a
separate context that holds only the one key and is synchronised after every call; and a sample of rows (first, last,
the last 256-row tile, a stride through the batch) against the oracle.
"""
import numpy as np
import pytest

import ntru_oracle as o

pytestmark = pytest.mark.gpu

CORE, TCGEN05, IMMA = 1, 2, 3          # ntru_circom_b200.PATH_CUDA_CORE, PATH_TENSOR, PATH_IMMA
ENC_KEYS = ("value", "quotientE", "remainderE")
DEC_KEYS = ("value", "quotient1", "remainder1", "quotient2", "remainder2")
GOT_FILL = (-1, 0xAB)                  # pre-fill of the outputs under test (int16 rows, byte rows) ...
REF_FILL = (0x1234, 0x5A)              # ... and of the reference's: a column neither call writes cannot match
SLICE = 1 << 18                        # rows per reference call


@pytest.fixture(scope="module")
def nb():
    import ntru_circom_b200 as nb
    return nb


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


def _keys(golden, cfg):
    """key A: the golden key of the parameter set; key B: random coefficients (the engine takes any h in [0, q),
    f in {-1, 0, 1} and fp in [0, p))"""
    g = golden(cfg)
    N, q = int(g["N"]), int(g["q"])
    rng = np.random.default_rng(N + 1)
    a = {"h": g["h"].astype(np.int64), "f": g["f"].astype(np.int64), "fp": g["fp"].astype(np.int64)}
    b = {"h": rng.integers(0, q, N), "f": rng.integers(-1, 2, N), "fp": rng.integers(0, 3, N)}
    return a, b


def _set_key(eng, key, op=None):
    if op in (None, "encrypt"):
        eng.set_public_key(key["h"].astype(np.uint16))
    if op in (None, "decrypt"):
        eng.set_private_key(key["f"].astype(np.int8), key["fp"].astype(np.uint8))


def _engine(nb, cfg, key):
    c = o.CONFIGS[cfg]
    eng = nb.Engine(c["N"], c["p"], c["q"], 0)          # no set_stream: the context's own non-blocking stream
    _set_key(eng, key)
    return eng


@pytest.fixture(scope="module")
def refs(nb, golden):
    """The synchronous references: one context per parameter set and key (0 = A, 1 = B)."""
    cache = {}

    def get(cfg, which):
        if (cfg, which) not in cache:
            cache[cfg, which] = _engine(nb, cfg, _keys(golden, cfg)[which])
        return cache[cfg, which]
    yield get
    for e in cache.values():
        e.close()


@pytest.fixture
def fresh(nb):
    """Contexts under test, closed when the test ends."""
    made = []

    def make(cfg, key):
        made.append(_engine(nb, cfg, key))
        return made[-1]
    yield make
    for e in made:
        e.close()


def _rows(torch, gen, B, P, N, lo, hi, dtype):
    t = torch.zeros((B, P), dtype=dtype, device="cuda")
    t[:, :N] = torch.randint(lo, hi, (B, N), generator=gen, device="cuda", dtype=dtype)
    return t


def _inputs(torch, eng, op, B, seed):
    """(r, m) of an encrypt or (e,) of a decrypt: B pitched device rows with zero pad columns"""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    N, P = eng.N, eng.pitch
    if op == "encrypt":
        return _rows(torch, gen, B, P, N, 0, 3, torch.uint8), _rows(torch, gen, B, P, N, 0, 2, torch.uint8)
    return (_rows(torch, gen, B, P, N, 0, eng.q, torch.int16),)


def _outs(torch, op, B, P, fill):
    w16, w8 = fill
    if op == "encrypt":
        return {k: torch.full((B, P), w16, dtype=torch.int16, device="cuda") for k in ENC_KEYS}
    return {k: torch.full((B, P), w16, dtype=torch.int16, device="cuda") if k in ("quotient1", "remainder1")
            else torch.full((B, P), w8, dtype=torch.uint8, device="cuda") for k in DEC_KEYS}


def _call(eng, op, x, out):
    if op == "encrypt":
        eng.encrypt_dev(x[0].shape[0], x[0], x[1], **out)
    else:
        eng.decrypt_dev(x[0].shape[0], x[0], **out)


def _warm(torch, eng, op, x, rows):
    """One call of `rows` rows before the sequence under test.  Kernel attributes, tensor maps and scratch are then set
    up, so the sequence allocates nothing: a cudaFree would synchronise the device and close the window under test."""
    xs = tuple(t[:rows] for t in x)
    out = _outs(torch, op, rows, x[0].shape[1], GOT_FILL)
    torch.cuda.synchronize()
    _call(eng, op, xs, out)
    eng.sync()


def _host(t):
    a = t.cpu().numpy()
    return a.view(np.uint16) if a.dtype == np.int16 else a


def _sample(B):
    """first and last rows, the last 256-row tile (a tcgen05 CTA pair's) and a stride through the batch"""
    return sorted({0, 1, B - 257, B - 256, B - 129, B - 128, B - 2, B - 1} | set(range(0, B, B // 16)))


def _check_ref(torch, ref, path, op, x, got, what):
    """got == the same call on the synchronous reference context, bit for bit over whole pitched rows.  The reference
    runs on slices of SLICE rows (a row's results depend on that row alone), which bounds its device memory."""
    B, P = x[0].shape
    ref.set_path(path)
    for s in range(0, B, SLICE):
        xs = tuple(t[s:s + SLICE] for t in x)
        want = _outs(torch, op, xs[0].shape[0], P, REF_FILL)
        torch.cuda.synchronize()
        _call(ref, op, xs, want)
        ref.sync()
        assert ref.last_path == path
        for k, w in want.items():
            assert torch.equal(got[k][s:s + SLICE], w), (what, k, s)


def _check_oracle(torch, cfg, key, op, x, got, what):
    c = o.CONFIGS[cfg]
    N, q, p = c["N"], c["q"], c["p"]
    idx = torch.tensor(_sample(x[0].shape[0]), device="cuda")
    rows = [_host(t[idx])[:, :N].astype(np.int64) for t in x]
    if op == "encrypt":
        want = o.encrypt_batch(key["h"], rows[0], rows[1], q)
    else:
        want = o.decrypt_batch(key["f"], key["fp"], rows[0], q, p)
    for k in got:
        a = _host(got[k][idx])
        w = want[k].shape[1]
        assert np.array_equal(a[:, :w], want[k]), (what, k)
        assert not a[:, w:].any(), (what, k, "pad")


def _check(torch, refs, cfg, which, key, path, op, x, got, what):
    _check_ref(torch, refs(cfg, which), path, op, x, got, what)
    _check_oracle(torch, cfg, key, op, x, got, what)


def _first_call_rows(cfg, path):
    """Several milliseconds of kernel time by DESIGN.md's rates.  N = 701 takes 2^19 rows on the tensor schedules: as
    much work as 2^20 rows at N = 509, with half the memory."""
    if path == CORE:
        return 1 << 17
    return 1 << 20 if cfg == "hps509" else 1 << 19


# ---- 1. key change with work in flight ------------------------------------------------------------------------------

@pytest.mark.parametrize("path", [CORE, IMMA, TCGEN05], ids=["cuda_core", "imma", "tcgen05"])
@pytest.mark.parametrize("op", ["encrypt", "decrypt"])
@pytest.mark.parametrize("cfg", ["hps509", "hrss701"])
def test_key_change_with_work_in_flight(cfg, op, path, torch, golden, refs, fresh):
    """encrypt_dev under key A, set_public_key(B) with no synchronisation, encrypt_dev of the same r and m: every row of
    the first batch is key A's, every row of the second key B's.  Likewise decrypt_dev and set_private_key, all five
    outputs.  The CUDA-core and IMMA schedules read the key rows while they run; the tcgen05 schedule reads the key
    matrices that the setter rebuilds from them.  hrss701 (q = 8192) runs the byte-limb first decrypt product."""
    key_a, key_b = _keys(golden, cfg)
    eng = fresh(cfg, key_a)
    eng.set_path(path)
    B = _first_call_rows(cfg, path)
    x = _inputs(torch, eng, op, B, seed=B + eng.N)
    _warm(torch, eng, op, x, 4096)
    got = [_outs(torch, op, B, eng.pitch, GOT_FILL) for _ in range(2)]
    torch.cuda.synchronize()
    _call(eng, op, x, got[0])
    _set_key(eng, key_b, op)
    _call(eng, op, x, got[1])
    eng.sync()
    assert eng.last_path == path
    for which, key in enumerate((key_a, key_b)):
        _check(torch, refs, cfg, which, key, path, op, x, got[which], (cfg, op, path, "AB"[which]))


# ---- 2. option changes with work in flight ---------------------------------------------------------------------------

# option -> (schedule of the calls, Engine setter, the values set before each of the queued calls).  The forms and
# arrangements give the same results bit for bit (include/ntru_b200.h), so every call equals the reference on its
# schedule.  dec1_form and epilogue rebuild key matrices in place (their buffers only grow) while calls that read them
# are queued.
OPTION_CHANGES = {
    "dec1_form": (TCGEN05, "set_dec1_form", [1, 2, 1]),
    "epilogue": (TCGEN05, "set_epilogue", [1, 2, 0]),
    "schedule": (TCGEN05, "set_schedule", [True, False, True]),
    "imma_form": (IMMA, "set_imma_form", [True, False, True]),
    "path": (None, "set_path", [TCGEN05, CORE, IMMA, 0]),
}


@pytest.mark.parametrize("option", list(OPTION_CHANGES))
def test_option_change_with_work_in_flight(option, torch, golden, refs, fresh):
    """Queued encrypt_dev + decrypt_dev of its ciphertexts, the option changed with no synchronisation, the same pair
    again, and so on: every call equals its reference and the oracle."""
    cfg, B = "hps509", 1 << 17
    path, setter, values = OPTION_CHANGES[option]
    key = _keys(golden, cfg)[0]
    eng = fresh(cfg, key)
    if path is not None:
        eng.set_path(path)
    set_option = getattr(eng, setter)
    x = _inputs(torch, eng, "encrypt", B, seed=7)
    for v in values:
        set_option(v)
        _warm(torch, eng, "encrypt", x, 4096)
        _warm(torch, eng, "decrypt", (x[1].to(torch.int16),), 4096)
    set_option(values[0])
    enc = [_outs(torch, "encrypt", B, eng.pitch, GOT_FILL) for _ in values]
    dec = [_outs(torch, "decrypt", B, eng.pitch, GOT_FILL) for _ in values]
    paths = []
    torch.cuda.synchronize()
    for i, v in enumerate(values):
        if i:
            set_option(v)
        _call(eng, "encrypt", x, enc[i])
        paths.append(eng.last_path)
        _call(eng, "decrypt", (enc[i]["value"],), dec[i])
        assert eng.last_path == paths[-1]
    eng.sync()
    assert paths == ([TCGEN05, CORE, IMMA, TCGEN05] if option == "path" else [path] * len(values))
    for i, v in enumerate(values):
        _check(torch, refs, cfg, 0, key, paths[i], "encrypt", x, enc[i], (option, v, "encrypt"))
        _check(torch, refs, cfg, 0, key, paths[i], "decrypt", (enc[i]["value"],), dec[i], (option, v, "decrypt"))


# ---- 3. stream switch with work in flight ----------------------------------------------------------------------------

def _two_streams(torch, eng):
    """A context moved onto caller stream S1; S2 is where it goes next."""
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    assert s1.cuda_stream != s2.cuda_stream
    eng.set_stream(s1.cuda_stream)
    return s1, s2


def test_stream_switch_decrypt_tcgen05(torch, golden, refs, fresh):
    """decrypt_dev on S1, set_stream(S2), decrypt_dev of other ciphertexts on S2: the tcgen05 schedule keeps the lifted
    polynomial b of both products in scratch the context owns."""
    cfg, B = "hps509", 1 << 19
    key = _keys(golden, cfg)[0]
    eng = fresh(cfg, key)
    eng.set_path(TCGEN05)
    s1, s2 = _two_streams(torch, eng)
    x = [_inputs(torch, eng, "decrypt", B, seed=s) for s in (1, 2)]
    _warm(torch, eng, "decrypt", x[0], B)
    got = [_outs(torch, "decrypt", B, eng.pitch, GOT_FILL) for _ in range(2)]
    torch.cuda.synchronize()
    _call(eng, "decrypt", x[0], got[0])
    eng.set_stream(s2.cuda_stream)
    _call(eng, "decrypt", x[1], got[1])
    torch.cuda.synchronize()
    for i in range(2):
        _check(torch, refs, cfg, 0, key, TCGEN05, "decrypt", x[i], got[i], ("S1", "S2")[i])


def _oracle_sum(e, N, q):
    """o.sum_batch over every row of device rows e, a slice at a time (the fold is associative modulo q)"""
    parts = [o.sum_batch(_host(e[s:s + SLICE])[:, :N].astype(np.int64), q) for s in range(0, e.shape[0], SLICE)]
    return o.sum_batch(np.stack(parts), q)


def test_stream_switch_sum(torch, golden, refs, fresh):
    """sum_partial_dev + sum_finalize_dev of 2^20 rows on S1, set_stream(S2), the same of other 2^20 rows on S2, then a
    small sum on S2.  The sum tree's rows and tickets belong to the context; two overlapping trees can leave a ticket
    non-zero, and the small sum (one CTA, expecting a zero ticket) then returns a wrong total."""
    cfg, B, small = "hps509", 1 << 20, 300
    key = _keys(golden, cfg)[0]
    eng = fresh(cfg, key)
    N, P, q = eng.N, eng.pitch, eng.q
    s1, s2 = _two_streams(torch, eng)
    e = [_inputs(torch, eng, "decrypt", n, seed=10 + i)[0] for i, n in enumerate((B, B, small))]
    partial = torch.zeros((3, P), dtype=torch.int32, device="cuda")
    out = torch.full((3, P), -1, dtype=torch.int16, device="cuda")
    warm_partial = torch.zeros(P, dtype=torch.int32, device="cuda")
    warm_out = torch.empty(P, dtype=torch.int16, device="cuda")
    torch.cuda.synchronize()
    eng.sum_partial_dev(small, e[2], warm_partial)         # allocates and zeroes the tree scratch
    eng.sum_finalize_dev(warm_partial, warm_out)
    eng.sync()
    eng.sum_partial_dev(B, e[0], partial[0])
    eng.sum_finalize_dev(partial[0], out[0])
    eng.set_stream(s2.cuda_stream)
    for i in (1, 2):
        eng.sum_partial_dev(e[i].shape[0], e[i], partial[i])
        eng.sum_finalize_dev(partial[i], out[i])
    torch.cuda.synchronize()
    ref = refs(cfg, 0)
    for i in range(3):
        rp = torch.zeros(P, dtype=torch.int32, device="cuda")
        ro = torch.full((P,), 0x1234, dtype=torch.int16, device="cuda")
        torch.cuda.synchronize()
        ref.sum_partial_dev(e[i].shape[0], e[i], rp)
        ref.sum_finalize_dev(rp, ro)
        ref.sync()
        assert torch.equal(out[i], ro), i
        got = _host(out[i])
        assert np.array_equal(got[:N], _oracle_sum(e[i], N, q)), i
        assert not got[N:].any(), i


def _keygen_outs(torch, B, P):
    return {"fq": torch.full((B, P), -1, dtype=torch.int16, device="cuda"),
            "fp": torch.full((B, P), 0xAB, dtype=torch.uint8, device="cuda"),
            "h": torch.full((B, P), -1, dtype=torch.int16, device="cuda"),
            "valid": torch.full((B,), 0xAB, dtype=torch.uint8, device="cuda")}


def _keygen(eng, f, g, out):
    eng.keygen_dev(f.shape[0], f, g, out["fq"], out["fp"], out["h"], out["valid"])


def test_stream_switch_keygen(torch, golden, refs, fresh):
    """keygen_dev on S1, set_stream(S2), keygen_dev of other f and g on S2: the Newton lifting and h run in scratch the
    context owns.  The oracle: validity of every row (at N = 509, Phi_N is irreducible modulo 2 and 3, so f is
    invertible modulo p iff f(1) != 0 mod p and f is not constant mod p) and fq, fp, h of the valid sampled rows."""
    cfg, B = "hps509", 1 << 16
    c = o.CONFIGS[cfg]
    eng = fresh(cfg, _keys(golden, cfg)[0])
    N, P = eng.N, eng.pitch
    s1, s2 = _two_streams(torch, eng)
    gen = torch.Generator(device="cuda").manual_seed(3)
    fg = [[_rows(torch, gen, B, P, N, -1, 2, torch.int8) for _ in range(2)] for _ in range(2)]
    warm = _keygen_outs(torch, B, P)
    got = [_keygen_outs(torch, B, P) for _ in range(2)]
    torch.cuda.synchronize()
    _keygen(eng, *fg[0], warm)                             # sizes the lifting scratch for B rows
    eng.sync()
    _keygen(eng, *fg[0], got[0])
    eng.set_stream(s2.cuda_stream)
    _keygen(eng, *fg[1], got[1])
    torch.cuda.synchronize()
    ref = refs(cfg, 0)
    for i in range(2):
        want = _keygen_outs(torch, B, P)
        for v in want.values():
            v.fill_(0x5A)
        torch.cuda.synchronize()
        _keygen(ref, *fg[i], want)
        ref.sync()
        for k in want:
            assert torch.equal(got[i][k], want[k]), (i, k)
        f, g = (_host(t)[:, :N].astype(np.int64) for t in fg[i])
        s = f.sum(axis=1)
        const2 = (f != 0).all(axis=1) | (f == 0).all(axis=1)
        const3 = (f == f[:, :1]).all(axis=1)
        valid = (s % 2 == 1) & (s % 3 != 0) & ~const2 & ~const3
        assert np.array_equal(_host(got[i]["valid"]).astype(bool), valid), i
        fq, fp, h = (_host(got[i][k]) for k in ("fq", "fp", "h"))
        checked = 0
        for b in _sample(B):
            if not valid[b]:
                assert not fq[b].any() and not fp[b].any() and not h[b].any(), (i, b)
                continue
            k = o.NTRU(dict(c))
            k.loadPrivateKeyF(f[b].tolist())
            k.g = g[b].tolist()
            k.generatePublicKeyH()
            assert fq[b].tolist() == o.expand_array(k.fq, P, 0), (i, b, "fq")
            assert fp[b].tolist() == o.expand_array(k.fp, P, 0), (i, b, "fp")
            assert h[b].tolist() == o.expand_array(k.h, P, 0), (i, b, "h")
            checked += 1
        assert checked >= 3, i


def _verify_oracle(f, fq, fp, g, out, N, q, p, rows):
    for i in rows:
        for case, a, b, mod in (("fq", fq[i], f[i], q), ("fp", fp[i], f[i], p), ("h", fq[i] * p, g[i], q)):
            # the reference multiplies by the witness value of a -1 (q-1 / p-1, index.js:151-156)
            d = o.divide_by_I_closed(o.multiply_polynomials_exact(list(map(int, a)), [mod - 1 if x == -1 else int(x) for x in b], mod),
                                     N, mod)
            assert out["quotient_" + case][i].tolist() == o.expand_array(d["quotient"], N + 1, 0), (i, case)
            assert out["remainder_" + case][i].tolist() == o.expand_array(d["remainder"], N + 1, 0), (i, case)


def test_stream_switch_decrypt_then_verify_keys(torch, golden, refs, fresh):
    """decrypt_dev on S1 (tcgen05), set_stream(S2), verify_keys_batch on S2: its h case scales fq into the same scratch
    that holds the decrypt's lifted b."""
    cfg, B, Bv = "hps509", 1 << 19, 4096
    key = _keys(golden, cfg)[0]
    eng = fresh(cfg, key)
    N, q, p = eng.N, eng.q, eng.p
    eng.set_path(TCGEN05)
    s1, s2 = _two_streams(torch, eng)
    rng = np.random.default_rng(19)
    f, g = rng.integers(-1, 2, size=(Bv, N)), rng.integers(-1, 2, size=(Bv, N))
    fq, fp = rng.integers(0, q, size=(Bv, N)), rng.integers(0, p, size=(Bv, N))
    vin = (f.astype(np.int8), fq.astype(np.uint16), fp.astype(np.uint8), g.astype(np.int8))
    x = _inputs(torch, eng, "decrypt", B, seed=5)
    _warm(torch, eng, "decrypt", x, B)                     # the lifted-b scratch holds B rows: no call below grows it
    eng.verify_keys_batch(*vin)                            # and the host pipeline's buffers are allocated
    got = _outs(torch, "decrypt", B, eng.pitch, GOT_FILL)
    torch.cuda.synchronize()
    _call(eng, "decrypt", x, got)
    eng.set_stream(s2.cuda_stream)
    ver = eng.verify_keys_batch(*vin)
    torch.cuda.synchronize()
    _check(torch, refs, cfg, 0, key, TCGEN05, "decrypt", x, got, "decrypt on S1")
    want = refs(cfg, 0).verify_keys_batch(*vin)
    for k in want:
        assert np.array_equal(ver[k], want[k]), k
    _verify_oracle(f, fq, fp, g, ver, N, q, p, _sample(Bv))


# ---- 4. host-buffer calls right after queued device work -------------------------------------------------------------

def test_host_buffer_calls_after_queued_device_work(torch, golden, refs, fresh):
    """encrypt_dev of 2^20 rows, then with no synchronisation encrypt_batch and sum on host buffers: all three correct."""
    cfg, B, Bh = "hps509", 1 << 20, 4096
    key = _keys(golden, cfg)[0]
    eng = fresh(cfg, key)
    N, q = eng.N, eng.q
    rng = np.random.default_rng(29)
    r_h = rng.integers(0, 3, size=(Bh, N)).astype(np.uint8)
    m_h = rng.integers(0, 2, size=(Bh, N)).astype(np.uint8)
    e_h = rng.integers(0, q, size=(Bh, N)).astype(np.uint16)
    x = _inputs(torch, eng, "encrypt", B, seed=31)
    _warm(torch, eng, "encrypt", x, 4096)
    eng.encrypt_batch(r_h, m_h)                            # the host pipeline's buffers are allocated
    eng.sum(e_h)
    got = _outs(torch, "encrypt", B, eng.pitch, GOT_FILL)
    torch.cuda.synchronize()
    _call(eng, "encrypt", x, got)
    path = eng.last_path
    enc_h = eng.encrypt_batch(r_h, m_h)
    sum_h = eng.sum(e_h)
    eng.sync()
    assert path == TCGEN05
    _check(torch, refs, cfg, 0, key, path, "encrypt", x, got, "encrypt_dev")
    want = o.encrypt_batch(key["h"], r_h.astype(np.int64), m_h.astype(np.int64), q)
    for k in ENC_KEYS:
        assert np.array_equal(enc_h[k], want[k]), k
    assert np.array_equal(sum_h, o.sum_batch(e_h, q))


# ---- 5. two contexts on one device -----------------------------------------------------------------------------------

def test_two_contexts_interleaved(torch, golden, refs, fresh):
    """Two contexts, keys A and B, each on its own stream, their encrypt, decrypt and sum calls interleaved: each
    context's results equal its own reference, so the two share no state."""
    cfg, B = "hps509", 1 << 18
    keys = _keys(golden, cfg)
    engs = [fresh(cfg, k) for k in keys]
    N, P, q = engs[0].N, engs[0].pitch, engs[0].q
    x = [_inputs(torch, engs[0], "encrypt", B, seed=41 + i) for i in range(2)]
    for i in range(2):
        _warm(torch, engs[i], "encrypt", x[i], 4096)
    enc = [_outs(torch, "encrypt", B, P, GOT_FILL) for _ in range(2)]
    dec = [_outs(torch, "decrypt", B, P, GOT_FILL) for _ in range(2)]
    partial = torch.zeros((2, P), dtype=torch.int32, device="cuda")
    sums = torch.full((2, P), -1, dtype=torch.int16, device="cuda")
    torch.cuda.synchronize()
    for i in range(2):
        _call(engs[i], "encrypt", x[i], enc[i])
    for i in range(2):
        _call(engs[i], "decrypt", (enc[i]["value"],), dec[i])
    for i in range(2):
        engs[i].sum_partial_dev(B, enc[i]["value"], partial[i])
    for i in range(2):
        engs[i].sum_finalize_dev(partial[i], sums[i])
    for i in range(2):
        engs[i].sync()
    for i in range(2):
        path = engs[i].last_path
        assert path == TCGEN05
        _check(torch, refs, cfg, i, keys[i], path, "encrypt", x[i], enc[i], ("encrypt", i))
        _check(torch, refs, cfg, i, keys[i], path, "decrypt", (enc[i]["value"],), dec[i], ("decrypt", i))
        got = _host(sums[i])
        assert np.array_equal(got[:N], _oracle_sum(enc[i]["value"], N, q)) and not got[N:].any(), i
