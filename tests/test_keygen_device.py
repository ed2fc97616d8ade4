"""Key generation on the device: the divstep inversions modulo 2 and 3 (ntru_keygen_dev), device-drawn key pairs
(ntru_generate_keys_dev) and NTRU.generateKeysDevice, against the oracle and an independent gcd."""
import numpy as np
import pytest

import ntru_oracle as o

pytestmark = pytest.mark.gpu

CFGS = ["tiny17", "default167", "hps509", "hps677", "hps821", "hrss701"]


@pytest.fixture(scope="module")
def nb():
    import ntru_circom_b200 as nb
    return nb


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


@pytest.fixture(scope="module")
def engines(nb, torch):
    cache = {}

    def get(cfg):
        if cfg not in cache:
            c = o.CONFIGS[cfg]
            eng = nb.Engine(c["N"], c["p"], c["q"], 0)
            eng.set_stream(torch.cuda.current_stream().cuda_stream)   # torch tensors and *_dev calls on one stream
            cache[cfg] = eng
        return cache[cfg]
    yield get
    for e in cache.values():
        e.close()


def _rows(torch, a, P, dtype):
    """host (B, N) -> device (B, P) with zero pad columns"""
    out = torch.zeros((a.shape[0], P), dtype=dtype, device="cuda")
    out[:, : a.shape[1]] = torch.from_numpy(np.ascontiguousarray(a)).to(device="cuda", dtype=dtype)
    return out


def _keygen_dev(torch, eng, f, g):
    """ntru_keygen_dev on host rows; outputs start as garbage so that every written column is checked."""
    B, P = f.shape[0], eng.pitch
    df, dg = _rows(torch, f, P, torch.int8), _rows(torch, g, P, torch.int8)
    fq = torch.full((B, P), -1, dtype=torch.int16, device="cuda")
    h = torch.full((B, P), -1, dtype=torch.int16, device="cuda")
    fp = torch.full((B, P), 0xAB, dtype=torch.uint8, device="cuda")
    valid = torch.full((B,), 0xAB, dtype=torch.uint8, device="cuda")
    eng.keygen_dev(B, df, dg, fq, fp, h, valid)
    eng.sync()
    return {"f": df, "g": dg, "fq": fq.cpu().numpy().view(np.uint16), "fp": fp.cpu().numpy(),
            "h": h.cpu().numpy().view(np.uint16), "valid": valid.cpu().numpy()}


# ---- independent truth: gcd(a, x^N - 1) over GF(2) and GF(3), polynomials as Python-int bit planes ----
def _gcd2_is_one(a, N):
    u = sum(1 << i for i, c in enumerate(a) if c % 2)
    v = (1 << N) | 1
    while u:
        while v.bit_length() >= u.bit_length():
            v ^= u << (v.bit_length() - u.bit_length())
        u, v = v, u
    return v == 1


def _add3(a, b):
    """a + b over GF(3), one-hot planes (coefficient = 1, coefficient = 2)"""
    (a1, a2), (b1, b2) = a, b
    a0, b0 = ~(a1 | a2), ~(b1 | b2)
    return (a1 & b0) | (b1 & a0) | (a2 & b2), (a2 & b0) | (b2 & a0) | (a1 & b1)


def _gcd3_is_one(a, N):
    def deg(x):
        return max(x[0].bit_length(), x[1].bit_length()) - 1

    def lead(x):
        return 1 if (x[0] >> deg(x)) & 1 else 2
    u = (sum(1 << i for i, c in enumerate(a) if c % 3 == 1), sum(1 << i for i, c in enumerate(a) if c % 3 == 2))
    v = (1 << N, 1)                                     # x^N - 1
    while deg(u) >= 0:
        while deg(v) >= deg(u):
            s = deg(v) - deg(u)
            t = (u[0] << s, u[1] << s)
            if lead(v) * lead(u) % 3 == 1:              # v -= c x^s u, c = lead(v) lead(u): add -c x^s u
                t = (t[1], t[0])
            v = _add3(v, t)
        u, v = v, u
    return deg(v) == 0


def _oracle_invertible(a, N, p):
    """the oracle's extended Euclid (index.js:425-459), its inverse checked by multiplying back"""
    try:
        inv = o.extended_euclidean_algorithm(a, [1] + [0] * (N - 1) + [-1], p)["inverse"]
    except (ValueError, ZeroDivisionError):
        return False
    c = np.convolve(np.array(a, dtype=np.int64), np.array(inv, dtype=np.int64))
    cyc = np.zeros(N, dtype=np.int64)
    np.add.at(cyc, np.arange(c.size) % N, c)
    return bool((np.mod(cyc, p) == np.eye(1, N, 0, dtype=np.int64)[0]).all())


def test_gcd_helpers_against_oracle_inverse():
    """the truth of the validity test agrees with the oracle's extended Euclid"""
    rng = np.random.default_rng(11)
    for N in (17, 31):
        for _ in range(60):
            a = rng.integers(-1, 2, size=N).tolist()
            for p, fn in ((2, _gcd2_is_one), (3, _gcd3_is_one)):
                assert fn(a, N) == _oracle_invertible(a, N, p), (N, p, a)


@pytest.mark.parametrize("cfg", CFGS)
def test_keygen_dev_vs_oracle(cfg, nb, torch, engines):
    """fq / fp / h of oracle keys bit for bit; the rejects have valid = 0 and all-zero outputs; pads are zero."""
    eng = engines(cfg)
    c = o.CONFIGS[cfg]
    N = c["N"]
    keys = [o.make_key(cfg, 500 + i) for i in range(6)]
    nk = len(keys)
    B = nk + 5
    f = np.zeros((B, N), dtype=np.int8)
    g = np.zeros((B, N), dtype=np.int8)
    for i, k in enumerate(keys):
        f[i], g[i] = k.f, k.g
    g[nk:] = keys[0].g
    f[nk] = 0                                           # zero polynomial
    f[nk + 1, :2] = 1                                   # f(1) even
    f[nk + 2, :3] = 1                                   # f(1) = 3
    f[nk + 3] = keys[1].f
    f[nk + 3, np.flatnonzero(f[nk + 3] == 0)[0]] = 2    # an entry outside {-1, 0, 1}
    f[nk + 4] = keys[2].f
    g[nk + 4, np.flatnonzero(g[nk + 4] == 0)[0]] = -2   # g outside {-1, 0, 1}
    out = _keygen_dev(torch, eng, f, g)
    assert out["valid"].tolist() == [1] * nk + [0] * 5
    for i, k in enumerate(keys):
        assert out["fq"][i, :N].tolist() == o.expand_array(k.fq, N, 0), (cfg, i, "fq")
        assert out["fp"][i, :N].tolist() == o.expand_array(k.fp, N, 0), (cfg, i, "fp")
        assert out["h"][i, :N].tolist() == o.expand_array(k.h, N, 0), (cfg, i, "h")
    for k in ("fq", "fp", "h"):
        assert not out[k][nk:].any(), (cfg, k)
        assert not out[k][:, N:].any(), (cfg, k, "pad")
    # the host-buffer form agrees (it runs the same device core)
    host = eng.keygen_batch(f, g)
    assert host["valid"].tolist() == [True] * nk + [False] * 5
    for k in ("fq", "fp", "h"):
        assert np.array_equal(host[k], out[k][:, :N]), (cfg, k)


def _check_inverses(torch, eng, f_rows, fq, fp, idx):
    """f fq = 1 (mod q, x^N - 1) and f fp = 1 (mod 3, x^N - 1) on the rows idx (numpy), through ntru_muldiv_dev"""
    N, P = eng.N, eng.pitch
    x = f_rows[torch.from_numpy(idx).to("cuda")].contiguous()
    B = x.shape[0]
    rq = torch.full((B, P), -1, dtype=torch.int16, device="cuda")
    rp = torch.full((B, P), 0xAB, dtype=torch.uint8, device="cuda")
    eng.muldiv_dev(B, x, torch.from_numpy(fq[idx].view(np.int16)).to("cuda").contiguous(), False, remainder=rq)
    eng.muldiv_dev(B, x, torch.from_numpy(fp[idx]).to("cuda").contiguous(), True, remainder=rp)
    eng.sync()
    one = np.zeros(N, dtype=np.int64)
    one[0] = 1
    assert (rq.cpu().numpy().view(np.uint16)[:, :N] == one).all()
    assert (rp.cpu().numpy()[:, :N] == one).all()


@pytest.mark.parametrize("cfg", CFGS)
def test_validity_verdicts_on_random_batches(cfg, nb, torch, engines):
    """Unweighted random ternary f.  For N in {509, 677, 701, 821} 2 and 3 have order N - 1 mod N, so Phi_N is
    irreducible mod 2 and mod 3 and f is invertible mod p iff f(1) != 0 (mod p) and f is not constant mod p.  At
    N = 17 and 167 Phi_N splits: every row is checked against a gcd over GF(2) and GF(3)."""
    eng = engines(cfg)
    c = o.CONFIGS[cfg]
    N = c["N"]
    B = {"tiny17": 4096, "default167": 1024}.get(cfg, 4096)
    rng = np.random.default_rng(N)
    f = rng.integers(-1, 2, size=(B, N)).astype(np.int8)
    g = rng.integers(-1, 2, size=(B, N)).astype(np.int8)
    f[0], f[1], f[2] = 1, -1, 0                          # constant rows: not invertible whatever f(1) is
    f[3] = 1
    f[3, 0] = -1                                         # all nonzero: constant mod 2
    out = _keygen_dev(torch, eng, f, g)
    if N in (17, 167):
        want = np.array([_gcd2_is_one(r.tolist(), N) and _gcd3_is_one(r.tolist(), N) for r in f])
    else:
        s = f.astype(np.int64).sum(axis=1)
        const2 = (f != 0).all(axis=1) | (f == 0).all(axis=1)
        const3 = (f == f[:, :1]).all(axis=1)
        want = (s % 2 == 1) & (s % 3 != 0) & ~const2 & ~const3
    assert np.array_equal(out["valid"].astype(bool), want), cfg
    assert 0.2 < want.mean() < 0.5                       # about (1/2) (2/3) of the rows
    for k in ("fq", "fp", "h"):
        assert not out[k][~want].any() and not out[k][:, N:].any(), (cfg, k)
    idx = np.flatnonzero(want)
    _check_inverses(torch, eng, out["f"], out["fq"], out["fp"], idx)


class _Draws:
    """rng stand-in for the oracle's generate_custom_array: hands out a fixed list of 32-bit draws."""

    def __init__(self, words):
        self.it = iter(words)

    def getrandbits(self, n):
        assert n == 32
        return next(self.it)


def _replay(nb, key, row, N, ones, neg_ones):
    """generateCustomArray(N, ones, neg_ones) of global row number `row` as the ORACLE computes it from the
    generator's draws (index.js:461-488)"""
    return o.generate_custom_array(N, ones, neg_ones, _Draws(nb.sampler_draws(key, row, N - 1)))


def _generate(torch, eng, B, df, dg, seed=None):
    P = eng.pitch
    out = {"f": torch.full((B, P), 7, dtype=torch.int8, device="cuda"),
           "g": torch.full((B, P), 7, dtype=torch.int8, device="cuda"),
           "fq": torch.full((B, P), -1, dtype=torch.int16, device="cuda"),
           "fp": torch.full((B, P), 0xAB, dtype=torch.uint8, device="cuda"),
           "h": torch.full((B, P), -1, dtype=torch.int16, device="cuda")}
    eng.generate_keys_dev(B, df, dg, out["f"], out["g"], out["fq"], out["fp"], out["h"], seed=seed)
    eng.sync()
    return out


@pytest.mark.parametrize("cfg,B,seed,R", [("tiny17", 300, 3, 1000), ("hps509", 64, 5, (1 << 40) + 3)])
def test_device_draws_replayed(cfg, B, seed, R, nb, torch, engines):
    """f and g are the oracle's generateCustomArray on the ChaCha20 draws of the documented row numbers, including
    the redraw rounds of non-invertible f (at N = 17, 1.3 % of weighted f are not invertible modulo 2); the keys
    are the oracle's keys of those f and g; the context's next row is R + (last round + 2) B."""
    eng = engines(cfg)
    c = o.CONFIGS[cfg]
    N, df, dg = c["N"], c["df"], c["dg"]
    key = nb.seed_key(seed)
    # host replay of the whole procedure
    want_f = [None] * B
    todo, last = list(range(B)), None
    for k in range(100):
        row0 = R if k == 0 else R + (k + 1) * B
        for b in todo:
            want_f[b] = _replay(nb, key, row0 + b, N, df, df - 1)
        todo = [b for b in todo if not (_gcd2_is_one(want_f[b], N) and _gcd3_is_one(want_f[b], N))]
        if not todo:
            last = k
            break
    if cfg == "tiny17":
        assert last >= 1                                 # the case exercises a redraw round
    want_g = [_replay(nb, key, R + B + b, N, dg, dg) for b in range(B)]
    eng.set_rng_key(key, R)
    out = _generate(torch, eng, B, df, dg)
    assert eng.rng_next_row == R + (last + 2) * B
    f = out["f"].cpu().numpy()
    g = out["g"].cpu().numpy()
    fq = out["fq"].cpu().numpy().view(np.uint16)
    fp = out["fp"].cpu().numpy()
    h = out["h"].cpu().numpy().view(np.uint16)
    assert np.array_equal(f[:, :N], np.array(want_f, dtype=np.int8)), cfg
    assert np.array_equal(g[:, :N], np.array(want_g, dtype=np.int8)), cfg
    for a in (f, g, fq, fp, h):
        assert not a[:, N:].any(), cfg
    for b in sorted({0, 1, B // 2, B - 1} | set(range(0, B, 37))):
        k = o.NTRU(dict(c))
        k.loadPrivateKeyF(want_f[b])
        k.g = want_g[b]
        k.generatePublicKeyH()
        assert fq[b, :N].tolist() == o.expand_array(k.fq, N, 0), (cfg, b, "fq")
        assert fp[b, :N].tolist() == o.expand_array(k.fp, N, 0), (cfg, b, "fp")
        assert h[b, :N].tolist() == o.expand_array(k.h, N, 0), (cfg, b, "h")
    _check_inverses(torch, eng, out["f"], fq, fp, np.arange(B))
    # the r sampler's numbering is unaffected: the next device-drawn r takes the next row
    r = torch.zeros((2, eng.pitch), dtype=torch.uint8, device="cuda")
    eng.sample_r_dev(2, c["dr"], eng.rng_next_row, r)
    eng.sync()
    want_r = [2 if x == -1 else x for x in _replay(nb, key, R + (last + 2) * B, N, c["dr"], c["dr"])]
    assert r[0, :N].cpu().tolist() == want_r


def test_generate_keys_device_end_to_end(nb, torch):
    """generateKeysDevice at N = 677: encrypt under h_rows, decrypt with f_rows / fp_rows, all on device rows; the
    decryptions are the oracle's for those keys and equal the messages (q = 2048 = 2 mod 3)."""
    c = o.CONFIGS["hps677"]
    N, q, p, B = c["N"], c["q"], c["p"], 3000
    kk = nb.NTRU(dict(c))
    eng = kk.engine()
    eng.set_stream(torch.cuda.current_stream().cuda_stream)
    eng.set_rng_key(nb.seed_key(21), 0)
    keys = kk.generateKeysDevice(B)
    P = eng.pitch
    assert all(keys[k].shape == (B, P) for k in ("f", "g", "fq", "fp", "h"))
    rng = np.random.default_rng(4)
    m = rng.integers(0, 2, size=(B, N)).astype(np.uint8)
    r = o.sample_ternary_rows(B, N, c["dr"], c["dr"], rng).astype(np.uint8)
    m_d, r_d = _rows(torch, m, P, torch.uint8), _rows(torch, r, P, torch.uint8)
    e = torch.empty((B, P), dtype=torch.int16, device="cuda")
    dec = torch.empty((B, P), dtype=torch.uint8, device="cuda")
    eng.encrypt_dev(B, r_d, m_d, value=e, h_rows=keys["h"])
    eng.decrypt_dev(B, e, value=dec, f_rows=keys["f"], fp_rows=keys["fp"])
    eng.sync()
    assert np.array_equal(dec[:, :N].cpu().numpy(), m)
    idx = np.arange(0, B, 7)
    f = keys["f"][:, :N].cpu().numpy().astype(np.int64)[idx]
    fp = keys["fp"][:, :N].cpu().numpy().astype(np.int64)[idx]
    h = keys["h"][:, :N].cpu().numpy().view(np.uint16).astype(np.int64)[idx]
    want_e = o.encrypt_batch(h, r[idx], m[idx], q)["value"]
    got_e = e[:, :N].cpu().numpy().view(np.uint16)[idx]
    assert np.array_equal(got_e, want_e)
    want = o.decrypt_batch(f, fp, got_e.astype(np.int64), q, p)["value"]
    assert np.array_equal(dec[:, :N].cpu().numpy()[idx], want)
    eng.close()


def test_keygen_timing_kind_and_argument_errors(nb, torch, engines):
    eng = engines("default167")
    N, P = 167, eng.pitch
    c = o.CONFIGS["default167"]
    z8 = torch.zeros((4, P), dtype=torch.int8, device="cuda")
    z16 = torch.zeros((4, P), dtype=torch.int16, device="cuda")
    zu = torch.zeros((4, P), dtype=torch.uint8, device="cuda")
    # the inversion has its own timing kind, separate from the lifting's products
    eng.set_timing(True)
    eng.timing_reset()
    _generate(torch, eng, 64, c["df"], c["dg"], seed=1)
    t = eng.timing_read()
    eng.set_timing(False)
    assert t["inverse"][1] >= 1 and t["muldiv"][1] >= 1
    # weights out of range (index.js:462-464)
    for df, dg in ((0, 20), ((N + 1) // 2 + 1, 20), (61, N // 2 + 1), (61, -1)):
        with pytest.raises(nb.NtruError, match="cannot exceed"):
            eng.generate_keys_dev(4, df, dg, z8, z8, z16, zu, z16)
    # NULL pointers
    with pytest.raises(nb.NtruError, match="required"):
        eng.generate_keys_dev(4, 61, 20, None, z8, z16, zu, z16)
    with pytest.raises(nb.NtruError, match="required"):
        eng.keygen_dev(4, z8, z8, z16, zu, None, zu)
    # B = 0 is a no-op and uses no row
    row = eng.rng_next_row
    eng.generate_keys_dev(0, 61, 20, None, None, None, None, None)
    eng.keygen_dev(0, None, None, None, None, None, None)
    assert eng.rng_next_row == row
