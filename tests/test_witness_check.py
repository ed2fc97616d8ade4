"""Witness checks on the GPU: ntru_check_encrypt / _decrypt / _inverse (VerifyEncrypt, VerifyDecrypt, VerifyInverse,
circuits/ntru.circom:155-256) against the oracle's restatement of the constraint systems.

`expected_verdict` is the reference every GPU verdict is compared with: the oracle's verify_* decides SATISFIED; CANONICAL
adds every quotient / remainder entry below its modulus and remainder[N] == 0; DOMAIN replaces both when an entry of the
small operand, reduced modulo the product's modulus M, is outside {M-1, 0, 1, 2}.  The CPU tests pin that helper on
hand-made witnesses; the GPU tests compare every row of mixed batches with it.
"""
import ctypes

import numpy as np
import pytest

import ntru_oracle as o

SAT, CANON, DOMAIN = 1, 2, 4
OK = SAT | CANON

# per kind: the small operand, the input arrays (width N), the divisions (quotient, remainder: width N + 1)
SPEC = {
    "encrypt": ("r", ("r", "m", "h"), (("quotientE", "remainderE"),)),
    "decrypt": ("f", ("f", "fp", "e"), (("quotient1", "remainder1"), ("quotient2", "remainder2"))),
    "inverse": ("f", ("f", "fq"), (("quotientI", "remainderI"),)),
}
VERIFY = {"encrypt": o.verify_encrypt, "decrypt": o.verify_decrypt, "inverse": o.verify_inverse}


def div_moduli(kind, params):
    return [params[0], params[2]] if kind == "decrypt" else [params[0]]


def expected_verdict(kind, w, params):
    """Verdict byte of one witness row (arrays may be longer than their width: the rest is ignored)."""
    small, inputs, divs = SPEC[kind]
    N, M = params[-1], params[0]
    x = np.asarray(w[small], dtype=np.int64)[:N] % M
    if not np.all((x == M - 1) | (x <= 2)):
        return DOMAIN
    row = {k: [int(v) for v in np.asarray(w[k])[:N]] for k in inputs}
    for qn, rn in divs:
        row[qn] = [int(v) for v in np.asarray(w[qn])[:N + 1]]
        row[rn] = [int(v) for v in np.asarray(w[rn])[:N + 1]]
    if not VERIFY[kind](row, params):
        return 0
    canon = all(max(row[qn]) < mod and max(row[rn]) < mod and row[rn][N] == 0
                for (qn, rn), mod in zip(divs, div_moduli(kind, params)))
    return SAT | (CANON if canon else 0)


def nq(q, N):
    return int(np.ceil(np.log2(q * q * N)))


def enc_params(N, q):
    return [q, nq(q, N), N]


def dec_params(N, q):
    return [q, nq(q, N), 3, nq(3, N), N]


# ---- oracle-made witnesses (no GPU) ---------------------------------------------------------------------------------

def _oracle_witnesses(N=17, q=32, seed=3):
    rng = np.random.default_rng(seed)
    h = rng.integers(0, q, N)
    f = rng.integers(-1, 2, N)
    fp = rng.integers(0, 3, N)
    r = rng.integers(0, 3, (1, N))
    m = rng.integers(0, 2, (1, N))
    enc = o.encrypt_batch(h, r, m, q)
    dec = o.decrypt_batch(f, fp, enc["value"], q)
    ew = {"r": r[0], "m": m[0], "h": h, "quotientE": enc["quotientE"][0], "remainderE": enc["remainderE"][0]}
    dw = {"f": np.where(f < 0, q - 1, f), "fp": fp, "e": enc["value"][0], "quotient1": dec["quotient1"][0],
          "remainder1": dec["remainder1"][0], "quotient2": dec["quotient2"][0], "remainder2": dec["remainder2"][0]}
    return ew, dw


def _copy(w):
    return {k: np.array(v, dtype=np.int64) for k, v in w.items()}


def test_expected_verdict_on_hand_made_witnesses():
    N, q = 17, 32
    ew, dw = _oracle_witnesses(N, q)
    ep, dp = enc_params(N, q), dec_params(N, q)
    assert expected_verdict("encrypt", ew, ep) == OK
    assert expected_verdict("decrypt", dw, dp) == OK
    # the t-shift family: every constraint still holds, the witness is not the one dividePolynomials returns
    for t in (1, 5, q - 1):
        w = _copy(ew)
        w["quotientE"][0] = (w["quotientE"][0] + t) % q
        w["remainderE"][N] = (w["remainderE"][N] + t) % q
        w["remainderE"][0] = (w["remainderE"][0] - t) % q
        assert expected_verdict("encrypt", w, ep) == SAT, t
        assert o.verify_encrypt({k: list(v) for k, v in w.items()}, ep)
    # an entry raised by q: satisfied, not canonical
    for name, k in (("quotientE", 3), ("remainderE", 0), ("quotientE", N)):
        w = _copy(ew)
        w[name][k] += q
        assert expected_verdict("encrypt", w, ep) == SAT, (name, k)
    # one coefficient tampered: not satisfied
    for name, k in (("quotientE", 1), ("remainderE", N - 1), ("quotientE", N - 1), ("quotientE", N), ("remainderE", N)):
        w = _copy(ew)
        w[name][k] = (w[name][k] + 1) % q
        assert expected_verdict("encrypt", w, ep) == 0, (name, k)
    # remainder2[0] + 1 (test/circuits.test.js:296-301)
    w = _copy(dw)
    w["remainder2"][0] = (w["remainder2"][0] + 1) % 3
    assert expected_verdict("decrypt", w, dp) == 0
    # remainder2 raised by 3: satisfied only
    w = _copy(dw)
    w["remainder2"][2] += 3
    assert expected_verdict("decrypt", w, dp) == SAT
    # small operands outside {M-1, 0, 1, 2}: not evaluated
    w = _copy(ew)
    w["r"][4] = 3
    assert expected_verdict("encrypt", w, ep) == DOMAIN
    w = _copy(dw)
    w["f"][0] = q - 2
    assert expected_verdict("decrypt", w, dp) == DOMAIN
    # inputs at any value are taken modulo q (h, e, m) or 3 (fp): the same witness stays satisfied and canonical
    w = _copy(ew)
    w["h"][2] += q
    w["m"][5] += 2 * q
    assert expected_verdict("encrypt", w, ep) == OK
    w = _copy(dw)
    w["fp"][1] += 3
    assert expected_verdict("decrypt", w, dp) == OK
    # columns beyond the witness width are ignored
    w = {k: np.concatenate([v, [7, 9]]) for k, v in _copy(ew).items()}
    assert expected_verdict("encrypt", w, ep) == OK


def test_expected_verdict_on_the_key_witness():
    k = o.make_key("tiny17", 5)
    wit = k.verifyKeysInputs()
    for case in ("fq", "fp", "h"):
        ins, params = wit[case]["inputs"], wit[case]["params"]
        assert expected_verdict("inverse", ins, params) == OK, case
        bad = _copy(ins)
        bad["remainderI"][0] = (bad["remainderI"][0] + 1) % params[0]
        assert expected_verdict("inverse", bad, params) == 0, case
        shifted = _copy(ins)
        shifted["quotientI"][0] = (shifted["quotientI"][0] + 1) % params[0]
        shifted["remainderI"][k.N] = (shifted["remainderI"][k.N] + 1) % params[0]
        shifted["remainderI"][0] = (shifted["remainderI"][0] - 1) % params[0]
        assert expected_verdict("inverse", shifted, params) == SAT, case


def test_check_entry_points_without_a_device():
    """Without a context every entry point refuses with NTRU_E_PARAM; without a device no context can be made (the
    Python calls raise NTRU_E_CUDA), so nothing falls back to a CPU path."""
    from ntru_circom_b200 import _lib
    import ntru_circom_b200 as nb
    lib = _lib.load()
    buf = (ctypes.c_uint8 * 64)()
    p = ctypes.addressof(buf)
    assert lib.ntru_check_encrypt_dev(None, 1, p, 0, p, p, p, p, p) == _lib.NTRU_E_PARAM
    assert lib.ntru_check_decrypt_dev(None, 1, p, p, 0, p, p, p, p, p, p) == _lib.NTRU_E_PARAM
    assert lib.ntru_check_inverse_dev(None, 1, 0, p, p, p, p, p) == _lib.NTRU_E_PARAM
    assert lib.ntru_check_encrypt_batch(None, 1, p, 1, p, p, p, p, p) == _lib.NTRU_E_PARAM
    assert lib.ntru_check_decrypt_batch(None, 1, p, p, 1, p, p, p, p, p, p) == _lib.NTRU_E_PARAM
    assert lib.ntru_check_inverse_batch(None, 1, 1, p, p, p, p, p) == _lib.NTRU_E_PARAM
    assert nb.NTRU_CHECK_SATISFIED == SAT and nb.NTRU_CHECK_CANONICAL == CANON and nb.NTRU_CHECK_DOMAIN == DOMAIN
    assert _lib.KERNEL_KINDS[12] == "check"
    import torch
    if not torch.cuda.is_available():
        with pytest.raises(nb.NtruError) as ei:
            nb.Engine(17, 3, 32, 0)
        assert ei.value.code == _lib.NTRU_E_CUDA
        ew, _ = _oracle_witnesses()
        with pytest.raises(nb.NtruError):
            nb.NTRU({"N": 17, "q": 32}).verifyEncryptBatch({k: np.asarray(v)[None] for k, v in ew.items()}, enc_params(17, 32))


# ---- GPU ------------------------------------------------------------------------------------------------------------

SHAPES = [(8, 32), (17, 32), (167, 128), (509, 2048), (677, 2048), (701, 8192), (821, 4096), (832, 8192)]

DTYPES = {
    "encrypt": {"r": np.uint8, "m": np.uint16, "h": np.uint16, "quotientE": np.uint16, "remainderE": np.uint16},
    "decrypt": {"f": np.uint16, "fp": np.uint8, "e": np.uint16, "quotient1": np.uint16, "remainder1": np.uint16,
                "quotient2": np.uint8, "remainder2": np.uint8},
    "inverse_q": {"f": np.uint16, "fq": np.uint16, "quotientI": np.uint16, "remainderI": np.uint16},
    "inverse_p": {"f": np.uint16, "fq": np.uint8, "quotientI": np.uint8, "remainderI": np.uint8},
}


@pytest.fixture(scope="module")
def nb():
    import ntru_circom_b200 as nb
    return nb


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


def _engine(nb, N, q):
    eng = nb.Engine(N, 3, q, 0)
    rng = np.random.default_rng(N + q)
    h, f, fp = rng.integers(0, q, N), rng.integers(-1, 2, N), rng.integers(0, 3, N)
    eng.set_public_key(h.astype(np.uint16))
    eng.set_private_key(f.astype(np.int8), fp.astype(np.uint8))
    return eng, rng, {"h": h, "f": f, "fp": fp}


def _honest_encrypt(eng, rng, key, B, shared):
    N, q = eng.N, eng.q
    r = rng.integers(0, 3, (B, N)).astype(np.uint8)
    m = rng.integers(0, min(q, 256), (B, N)).astype(np.uint8)       # byte messages: the per-row-key encrypt takes no wide m
    h = key["h"].astype(np.uint16) if shared else rng.integers(0, q, (B, N)).astype(np.uint16)
    out = eng.encrypt_batch(r, m, h=None if shared else h)
    m = m.astype(np.uint16)
    return {"r": r, "m": m, "h": h, "quotientE": out["quotientE"], "remainderE": out["remainderE"]}, out["value"]


def _honest_decrypt(eng, rng, key, e, shared):
    B, N, q = e.shape[0], eng.N, eng.q
    if shared:
        f, fp = key["f"], key["fp"]
        out = eng.decrypt_batch(e)
    else:
        f, fp = rng.integers(-1, 2, (B, N)), rng.integers(0, 3, (B, N))
        out = eng.decrypt_batch(e, f=f.astype(np.int8), fp=fp.astype(np.uint8))
    return {"f": np.where(f < 0, q - 1, f).astype(np.uint16), "fp": fp.astype(np.uint8), "e": e.astype(np.uint16),
            **{k: out[k] for k in ("quotient1", "remainder1", "quotient2", "remainder2")}}


def _honest_inverse(eng, rng, B):
    N, q = eng.N, eng.q
    f, g = rng.integers(-1, 2, (B, N)), rng.integers(-1, 2, (B, N))
    fq, fp = rng.integers(0, q, (B, N)), rng.integers(0, 3, (B, N))
    o_ = eng.verify_keys_batch(f.astype(np.int8), fq.astype(np.uint16), fp.astype(np.uint8), g.astype(np.int8))
    return {
        "fq": ({"f": np.where(f < 0, q - 1, f), "fq": fq, "quotientI": o_["quotient_fq"], "remainderI": o_["remainder_fq"]}, False),
        "fp": ({"f": np.where(f < 0, 2, f), "fq": fp, "quotientI": o_["quotient_fp"], "remainderI": o_["remainder_fp"]}, True),
        "h": ({"f": np.where(g < 0, q - 1, g), "fq": 3 * fq, "quotientI": o_["quotient_h"], "remainderI": o_["remainder_h"]}, False),
    }


def _check(eng, kind, w, mod_p=False):
    if kind == "encrypt":
        return eng.check_encrypt(w["h"], w["r"], w["m"], w["quotientE"], w["remainderE"])
    if kind == "decrypt":
        return eng.check_decrypt(w["f"], w["fp"], w["e"], w["quotient1"], w["remainder1"], w["quotient2"], w["remainder2"])
    return eng.check_inverse(w["f"], w["fq"], w["quotientI"], w["remainderI"], mod_p=mod_p)


@pytest.mark.gpu
@pytest.mark.parametrize("N,q", SHAPES, ids=[f"N{n}q{q}" for n, q in SHAPES])
def test_honest_witnesses_are_canonical(nb, N, q):
    eng, rng, key = _engine(nb, N, q)
    for shared, B in ((True, 5000), (False, 300)):
        ew, value = _honest_encrypt(eng, rng, key, B, shared)
        v = _check(eng, "encrypt", ew)
        assert v.shape == (B,) and np.all(v == OK), (shared, np.flatnonzero(v != OK)[:8])
        dw = _honest_decrypt(eng, rng, key, value, shared)
        v = _check(eng, "decrypt", dw)
        assert np.all(v == OK), (shared, np.flatnonzero(v != OK)[:8])
    for case, (w, mod_p) in _honest_inverse(eng, rng, 200).items():
        v = _check(eng, "inverse", w, mod_p)
        assert np.all(v == OK), (case, np.flatnonzero(v != OK)[:8])
    # the oracle agrees on a sample
    assert expected_verdict("encrypt", {k: a[0] if a.ndim == 2 else a for k, a in ew.items()}, enc_params(N, q)) == OK
    eng.close()


def _modulus(kind, name, q):
    dt = DTYPES[kind][name]
    if kind == "encrypt" and name == "r":
        return None
    if dt == np.uint16:
        return q
    return 3


def _crafted(kind, w0, N, q, M, rng):
    """(label, row dict, dirty pad) for every crafted case, derived from the honest row w0."""
    dts = DTYPES[kind]
    small = "r" if kind == "encrypt" else "f"
    out = []

    def add(label, fn, pad=False):
        w = {k: np.array(v, dtype=np.int64) for k, v in w0.items()}
        fn(w)
        for k, v in w.items():
            assert v.min() >= 0 and v.max() <= np.iinfo(dts[k]).max, (label, k)
        out.append((label, w, pad))

    for name in w0:
        width = len(w0[name])
        top = np.iinfo(dts[name]).max
        for k in (0, 1, N - 2, N - 1, N):
            if k < width:
                add(f"+1 {name}[{k}]", lambda w, n=name, k=k, t=top: w[n].__setitem__(k, (w[n][k] + 1) % (t + 1)))
        mod = _modulus(kind, name, q)
        if mod:
            for k in (0, N // 2, width - 1):
                add(f"+mod {name}[{k}]", lambda w, n=name, k=k, m=mod, t=top: w[n].__setitem__(k, w[n][k] + m if w[n][k] + m <= t else w[n][k] - m))
    divs = SPEC["encrypt" if kind == "encrypt" else ("decrypt" if kind == "decrypt" else "inverse")][2]
    mods = [M] if kind != "decrypt" else [q, 3]
    for (qn, rn), mod in zip(divs, mods):
        top = np.iinfo(dts[qn]).max
        for t in sorted({1, 5 % mod or 1, mod - 1}):
            def shift(w, t=t, qn=qn, rn=rn, mod=mod):
                w[qn][0] = (w[qn][0] + t) % mod
                w[rn][N] = (w[rn][N] + t) % mod
                w[rn][0] = (w[rn][0] - t) % mod
            add(f"t-shift {t} {qn}", shift)

            def shift_raw(w, t=t, qn=qn, rn=rn, mod=mod, top=top):
                w[qn][0] = w[qn][0] + t if w[qn][0] + t <= top else w[qn][0] + t - mod
                w[rn][N] = w[rn][N] + t
                w[rn][0] = (w[rn][0] - t) % mod
            add(f"raw t-shift {t} {qn}", shift_raw)
        add(f"{qn}[N-1] = M", lambda w, qn=qn, mod=mod: w[qn].__setitem__(N - 1, mod))
        add(f"{qn}[N] = M", lambda w, qn=qn, mod=mod: w[qn].__setitem__(N, mod))
        add(f"{qn}[N] = 1", lambda w, qn=qn: w[qn].__setitem__(N, 1))
    stop = np.iinfo(dts[small]).max
    for val in sorted(v for v in {3, M - 2, stop, 2 * M - 1} if v <= stop):
        for k in (0, N - 1):
            add(f"domain {small}[{k}]={val}", lambda w, k=k, v=val: w[small].__setitem__(k, v))
    for name in w0:
        if name != small and len(w0[name]) == N:
            add(f"top {name}", lambda w, n=name: w[n].__setitem__(slice(0, N, 3), np.iinfo(dts[n]).max))
    if kind == "decrypt":       # remainder1 entries >= q: same residue, another lift
        for k in (0, 2, N - 1):
            add(f"remainder1[{k}] + q", lambda w, k=k: w["remainder1"].__setitem__(k, w["remainder1"][k] + q))
    add("dirty pad", lambda w: None, pad=True)
    for i in range(3):
        def rand(w, i=i):
            for k in w:
                hi = 3 if (k == small and i == 0) else (np.iinfo(dts[k]).max + 1 if i < 2 else _modulus(kind, k, q) or 3)
                w[k][:] = rng.integers(0, hi, w[k].shape)
        add(f"random {i}", rand, pad=i == 1)
    return out


def _to_dev(torch, rows, dt, P, width, pad):
    """(B, width) numpy rows -> (B, P) device tensor; pad[b]: columns >= width hold 0xFF."""
    a = np.zeros((len(rows), P), dtype=dt)
    a[:, :width] = rows
    a[pad, width:] = np.iinfo(dt).max
    t = torch.from_numpy(a.view(np.int16) if dt == np.uint16 else a)
    return t.cuda()


def _run_dev(torch, eng, kind, rows, pads, mod_p=False):
    """every row its own key (key_stride = pitch); returns the verdicts"""
    P, N, B = eng.pitch, eng.N, len(rows)
    dts = DTYPES["inverse_p" if mod_p else "inverse_q"] if kind == "inverse" else DTYPES[kind]
    dev = {k: _to_dev(torch, np.stack([r[k] for r in rows]).astype(dt), dt, P, len(rows[0][k]), pads) for k, dt in dts.items()}
    verdict = torch.full((B,), 0xEE, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    if kind == "encrypt":
        eng.check_encrypt_dev(B, dev["h"], P, dev["r"], dev["m"], dev["quotientE"], dev["remainderE"], verdict)
    elif kind == "decrypt":
        eng.check_decrypt_dev(B, dev["f"], dev["fp"], P, dev["e"], dev["quotient1"], dev["remainder1"], dev["quotient2"],
                              dev["remainder2"], verdict)
    else:
        eng.check_inverse_dev(B, mod_p, dev["f"], dev["fq"], dev["quotientI"], dev["remainderI"], verdict)
    eng.sync()
    return verdict.cpu().numpy()


CRAFT_SHAPES = [(17, 32), (509, 2048), (821, 4096)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["encrypt", "decrypt", "inverse_q", "inverse_p"])
@pytest.mark.parametrize("N,q", CRAFT_SHAPES, ids=[f"N{n}q{q}" for n, q in CRAFT_SHAPES])
def test_every_row_against_the_oracle(nb, torch, kind, N, q):
    """Honest rows and crafted rows in one batch; each crafted row sits in the first warp, a middle one and the last."""
    eng, rng, key = _engine(nb, N, q)
    F = 40
    if kind == "encrypt":
        w, value = _honest_encrypt(eng, rng, key, F + 1, False)
        params, kk, M, mod_p = enc_params(N, q), "encrypt", q, False
    elif kind == "decrypt":
        ew, value = _honest_encrypt(eng, rng, key, F + 1, False)
        w = _honest_decrypt(eng, rng, key, value, False)
        params, kk, M, mod_p = dec_params(N, q), "decrypt", q, False
    else:
        mod_p = kind == "inverse_p"
        w = _honest_inverse(eng, rng, F + 1)["fp" if mod_p else "fq"][0]
        M = 3 if mod_p else q
        params, kk = ([3, nq(3, N), N] if mod_p else [q, nq(q, N), N]), "inverse"
    rows = [{k: np.asarray(v[b]).astype(np.int64) for k, v in w.items()} for b in range(F + 1)]
    crafted = _crafted(kind, rows[0], N, q, M, rng)
    labels = [c[0] for c in crafted]
    C = [c[1] for c in crafted]
    Cp = [c[2] for c in crafted]
    fill = rows[1:]
    batch = C + fill + C + fill + C
    pads = np.array(Cp + [False] * F + Cp + [False] * F + Cp)
    got = _run_dev(torch, eng, kk, batch, pads, mod_p)
    want_c = [expected_verdict(kk, c, params) for c in C]
    want = np.array(want_c + [OK] * F + want_c + [OK] * F + want_c)
    assert expected_verdict(kk, fill[0], params) == OK
    bad = np.flatnonzero(got != want)
    nC = len(C)
    assert bad.size == 0, [(int(i), labels[i % (nC + F)] if i % (nC + F) < nC else "honest", int(got[i]), int(want[i]))
                           for i in bad[:12]]
    # every kind of verdict occurs
    assert {0, SAT, OK, DOMAIN} <= set(want_c) or kind == "inverse_p", set(want_c)
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("N,q", [(509, 2048), (821, 4096)], ids=["N509q2048", "N821q4096"])
def test_full_size_tcgen05_batch(nb, torch, N, q):
    """2^20 same-key rows encrypted and decrypted on the tcgen05 schedule, every row checked on the device; one flipped
    coefficient in 16 chosen rows fails exactly those rows."""
    eng, rng, key = _engine(nb, N, q)
    P, B = eng.pitch, 1 << 20
    gen = torch.Generator(device="cuda").manual_seed(N)
    r = torch.zeros((B, P), dtype=torch.uint8, device="cuda")
    r[:, :N] = torch.randint(0, 3, (B, N), generator=gen, device="cuda", dtype=torch.uint8)
    m = torch.zeros((B, P), dtype=torch.uint8, device="cuda")
    m[:, :N] = torch.randint(0, 2, (B, N), generator=gen, device="cuda", dtype=torch.uint8)
    m16 = m.to(torch.int16)
    enc = {k: torch.empty((B, P), dtype=torch.int16, device="cuda") for k in ("value", "quotientE", "remainderE")}
    dec = {"value": torch.empty((B, P), dtype=torch.uint8, device="cuda"),
           "quotient1": torch.empty((B, P), dtype=torch.int16, device="cuda"),
           "remainder1": torch.empty((B, P), dtype=torch.int16, device="cuda"),
           "quotient2": torch.empty((B, P), dtype=torch.uint8, device="cuda"),
           "remainder2": torch.empty((B, P), dtype=torch.uint8, device="cuda")}
    torch.cuda.synchronize()
    eng.encrypt_dev(B, r, m, **enc)
    assert eng.last_path == nb.PATH_TENSOR
    eng.decrypt_dev(B, enc["value"], **dec)
    assert eng.last_path == nb.PATH_TENSOR
    h = torch.zeros(P, dtype=torch.int16, device="cuda")
    h[:N] = torch.from_numpy(key["h"].astype(np.int16)).cuda()
    f = torch.zeros(P, dtype=torch.int16, device="cuda")
    f[:N] = torch.from_numpy(np.where(key["f"] < 0, q - 1, key["f"]).astype(np.uint16).view(np.int16)).cuda()
    fp = torch.zeros(P, dtype=torch.uint8, device="cuda")
    fp[:N] = torch.from_numpy(key["fp"].astype(np.uint8)).cuda()
    ve = torch.empty(B, dtype=torch.uint8, device="cuda")
    vd = torch.empty(B, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def run():
        eng.check_encrypt_dev(B, h, 0, r, m16, enc["quotientE"], enc["remainderE"], ve)
        eng.check_decrypt_dev(B, f, fp, 0, enc["value"], dec["quotient1"], dec["remainder1"], dec["quotient2"],
                              dec["remainder2"], vd)
        eng.sync()
        return ve.cpu().numpy(), vd.cpu().numpy()

    a, b = run()
    assert np.all(a == OK) and np.all(b == OK), (np.flatnonzero(a != OK)[:8], np.flatnonzero(b != OK)[:8])
    rows = np.unique(np.concatenate([[0, 1, B // 2, B - 1], rng.choice(B, 12, replace=False)]))[:16]
    cols = rng.integers(0, N + 1, len(rows))
    for i, (row, col) in enumerate(zip(rows.tolist(), cols.tolist())):
        enc["quotientE" if i % 2 else "remainderE"][row, col] += 1
        dec["remainder2" if i % 2 else "quotient1"][row, col] += 1
    torch.cuda.synchronize()
    a, b = run()
    assert np.array_equal(np.flatnonzero(a != OK), rows) and np.all(a[rows] == 0)
    assert np.array_equal(np.flatnonzero(b != OK), rows) and np.all(b[rows] == 0)
    eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("shared", [True, False], ids=["shared", "per_row"])
def test_host_form_equals_device_form(nb, torch, shared):
    N, q = 509, 2048
    eng, rng, key = _engine(nb, N, q)
    eng.set_option(nb._lib.NTRU_OPT_CHUNK_ROWS, 128)
    B = 1000
    ew, value = _honest_encrypt(eng, rng, key, B, shared)
    dw = _honest_decrypt(eng, rng, key, value, shared)
    # mixed verdicts: tamper every seventh row, push r out of the domain in every thirteenth
    ew["quotientE"][::7, 3] ^= 1
    ew["r"][::13, 5] = 7
    dw["remainder2"][::5, 0] = (dw["remainder2"][::5, 0] + 1) % 3
    dw["quotient1"][::11, 2] += q
    hv = _check(eng, "encrypt", ew)
    hd = _check(eng, "decrypt", dw)
    assert len(set(hv.tolist())) >= 3 and len(set(hd.tolist())) >= 3
    pads = np.zeros(B, dtype=bool)
    key_rows = lambda a: np.broadcast_to(a, (B, a.shape[-1])) if a.ndim == 1 else a   # noqa: E731
    erows = [{k: key_rows(np.asarray(v))[b] for k, v in ew.items()} for b in range(B)]
    drows = [{k: key_rows(np.asarray(v))[b] for k, v in dw.items()} for b in range(B)]
    assert np.array_equal(_run_dev(torch, eng, "encrypt", erows, pads), hv)
    assert np.array_equal(_run_dev(torch, eng, "decrypt", drows, pads), hd)
    # guard bytes around the host verdicts, and B = 0
    lib, G = eng.lib, 32
    out = np.full(B + 2 * G, 0xA5, dtype=np.uint8)
    h = np.ascontiguousarray(ew["h"], dtype=np.uint16)
    args = [np.ascontiguousarray(ew[k], dtype=dt) for k, dt in (("r", np.uint8), ("m", np.uint16), ("quotientE", np.uint16),
                                                                ("remainderE", np.uint16))]
    rc = lib.ntru_check_encrypt_batch(eng._h, B, h.ctypes.data, int(shared), *[a.ctypes.data for a in args], out.ctypes.data + G)
    assert rc == 0
    assert np.array_equal(out[G:G + B], hv) and np.all(out[:G] == 0xA5) and np.all(out[G + B:] == 0xA5)
    out[:] = 0xA5
    assert lib.ntru_check_encrypt_batch(eng._h, 0, h.ctypes.data, int(shared), *[a.ctypes.data for a in args], out.ctypes.data + G) == 0
    assert np.all(out == 0xA5)
    assert eng.check_encrypt(ew["h"] if shared else ew["h"][:0], ew["r"][:0], ew["m"][:0], ew["quotientE"][:0], ew["remainderE"][:0]).shape == (0,)
    # device form: guard bytes around the verdicts
    dev_out = torch.full((B + 2 * G,), 0xA5, dtype=torch.uint8, device="cuda")
    P = eng.pitch
    dts = DTYPES["encrypt"]
    dev = {k: _to_dev(torch, np.stack([r_[k] for r_ in erows]).astype(dt), dt, P, len(erows[0][k]), pads) for k, dt in dts.items()}
    torch.cuda.synchronize()
    eng.check_encrypt_dev(B, dev["h"], P, dev["r"], dev["m"], dev["quotientE"], dev["remainderE"], dev_out[G:].data_ptr())
    eng.sync()
    got = dev_out.cpu().numpy()
    assert np.array_equal(got[G:G + B], hv) and np.all(got[:G] == 0xA5) and np.all(got[G + B:] == 0xA5)
    eng.close()


@pytest.mark.gpu
def test_argument_errors(nb, torch):
    from ntru_circom_b200 import _lib
    N, q = 167, 128
    eng, _, _ = _engine(nb, N, q)
    P = eng.pitch
    t = torch.zeros((4, P), dtype=torch.int16, device="cuda")
    v = torch.zeros(4, dtype=torch.uint8, device="cuda")
    p, vp = t.data_ptr(), v.data_ptr()
    lib, h = eng.lib, eng._h
    assert lib.ntru_check_encrypt_dev(h, 4, p, 0, p, p, p, p, vp) == 0
    eng.sync()
    assert lib.ntru_check_encrypt_dev(h, 4, p, 1, p, p, p, p, vp) == _lib.NTRU_E_PARAM
    assert lib.ntru_check_encrypt_dev(h, 4, p, P + 16, p, p, p, p, vp) == _lib.NTRU_E_PARAM
    assert lib.ntru_check_encrypt_dev(h, 4, p, P, p, None, p, p, vp) == _lib.NTRU_E_PARAM
    assert lib.ntru_check_decrypt_dev(h, 4, p, p, 3, p, p, p, p, p, vp) == _lib.NTRU_E_PARAM
    assert lib.ntru_check_decrypt_dev(h, 4, p, p, 0, p, p, p, p, None, vp) == _lib.NTRU_E_PARAM
    assert lib.ntru_check_inverse_dev(h, 4, 0, p, p, p, p, None) == _lib.NTRU_E_PARAM
    assert lib.ntru_check_inverse_batch(h, 4, 1, None, p, p, p, vp) == _lib.NTRU_E_PARAM
    eng.close()
    big = nb.Engine(1024, 3, 2048, 0)
    with pytest.raises(nb.NtruError) as ei:
        big.check_inverse(np.zeros((1, 1024)), np.zeros((1, 1024)), np.zeros((1, 1025)), np.zeros((1, 1025)))
    assert ei.value.code == _lib.NTRU_E_UNSUPPORTED
    big.close()


@pytest.mark.gpu
def test_check_sees_the_outputs_of_a_queued_encrypt(nb, torch):
    """encrypt_dev and check_encrypt_dev queued back to back on the context's stream, no synchronisation between them."""
    N, q = 821, 4096
    eng, rng, key = _engine(nb, N, q)
    P, B = eng.pitch, 1 << 16
    gen = torch.Generator(device="cuda").manual_seed(5)
    r = torch.zeros((B, P), dtype=torch.uint8, device="cuda")
    r[:, :N] = torch.randint(0, 3, (B, N), generator=gen, device="cuda", dtype=torch.uint8)
    m = torch.zeros((B, P), dtype=torch.uint8, device="cuda")
    h_rows = torch.zeros((B, P), dtype=torch.int16, device="cuda")
    h_rows[:, :N] = torch.randint(0, q, (B, N), generator=gen, device="cuda", dtype=torch.int16)
    m16 = m.to(torch.int16)
    quo = torch.full((B, P), -1, dtype=torch.int16, device="cuda")
    rem = torch.full((B, P), -1, dtype=torch.int16, device="cuda")
    v = torch.zeros(B, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    eng.encrypt_dev(B, r, m, None, quo, rem, h_rows=h_rows)
    eng.check_encrypt_dev(B, h_rows, P, r, m16, quo, rem, v)
    eng.sync()
    got = v.cpu().numpy()
    assert np.all(got == OK), np.flatnonzero(got != OK)[:8]
    eng.close()


@pytest.mark.gpu
def test_class_api(nb):
    N, q = 167, 128
    k = nb.NTRU({"N": N, "q": q})
    eng, rng, key = _engine(nb, N, q)
    ew, value = _honest_encrypt(eng, rng, key, 64, False)
    dw = _honest_decrypt(eng, rng, key, value, False)
    ew["remainderE"][3, 0] ^= 1
    dw["quotient2"][5, 1] = (dw["quotient2"][5, 1] + 1) % 3
    wit = _honest_inverse(eng, rng, 16)
    ep, dp = enc_params(N, q), dec_params(N, q)
    assert np.array_equal(k.verifyEncryptBatch(ew, ep), _check(eng, "encrypt", ew))
    assert np.array_equal(k.verifyDecryptBatch(dw, dp), _check(eng, "decrypt", dw))
    assert k.verifyEncryptBatch(ew, ep)[3] == 0 and k.verifyDecryptBatch(dw, dp)[5] == 0
    for case, (w, mod_p) in wit.items():
        params = [3, nq(3, N), N] if mod_p else [q, nq(q, N), N]
        got = k.verifyInverseBatch(w, params)
        assert np.array_equal(got, _check(eng, "inverse", w, mod_p)) and np.all(got == OK), case
    # a shared key row (1-D) gives the same verdicts as the same key on every row
    sw, _ = _honest_encrypt(eng, rng, key, 32, True)
    assert np.array_equal(k.verifyEncryptBatch(sw, ep), k.verifyEncryptBatch({**sw, "h": np.tile(sw["h"], (32, 1))}, ep))
    for bad in ([q * 2, nq(q, N), N], [q, nq(q, N) + 1, N], [q, nq(q, N), N + 1], [q, nq(q, N)]):
        with pytest.raises(ValueError):
            k.verifyEncryptBatch(ew, bad)
    for bad in ([q, nq(q, N), 5, nq(3, N), N], [q, nq(q, N), 3, nq(3, N) + 1, N], [q, nq(q, N), 3, nq(3, N), N - 1]):
        with pytest.raises(ValueError):
            k.verifyDecryptBatch(dw, bad)
    for bad in ([3, nq(q, N), N], [q, nq(3, N), N], [7, 1, N]):
        with pytest.raises(ValueError):
            k.verifyInverseBatch(wit["fq"][0], bad)
    eng.close()
