"""Every subset of requested outputs on every schedule, with guard rows around device and host outputs.

include/ntru_b200.h lets any output pointer be NULL.  On the tcgen05 schedule the set of non-NULL pointers also picks
the kernel's work: whether the quotient phases run (csrc/umma_kernels.cu: umma_encrypt / umma_decrypt set with_hi),
which store slot an array goes to (value, else the remainder, takes the first cyclic slot), which TMA stores are issued
(out_mask) and which pad-column memsets run (launch_product).  The IMMA and CUDA-core kernels test each pointer on its
own.  So every requested array is compared bit for bit, pad columns included, with a run that requested everything.

Every output is a separate (G + B + G)-row allocation: the call gets rows [G, G + B), every row is pre-filled with a
sentinel, and after the call the G guard rows on either side must still hold it (torch allocations lie next to each
other, so a store past row B - 1 would corrupt another tensor without an error).  Outputs that were not requested must
be untouched, and so must every input.

The engines use random keys (the engine takes any h in [0, q), f in {-1, 0, 1}, fp in [0, p)) and random inputs: r and
m in {0, 1, 2}, e uniform in [0, q).
"""
import ctypes
import itertools

import numpy as np
import pytest

import ntru_oracle as o

pytestmark = pytest.mark.gpu

AUTO, CORE, TCGEN05, IMMA = 0, 1, 2, 3         # ntru_circom_b200.PATH_*
ENC_KEYS = ("value", "quotientE", "remainderE")
DEC_KEYS = ("value", "quotient1", "remainder1", "quotient2", "remainder2")
WIDE = {"quotientE", "remainderE", "quotient1", "remainder1"}     # uint16 arrays (enc value too)
G = 256                                        # guard rows: one tcgen05 tile (a CTA pair's 256 rows)
B = 2 * 74 * 256 + 77                          # every CTA pair of a B200 gets > 1 tile; the last tile holds 77 rows
S16, S8 = 0x5A5A, 0xA5                         # sentinels of 16-bit and byte arrays

# (N, q) and the tcgen05 branch of launch_product / geometry() (csrc/umma_kernels.cu) that each one is here for.
SHAPES = [
    (167, 128, "dec1_one_limb"),                     # q <= 256: one K limb in the first decrypt product
    (509, 2048, "dec1f_one_group"),                  # fp16 first decrypt product, one epilogue group, resident A
    (512, 2048, "pad_memset"),                       # chunks cover 512 < pitch 528 columns: the pad memsets run
    (677, 2048, "enc_one_unit_dec1f_streamed"),      # ENC one-unit passes, message from global; fp16 DEC1, A streamed
    (701, 8192, "dec1_two_limb_one_group"),          # two K limbs, one epilogue group
    (821, 4096, "dec1_two_limb_two_groups_tma_a"),   # two K limbs, two epilogue groups, A operand streamed by TMA
    (1024, 8192, "eight_chunks_pad_memset_no_imma"), # ENC at kMaxChunks chunks, pad memsets; IMMA supports N <= 832
]
SHAPE_IDS = [f"N{n}q{q}-{name}" for n, q, name in SHAPES]


def _subsets(keys):
    return [s for k in range(len(keys) + 1) for s in itertools.combinations(keys, k)]


ALL_SETS = {"encrypt": _subsets(ENC_KEYS), "decrypt": _subsets(DEC_KEYS)}
VARIANT_SETS = {
    "encrypt": [("quotientE",), ("remainderE",), ("value", "remainderE"), ("quotientE", "remainderE")],
    "decrypt": [("quotient1",), ("remainder1",), ("quotient2",), ("remainder2",), ("quotient1", "remainder2"),
                ("value", "remainder2"), ("remainder1", "quotient2"), ("value", "quotient1")],
}


def _imma_ok(N):
    return N <= 832                                  # csrc/imma_kernels.cu: imma_supported


def _sample(n):
    """first row, the end of the first tile, the first row of the second, the first row of the last tile, last row"""
    return [0, 255, 256, (n - 1) // 256 * 256, n - 1]


def _host(t):
    a = t.cpu().numpy()
    return a.view(np.uint16) if a.dtype == np.int16 else a


@pytest.fixture(scope="module")
def nb():
    import ntru_circom_b200 as nb
    return nb


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


def _rows(torch, gen, n, P, N, lo, hi, dtype):
    t = torch.zeros((n, P), dtype=dtype, device="cuda")
    t[:, :N] = torch.randint(lo, hi, (n, N), generator=gen, device="cuda", dtype=dtype)
    return t


def _guarded(torch, op, P):
    if op == "encrypt":
        return {k: torch.empty((G + B + G, P), dtype=torch.int16, device="cuda") for k in ENC_KEYS}
    return {k: torch.empty((G + B + G, P), dtype=torch.int16 if k in WIDE else torch.uint8, device="cuda")
            for k in DEC_KEYS}


def _sentinel(t):
    return S16 if t.element_size() == 2 else S8


class Case:
    """One engine per (N, q), its inputs (and clones to check them against), guarded outputs, and the full-output
    references: same key on the default tcgen05 schedule, distinct keys on the CUDA-core schedule."""

    def __init__(self, nb, torch, N, q):
        self.torch, self.N, self.q, self.p = torch, N, q, 3
        rng = np.random.default_rng(N * 7 + q)
        self.key = {"h": rng.integers(0, q, N), "f": rng.integers(-1, 2, N), "fp": rng.integers(0, 3, N)}
        self.eng = eng = nb.Engine(N, 3, q, 0)
        eng.set_public_key(self.key["h"].astype(np.uint16))
        eng.set_private_key(self.key["f"].astype(np.int8), self.key["fp"].astype(np.uint8))
        self.P = P = eng.pitch
        gen = torch.Generator(device="cuda").manual_seed(N + q)
        self.x = {"r": _rows(torch, gen, B, P, N, 0, 3, torch.uint8), "m": _rows(torch, gen, B, P, N, 0, 3, torch.uint8),
                  "e": _rows(torch, gen, B, P, N, 0, q, torch.int16), "h_rows": _rows(torch, gen, B, P, N, 0, q, torch.int16),
                  "f_rows": _rows(torch, gen, B, P, N, -1, 2, torch.int8),
                  "fp_rows": _rows(torch, gen, B, P, N, 0, 3, torch.uint8)}
        self.x0 = {k: v.clone() for k, v in self.x.items()}
        self.bufs = {op: _guarded(torch, op, P) for op in ("encrypt", "decrypt")}
        self.ref = {}
        for op in ("encrypt", "decrypt"):
            keys = ENC_KEYS if op == "encrypt" else DEC_KEYS
            eng.set_path(AUTO)
            self.ref[op, False] = self.run(op, keys, False, TCGEN05, None, ("reference", op))
            self.check_oracle(op, False)
            eng.set_path(CORE)
            self.ref[op, True] = self.run(op, keys, True, CORE, None, ("reference", op, "keys"))
            self.check_oracle(op, True)
        eng.set_path(AUTO)
        torch.cuda.synchronize()

    def run(self, op, req, distinct, path, want, what):
        """One call with the outputs `req` into the middle rows of the guarded buffers; checks the guard rows, the
        outputs not requested and the inputs, and each requested array against want (if given).  Returns clones of
        the requested arrays."""
        torch, eng, x = self.torch, self.eng, self.x
        bufs = self.bufs[op]
        for t in bufs.values():
            t.fill_(_sentinel(t))
        out = {k: bufs[k][G:G + B] for k in req}
        torch.cuda.synchronize()                    # the engine runs on its own non-blocking stream
        if op == "encrypt":
            eng.encrypt_dev(B, x["r"], x["m"], h_rows=x["h_rows"] if distinct else None, **out)
        else:
            eng.decrypt_dev(B, x["e"], f_rows=x["f_rows"] if distinct else None,
                            fp_rows=x["fp_rows"] if distinct else None, **out)
        eng.sync()
        assert eng.last_path == path, what
        for k, t in bufs.items():
            s = _sentinel(t)
            if k not in req:
                assert bool((t == s).all()), (what, k, "written but not requested")
                continue
            assert bool((t[:G] == s).all()), (what, k, "guard rows before row 0")
            assert bool((t[G + B:] == s).all()), (what, k, "guard rows after row B - 1")
            if want is not None:
                assert torch.equal(t[G:G + B], want[k]), (what, k)
        for k, v in x.items():
            assert torch.equal(v, self.x0[k]), (what, k, "input changed")
        return {k: bufs[k][G:G + B].clone() for k in req}

    def check_oracle(self, op, distinct):
        torch, N, q, p = self.torch, self.N, self.q, self.p
        idx = torch.tensor(_sample(B), device="cuda")
        rows = {k: _host(v[idx])[:, :N].astype(np.int64) for k, v in self.x.items()}
        if op == "encrypt":
            want = o.encrypt_batch(rows["h_rows"] if distinct else self.key["h"], rows["r"], rows["m"], q)
        else:
            want = o.decrypt_batch(rows["f_rows"] if distinct else self.key["f"],
                                   rows["fp_rows"] if distinct else self.key["fp"], rows["e"], q, p)
        for k, got in self.ref[op, distinct].items():
            a = _host(got[idx])
            w = want[k].shape[1]
            assert np.array_equal(a[:, :w], want[k]), ("oracle", op, distinct, k)
            assert not a[:, w:].any(), ("oracle", op, distinct, k, "pad columns")


@pytest.fixture(scope="module")
def cases(nb, torch):
    made = {}

    def get(N, q):
        if (N, q) not in made:
            made[N, q] = Case(nb, torch, N, q)
        return made[N, q]
    yield get
    for c in made.values():
        c.eng.close()


# ---- 1 + 2. device-resident output sets, guard rows and untouched inputs ------------------------------------------

# schedule -> (path option, distinct keys, path the call must report)
SCHEDULES = {"tcgen05": (AUTO, False, TCGEN05), "imma": (IMMA, False, IMMA), "cuda_core": (CORE, False, CORE),
             "imma_keys": (IMMA, True, IMMA), "cuda_core_keys": (CORE, True, CORE)}


@pytest.mark.parametrize("schedule", list(SCHEDULES))
@pytest.mark.parametrize("op", ["encrypt", "decrypt"])
@pytest.mark.parametrize("N,q", [s[:2] for s in SHAPES], ids=SHAPE_IDS)
def test_device_output_sets(N, q, op, schedule, cases):
    """All 8 subsets of the encrypt outputs and all 32 of the decrypt outputs, the empty set included: each requested
    array equals the full-output reference of the same keys on every row, pad columns included."""
    path, distinct, want_path = SCHEDULES[schedule]
    if want_path == IMMA and not _imma_ok(N):
        pytest.skip("the IMMA schedule supports N <= 832")
    c = cases(N, q)
    c.eng.set_path(path)
    try:
        for req in ALL_SETS[op]:
            c.run(op, req, distinct, want_path, c.ref[op, distinct], (schedule, op, req))
    finally:
        c.eng.set_path(AUTO)


# variant -> (Engine setter, value, default value, ops)
VARIANTS = {"cyc_hi_schedule": ("set_schedule", True, False, ("encrypt", "decrypt")),
            "epilogue1": ("set_epilogue", 1, 0, ("encrypt", "decrypt")),
            "epilogue2": ("set_epilogue", 2, 0, ("encrypt", "decrypt")),
            "dec1_form1": ("set_dec1_form", 1, 0, ("decrypt",)),
            "dec1_form2": ("set_dec1_form", 2, 0, ("decrypt",))}
VARIANT_PARAMS = [pytest.param(n, q, op, v, id=f"{sid}-{op}-{v}")
                  for (n, q, _), sid in zip(SHAPES, SHAPE_IDS) for op in ("encrypt", "decrypt") for v in VARIANTS
                  if op in VARIANTS[v][3] and (not v.startswith("dec1_form") or 256 < q <= 2048)]


@pytest.mark.parametrize("N,q,op,variant", VARIANT_PARAMS)
def test_tcgen05_variant_output_sets(N, q, op, variant, cases):
    """The round-1 phase order, both epilogue arrangements and both first-decrypt-product forms, each with the output
    sets that move arrays between store slots or drop the phases of one part: equal to the default full-output run."""
    setter, value, default, _ = VARIANTS[variant]
    c = cases(N, q)
    c.eng.set_path(TCGEN05)
    getattr(c.eng, setter)(value)
    try:
        for req in VARIANT_SETS[op]:
            c.run(op, req, False, TCGEN05, c.ref[op, False], (variant, op, req))
    finally:
        getattr(c.eng, setter)(default)
        c.eng.set_path(AUTO)


# ---- 3. host-buffer entry points across pipeline chunks -----------------------------------------------------------

CHUNK = 8192
BH = 3 * CHUNK + 1000          # four chunks on two pipeline slots; the last (1000 rows) is below the 4096-row switch
HOST_SETS = {"encrypt": [(), ("value",), ("quotientE",), ("remainderE",), ("value", "remainderE"),
                         ("quotientE", "remainderE")],
             "decrypt": [(), ("value",), ("remainder2",), ("quotient1", "remainder2"), ("remainder1", "quotient2"),
                         ("value", "quotient1", "remainder1", "quotient2", "remainder2")]}
HOST_SAMPLE = [0, CHUNK - 1, CHUNK, 3 * CHUNK - 1, 3 * CHUNK, BH - 1]


class HostMem:
    """numpy arrays in pageable memory or in ntru_host_alloc (pinned) memory, freed by close()"""

    def __init__(self, lib, pinned):
        self.lib, self.pinned, self.ptrs = lib, pinned, []

    def array(self, shape, dtype):
        if not self.pinned:
            return np.empty(shape, dtype)
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = self.lib.ntru_host_alloc(n)
        assert p, "ntru_host_alloc"
        self.ptrs.append(p)
        return np.ctypeslib.as_array((ctypes.c_uint8 * n).from_address(p)).view(dtype).reshape(shape)

    def copy(self, a):
        out = self.array(a.shape, a.dtype)
        out[...] = a
        return out

    def close(self):
        for p in self.ptrs:
            self.lib.ntru_host_free(p)
        self.ptrs = []


def _fe_words(values):
    """BN254 field elements (Python ints) -> (elems, 8) uint32 little-endian words"""
    return np.array([[(v >> (32 * i)) & 0xFFFFFFFF for i in range(8)] for v in values], dtype=np.uint32)


def _ptr(a):
    return None if a is None else a.ctypes.data


@pytest.mark.parametrize("memory", ["pageable", "pinned"])
@pytest.mark.parametrize("form", ["plain", "keys", "packed"])
@pytest.mark.parametrize("N,q", [(509, 2048), (1024, 8192)], ids=["N509q2048", "N1024q8192"])
def test_host_output_sets(N, q, form, memory, cases, nb):
    """ntru_encrypt_batch / ntru_decrypt_batch, their _keys and _packed forms with explicit NULL outputs, 8192-row
    chunks: one call reuses both pipeline slots, and on the same-key path its last chunk runs on the IMMA schedule
    where N allows it, the others on tcgen05.  Outputs are host arrays with sentinel guard rows; plain rows must equal
    the device-resident full-output run, packed rows its packOutput (the library's packer on every row, the oracle's
    on the chunk boundaries)."""
    c = cases(N, q)
    eng, lib, p = c.eng, c.eng.lib, c.p
    distinct = form == "keys"
    mem = HostMem(lib, memory == "pinned")
    eng.set_option(nb._lib.NTRU_OPT_CHUNK_ROWS, CHUNK)
    eng.set_path(AUTO)
    try:
        x = {k: _host(v[:BH])[:, :N].copy() for k, v in c.x.items()}
        if form == "packed":
            x = {"r": eng.pack_output(p - 1, x["r"]), "m": eng.pack_output(p - 1, x["m"]),
                 "e": eng.pack_output(q - 1, x["e"])}
        x = {k: mem.copy(v) for k, v in x.items()}
        x0 = {k: v.copy() for k, v in x.items()}
        for op in ("encrypt", "decrypt"):
            keys = ENC_KEYS if op == "encrypt" else DEC_KEYS
            ref = {k: _host(v[:BH]) for k, v in c.ref[op, distinct].items()}
            width = {k: N if k == "value" else N + 1 for k in keys}
            mod_q = {k: k in WIDE or (op == "encrypt") for k in keys}
            want = {}
            for k in keys:
                rows = np.ascontiguousarray(ref[k][:, :width[k]])
                if form == "packed":
                    mv = q - 1 if mod_q[k] else p - 1
                    want[k] = eng.pack_output(mv, rows)
                    for b in HOST_SAMPLE:
                        fe = o.pack_output(mv, width[k], rows[b].tolist())["expected"]
                        assert np.array_equal(want[k][b], _fe_words(fe)), (op, k, b, "packOutput")
                else:
                    want[k] = rows
            bufs = {}
            for k in keys:
                shape = (G + BH + G,) + want[k].shape[1:]
                bufs[k] = mem.array(shape, want[k].dtype)
            for req in HOST_SETS[op]:
                what = (form, memory, op, req)
                for k in req:
                    bufs[k].view(np.uint8)[...] = S8 if want[k].dtype == np.uint8 else 0x5A
                arg = {k: bufs[k][G:G + BH] if k in req else None for k in keys}
                if op == "encrypt":
                    outs = [_ptr(arg[k]) for k in ENC_KEYS] + [None]
                    if form == "plain":
                        rc = lib.ntru_encrypt_batch(eng._h, BH, _ptr(x["r"]), _ptr(x["m"]), *outs)
                    elif form == "keys":
                        rc = lib.ntru_encrypt_batch_keys(eng._h, BH, _ptr(x["h_rows"]), _ptr(x["r"]), _ptr(x["m"]), *outs)
                    else:
                        rc = lib.ntru_encrypt_batch_packed(eng._h, BH, _ptr(x["r"]), _ptr(x["m"]), *outs)
                else:
                    outs = [_ptr(arg[k]) for k in DEC_KEYS]
                    if form == "plain":
                        rc = lib.ntru_decrypt_batch(eng._h, BH, _ptr(x["e"]), *outs)
                    elif form == "keys":
                        rc = lib.ntru_decrypt_batch_keys(eng._h, BH, _ptr(x["f_rows"]), _ptr(x["fp_rows"]), _ptr(x["e"]),
                                                         *outs)
                    else:
                        rc = lib.ntru_decrypt_batch_packed(eng._h, BH, _ptr(x["e"]), *outs)
                assert rc == 0, (what, rc, lib.ntru_last_error(eng._h))
                last = (IMMA if _imma_ok(N) else CORE) if distinct else (IMMA if _imma_ok(N) else TCGEN05)
                assert eng.last_path == last, what
                for k in req:
                    s = S8 if want[k].dtype == np.uint8 else 0x5A
                    assert (bufs[k][:G].view(np.uint8) == s).all(), (what, k, "guard rows before row 0")
                    assert (bufs[k][G + BH:].view(np.uint8) == s).all(), (what, k, "guard rows after row B - 1")
                    assert np.array_equal(bufs[k][G:G + BH], want[k]), (what, k)
                for k, v in x.items():
                    assert np.array_equal(v, x0[k]), (what, k, "input changed")
    finally:
        eng.set_option(nb._lib.NTRU_OPT_CHUNK_ROWS, 32768)
        mem.close()


# ---- 4. ntru_sum_partial_dev ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("fill", ["all_q_minus_1", "uniform"])
def test_sum_partial_dev_contract(fill, nb, torch):
    """hrss701 (q = 8192), 2^20 rows, two sum_partial_dev calls into one partial that starts at random words: every
    column of partial is congruent to its start plus twice the column sum modulo 2^16 (so modulo q), and
    sum_finalize_dev returns that total modulo q, with zeros up to the pitch."""
    N, q, n = 701, 8192, 1 << 20
    eng = nb.Engine(N, 3, q, 0)
    try:
        P = eng.pitch
        gen = torch.Generator(device="cuda").manual_seed(701)
        if fill == "uniform":
            e = _rows(torch, gen, n, P, N, 0, q, torch.int16)
        else:
            e = torch.zeros((n, P), dtype=torch.int16, device="cuda")
            e[:, :N] = q - 1
        start = torch.randint(-(1 << 31), 1 << 31, (P,), generator=gen, device="cuda", dtype=torch.int64)
        partial = start.to(torch.int32)
        out = torch.full((P,), S16, dtype=torch.int16, device="cuda")
        colsum = torch.sum(e, dim=0, dtype=torch.int64)
        torch.cuda.synchronize()
        eng.sum_partial_dev(n, e, partial)
        eng.sum_partial_dev(n, e, partial)
        eng.sum_finalize_dev(partial, out)
        eng.sync()
        total = start + 2 * colsum
        got = partial.to(torch.int64) & 0xFFFF
        bad = torch.nonzero(got != (total & 0xFFFF)).flatten().tolist()
        assert not bad, (fill, "partial columns not congruent modulo 2^16", bad[:8])
        fin = _host(out)
        assert np.array_equal(fin[:N], _host(total[:N] % q).astype(np.uint16)), (fill, "finalize")
        assert not fin[N:].any(), (fill, "finalize pad columns")
    finally:
        eng.close()
