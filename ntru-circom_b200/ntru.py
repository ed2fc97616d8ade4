"""``class NTRU`` -- host-side mirror of the reference's scheme API (index.js:7-207).

Same constructor options and defaults, same field and method names, same
``{value, inputs, params}`` results (``inputs`` is the key the reference's code
uses; ``input`` is offered as an alias because the README spells it that way).
``encryptBits`` / ``decryptBits`` / ``encryptStr`` / ``decryptStr`` run on the
GPU through libntru_b200.so; single-key generation and inversion stay on the host
(``poly.py``), batched key generation (``generateKeysBatch``, ``generateKeysDevice``)
runs on the GPU.  Additional batch methods (``encryptBitsBatch``,
``decryptBitsBatch``, ``sumCiphertexts``) expose the engine's real unit of
work: many ciphertexts per call.
"""
from __future__ import annotations

import math
from typing import Callable, List, Optional, Sequence

import numpy as np

from . import poly
from .engine import Engine
from ._lib import NtruError


class _Result(dict):
    """dict with the README's ``input`` alias for ``inputs`` (index.js:96 vs README.md:123)."""

    def __getitem__(self, k):
        return super().__getitem__("inputs" if k == "input" else k)


class NTRU:
    def __init__(self, options: Optional[dict] = None, **kw):
        # index.js:9-23
        self.N, self.p, self.q = 167, 3, 128
        self.df, self.dg, self.dr = 61, 20, 18
        self.f = self.fp = self.fq = self.g = self.h = None
        self.device = 0                 # extension: which GPU this instance computes on
        self.rand32: Optional[Callable[[], int]] = None   # extension: replaces crypto.getRandomValues
        for k, v in {**(options or {}), **kw}.items():
            setattr(self, k, v)
        # index.js:25-27
        self.I = [0] * (self.N + 1)
        self.I[0] = 1
        self.I[-1] = -1
        self._eng: Optional[Engine] = None
        self._pub_loaded = None
        self._priv_loaded = None

    # ---- engine plumbing -----------------------------------------------------------
    def engine(self) -> Engine:
        if self._eng is None:
            self._eng = Engine(self.N, self.p, self.q, self.device)
        return self._eng

    def _load_public(self) -> Engine:
        if self.h is None:
            raise TypeError("Cannot read properties of null (reading 'length')")   # index.js:90 on h === null
        eng = self.engine()
        key = tuple(int(x) for x in self.h)
        if key != self._pub_loaded:
            eng.set_public_key(np.array(poly.expandArray(self.h, self.N, 0), dtype=np.uint16))
            self._pub_loaded = key
        return eng

    def _load_private(self) -> Engine:
        if self.f is None:
            raise TypeError("Cannot read properties of null (reading 'map')")       # index.js:112 on f === null
        if self.fp is None:
            raise TypeError("Cannot read properties of null (reading 'length')")
        eng = self.engine()
        key = (tuple(int(x) for x in self.f), tuple(int(x) for x in self.fp))
        if key != self._priv_loaded:
            f = np.array(poly.expandArray(self.f, self.N, 0), dtype=np.int64)
            if np.any(np.abs(f) > 1):
                raise NtruError(-7, "the engine needs a ternary private key f in {-1,0,1}")
            eng.set_private_key(f.astype(np.int8), np.array(poly.expandArray(self.fp, self.N, 0), dtype=np.uint8))
            self._priv_loaded = key
        return eng

    # ---- keys: host reference code (index.js:30-79) --------------------------------------
    def loadPrivateKeyF(self, fArr: Sequence[int]) -> bool:
        p, q = self.p, self.q
        self.f = [int(x) for x in fArr]
        self.fq = poly.polyInv(self.f, self.I, q)
        self.fp = poly.polyInv(self.f, self.I, p)
        fmodq = [q - 1 if x == -1 else x for x in self.f]
        fmodp = [p - 1 if x == -1 else x for x in self.f]
        fqDiv = poly.dividePolynomials(poly.multiplyPolynomials(self.fq, fmodq, q), self.I, q)
        if len(fqDiv["remainder"]) != 1 and fqDiv["remainder"][0] != 1:     # sic: index.js:42
            raise ValueError("invalid fq")
        fpDiv = poly.dividePolynomials(poly.multiplyPolynomials(self.fp, fmodp, p), self.I, p)
        if len(fpDiv["remainder"]) != 1 and fpDiv["remainder"][0] != 1:     # sic: index.js:45
            raise ValueError("invalid fp")
        return True

    def generatePrivateKeyF(self):
        tries, ok = 0, False
        while (not ok or not (self.fq and self.fp)) and tries < 100:
            tries += 1
            try:
                ok = self.loadPrivateKeyF(poly.generateCustomArray(self.N, self.df, self.df - 1, self.rand32))
            except ValueError:
                pass
        if not self.fq or not self.fp:
            raise ValueError("Could not find invertible f")

    def generateKeysBatch(self, B: int) -> dict:
        """B key pairs at once (SURVEY 8f-3): generatePrivateKeyF + generateNewPublicKeyGH (index.js:51-79) with the
        same draws (generateCustomArray with weights (df, df - 1) for f and (dg, dg) for g) and the same retry rule
        (redraw f while it is not invertible, at most 100 times).  The draws come from rand32 on the host; the inversions,
        the lifting to q and h run on the GPU (ntru_keygen_batch).  Returns fixed-length numpy arrays."""
        N = self.N
        eng = self.engine()
        f = np.zeros((B, N), dtype=np.int8)
        g = np.array([poly.generateCustomArray(N, self.dg, self.dg, self.rand32) for _ in range(B)], dtype=np.int8).reshape(B, N)
        out = {"fq": np.zeros((B, N), dtype=np.uint16), "fp": np.zeros((B, N), dtype=np.uint8), "h": np.zeros((B, N), dtype=np.uint16)}
        todo = np.arange(B)
        for _ in range(100):
            if todo.size == 0:
                break
            f[todo] = np.array([poly.generateCustomArray(N, self.df, self.df - 1, self.rand32) for _ in todo], dtype=np.int8).reshape(-1, N)
            res = eng.keygen_batch(f[todo], g[todo])
            ok = res["valid"]
            for k in out:
                out[k][todo[ok]] = res[k][ok]
            todo = todo[~ok]
        if todo.size:
            raise ValueError("Could not find invertible f")              # index.js:63
        return {"f": f, "g": g, **out}

    def generateKeysDevice(self, B: int) -> dict:
        """B key pairs drawn and computed entirely on the GPU (ntru_generate_keys_dev): f with weights (df, df - 1), g
        with (dg, dg) from the engine's ChaCha20 generator, non-invertible f redrawn there (at most 100 rounds).  Returns
        torch CUDA tensors (B, pitch) f, g (int8), fq, h (int16 holding uint16), fp (uint8), ready to pass as h_rows /
        f_rows / fp_rows to Engine.encrypt_dev / decrypt_dev.  The tensors are complete on return."""
        import torch
        eng = self.engine()
        dev = torch.device("cuda", eng.device)
        P = eng.pitch
        out = {"f": torch.empty((B, P), dtype=torch.int8, device=dev), "g": torch.empty((B, P), dtype=torch.int8, device=dev),
               "fq": torch.empty((B, P), dtype=torch.int16, device=dev), "fp": torch.empty((B, P), dtype=torch.uint8, device=dev),
               "h": torch.empty((B, P), dtype=torch.int16, device=dev)}
        eng.generate_keys_dev(B, self.df, self.dg, out["f"], out["g"], out["fq"], out["fp"], out["h"])
        eng.sync()
        return out

    def generateNewPublicKeyGH(self):
        self.g = poly.generateCustomArray(self.N, self.dg, self.dg, self.rand32)
        self.generatePublicKeyH()

    def generatePublicKeyH(self):
        if not self.f:
            raise ValueError("missing private key F")
        if not self.g:
            raise ValueError("missing private key G")
        pFq = poly.multiplyPolynomialsByScalar(self.fq, self.p, self.q)
        pFqG = poly.multiplyPolynomials(pFq, self.g, self.q)
        self.h = poly.trimPolynomial(poly.dividePolynomials(pFqG, self.I, self.q)["remainder"])

    # ---- strings (index.js:80-86) ------------------------------------------------------
    def encryptStr(self, inputPlain: str) -> List[int]:
        return self.encryptBits(poly.stringToBits(inputPlain))["value"]

    def decryptStr(self, encrypted: Sequence[int]) -> str:
        return poly.bitsToString(poly.expandArrayToMultiple(self.decryptBits(encrypted)["value"], 8))

    # ---- strings, many per call (SURVEY 8f-4: the codec of index.js:80-86, 516-556 around the batch engine) ----
    def encryptStrBatch(self, strings: Sequence[str], *, split: bool = False) -> np.ndarray:
        """encryptStr for every string: 8 bits per character, MSB first (stringToBits, index.js:538-546).  Returns the
        (B, N) ciphertext rows, fixed length (un-trimmed).  The reference has "no provision to split into words"
        (index.js:81): a string longer than floor(N / 8) characters raises like expandArray does, unless
        ``split=True`` -- then it is cut into blocks of floor(N / 8) characters and the result is a list of
        (blocks_i, N) arrays, one per string (the last block zero padded)."""
        N, cpb = self.N, self.N // 8
        blocks, owner = [], []
        for si, text in enumerate(strings):
            codes = [ord(ch) for ch in text]
            if any(c > 0xFF for c in codes):
                raise NtruError(-1, "encryptStrBatch handles characters up to 0xFF (8 bits each, index.js:541-543)")
            if len(codes) > cpb and not split:
                raise IndexError("RangeError: Invalid array length")          # index.js:98 via expandArray
            for b0 in range(0, max(len(codes), 1), cpb):
                blocks.append(codes[b0:b0 + cpb])
                owner.append(si)
        ms = np.zeros((len(blocks), N), dtype=np.uint8)
        for bi, codes in enumerate(blocks):
            if codes:
                ms[bi, :8 * len(codes)] = np.unpackbits(np.array(codes, dtype=np.uint8), bitorder="big")
        value = self.encryptBitsBatch(ms, witness=False)["value"] if len(blocks) else np.zeros((0, N), dtype=np.uint16)
        if not split:
            return value
        owner = np.array(owner, dtype=np.int64)
        return [value[owner == si] for si in range(len(strings))]

    def decryptStrBatch(self, es) -> List[str]:
        """decryptStr for every row of es ((B, N) ciphertexts) -- or, for a list of (blocks_i, N) arrays as returned by
        encryptStrBatch(split=True), one string per entry with its blocks concatenated.  Like the reference
        (index.js:84-86, 548-556) the plaintext is trimmed, padded to a multiple of 8 and read 8 bits per character:
        trailing NUL characters of a block are lost."""
        if isinstance(es, (list, tuple)) and len(es) and np.asarray(es[0]).ndim == 2:
            sizes = [np.asarray(e).shape[0] for e in es]
            flat = self.decryptStrBatch(np.concatenate([np.asarray(e) for e in es], axis=0))
            out, pos = [], 0
            for n in sizes:
                out.append("".join(flat[pos:pos + n]))
                pos += n
            return out
        es = np.asarray(es)
        if es.shape[0] == 0:
            return []
        plain = self.decryptBitsBatch(es, witness=False)["value"]
        out = []
        for row in plain:
            bits = poly.expandArrayToMultiple(poly.trimPolynomial(row.tolist()), 8)
            out.append(poly.bitsToString(bits))
        return out

    # ---- hot path: one ciphertext (index.js:87-140) -----------------------------------------
    def sampleR(self) -> List[int]:
        """index.js:89."""
        return [self.p - 1 if x == -1 else x
                for x in poly.generateCustomArray(self.N, self.dr, self.dr, self.rand32)]

    def encryptBits(self, m: Sequence[int], r: Optional[Sequence[int]] = None):
        N, q = self.N, self.q
        eng = self._load_public()
        r = self.sampleR() if r is None else [int(x) for x in r]
        m = [int(x) for x in m]
        m_exp = poly.expandArray(m, N, 0)                        # RangeError when len(m) > N (index.js:98)
        if len(r) != N:
            raise IndexError("RangeError: r must have N coefficients")
        out = eng.encrypt_batch(np.array([r], dtype=np.uint8), np.mod(np.array([m_exp], dtype=np.int64), q))
        rem = out["remainderE"][0].tolist()
        return _Result(
            value=poly.trimPolynomial(rem),
            inputs={
                "r": r,
                "m": m_exp,
                "h": poly.expandArray(self.h, N, 0),
                "quotientE": out["quotientE"][0].tolist(),
                "remainderE": rem,
            },
            params=[q, self.calculateNq(), N],
        )

    def decryptBits(self, e: Sequence[int]):
        N, q, p = self.N, self.q, self.p
        eng = self._load_private()
        e = [int(x) for x in e]
        e_exp = poly.expandArray(e, N, 0)                        # RangeError when len(e) > N (index.js:126)
        out = eng.decrypt_batch(np.mod(np.array([e_exp], dtype=np.int64), q).astype(np.uint16))
        rem2 = out["remainder2"][0].tolist()
        return _Result(
            value=poly.trimPolynomial(rem2),
            inputs={
                "f": poly.expandArray([q - 1 if x == -1 else x for x in self.f], N, 0),
                "fp": poly.expandArray(self.fp, N, 0),
                "e": e_exp,
                "quotient1": out["quotient1"][0].tolist(),
                "remainder1": out["remainder1"][0].tolist(),
                "quotient2": out["quotient2"][0].tolist(),
                "remainder2": rem2,
            },
            params=[q, self.calculateNq(), p, self.calculateNp(), N],
        )

    # ---- hot path: batches (engine-native unit of work) ------------------------------------------
    def encryptBitsBatch(self, ms, rs=None, *, hs=None, witness: bool = True):
        """ms: (B,N) messages (zero padded); rs: (B,N) in {0,1,2} or None: drawn like index.js:89 -- on the DEVICE by
        the engine's entropy-keyed ChaCha20 generator, or on the host when a ``rand32`` was injected (tests);
        hs: optional (B,N) distinct public keys.  Returns fixed-length numpy arrays (un-trimmed); "r" is included
        whenever the call drew it (inputs.r, index.js:97)."""
        ms = np.asarray(ms)
        B = ms.shape[0]
        if ms.ndim != 2 or ms.shape[1] > self.N:
            raise IndexError("RangeError: Invalid array length")
        if ms.shape[1] < self.N:
            ms = np.pad(ms, ((0, 0), (0, self.N - ms.shape[1])))
        drew = rs is None
        if drew and self.rand32 is not None:
            rs = np.array([self.sampleR() for _ in range(B)], dtype=np.uint8).reshape(B, self.N)
        eng = self.engine() if hs is not None else self._load_public()
        return eng.encrypt_batch(rs, np.mod(ms.astype(np.int64), self.q) if ms.dtype.kind == "i" else ms,
                                 h=hs, witness=witness, dr=self.dr if rs is None else None, return_r=drew)

    def decryptBitsBatch(self, es, *, fs=None, fps=None, witness: bool = True):
        es = np.asarray(es)
        if es.ndim != 2 or es.shape[1] > self.N:
            raise IndexError("RangeError: Invalid array length")
        if es.shape[1] < self.N:
            es = np.pad(es, ((0, 0), (0, self.N - es.shape[1])))
        eng = self.engine() if fs is not None else self._load_private()
        return eng.decrypt_batch(es, f=fs, fp=fps, witness=witness)

    def sumCiphertexts(self, es) -> List[int]:
        """Fold of addPolynomials(., ., q) over the rows of es (test/reference.test.js:58), trimmed."""
        es = np.asarray(es)
        if es.ndim != 2 or es.shape[1] > self.N:
            raise IndexError("RangeError: Invalid array length")
        if es.shape[1] < self.N:
            es = np.pad(es, ((0, 0), (0, self.N - es.shape[1])))
        return poly.trimPolynomial(self.engine().sum(es).tolist())

    # ---- key witness: host reference code (index.js:141-197) -------------------------------------
    def verifyKeysInputs(self):
        for name, label in (("f", "private key F"), ("fq", "private key Fq"), ("fp", "private key Fp"),
                            ("g", "private key G")):
            if not getattr(self, name):
                raise ValueError(f"missing {label}")
        if not self.h:
            raise ValueError("missing public key H")
        q, p, N = self.q, self.p, self.N
        nq, np_ = self.calculateNq(), self.calculateNp()
        fmodq = [q - 1 if x == -1 else x for x in self.f]
        fmodp = [p - 1 if x == -1 else x for x in self.f]
        fq, fp = self.fq, self.fp
        fqp = [x * p for x in fq]
        g = [q - 1 if x == -1 else x for x in self.g]
        # the three multiplyPolynomials + dividePolynomials(., I, .) pairs (index.js:158-166) run on the GPU
        # (ntru_verify_keys_batch); trimming and the reference's checks stay here
        ex0 = lambda a: poly.expandArray(a, N, 0)   # noqa: E731
        if any(abs(int(x)) > 1 for x in self.f) or any(abs(int(x)) > 1 for x in self.g):
            raise NtruError(-7, "the engine needs ternary f and g in {-1,0,1}")
        gpu = self.engine().verify_keys_batch(np.array([ex0(self.f)], dtype=np.int8), np.array([ex0(fq)], dtype=np.uint16),
                                              np.array([ex0(fp)], dtype=np.uint8), np.array([ex0(self.g)], dtype=np.int8))
        div = lambda c: {"quotient": poly.trimPolynomial([int(x) for x in gpu["quotient_" + c][0]]),   # noqa: E731
                         "remainder": poly.trimPolynomial([int(x) for x in gpu["remainder_" + c][0]])}
        fqDiv, fpDiv, hDiv = div("fq"), div("fp"), div("h")
        if len(fqDiv["remainder"]) != 1 and fqDiv["remainder"][0] != 1:
            raise ValueError("invalid fq")
        if len(fpDiv["remainder"]) != 1 and fpDiv["remainder"][0] != 1:
            raise ValueError("invalid fp")
        if any((hDiv["remainder"][i] if i < len(hDiv["remainder"]) else None) != cur for i, cur in enumerate(self.h)):
            raise ValueError("invalid h")
        ex = poly.expandArray
        return {
            "fq": {"params": [q, nq, N],
                   "inputs": {"f": ex(fmodq, N, 0), "fq": ex(fq, N, 0),
                              "quotientI": ex(fqDiv["quotient"], N + 1, 0), "remainderI": ex(fqDiv["remainder"], N + 1, 0)}},
            "fp": {"params": [p, np_, N],
                   "inputs": {"f": ex(fmodp, N, 0), "fq": ex(fp, N, 0),
                              "quotientI": ex(fpDiv["quotient"], N + 1, 0), "remainderI": ex(fpDiv["remainder"], N + 1, 0)}},
            "h": {"params": [q, nq, N],
                  "inputs": {"f": ex(g, N, 0), "fq": ex(fqp, N, 0),
                             "quotientI": ex(hDiv["quotient"], N + 1, 0), "remainderI": ex(hDiv["remainder"], N + 1, 0)}},
        }

    # ---- witness checks: the circuits' constraint systems (ntru.circom:155-256) for many witnesses at once ------------
    def _check_params(self, params, want, what):
        got = [int(x) for x in params]
        if got != want:
            raise ValueError(f"{what} params {got} do not match this instance's {want}")

    def verifyEncryptBatch(self, inputs: dict, params) -> np.ndarray:
        """VerifyEncrypt for B witnesses: inputs under the reference's names (r, m, h, quotientE, remainderE), each
        (B, width); h may be one (N,) row.  Returns the uint8 verdicts (NTRU_CHECK_SATISFIED | _CANONICAL | _DOMAIN)."""
        self._check_params(params, [self.q, self.calculateNq(), self.N], "VerifyEncrypt")
        return self.engine().check_encrypt(inputs["h"], inputs["r"], inputs["m"], inputs["quotientE"], inputs["remainderE"])

    def verifyDecryptBatch(self, inputs: dict, params) -> np.ndarray:
        """VerifyDecrypt for B witnesses (f, fp, e, quotient1, remainder1, quotient2, remainder2); f and fp may be one
        (N,) row each."""
        self._check_params(params, [self.q, self.calculateNq(), self.p, self.calculateNp(), self.N], "VerifyDecrypt")
        return self.engine().check_decrypt(inputs["f"], inputs["fp"], inputs["e"], inputs["quotient1"], inputs["remainder1"],
                                           inputs["quotient2"], inputs["remainder2"])

    def verifyInverseBatch(self, inputs: dict, params) -> np.ndarray:
        """VerifyInverse for B witnesses (f, fq, quotientI, remainderI) as verifyKeysInputs emits them; params[0] picks the
        case: q (the fq and h cases) or p (the fp case)."""
        mod_p = len(params) > 0 and int(params[0]) == self.p
        want = [self.p, self.calculateNp(), self.N] if mod_p else [self.q, self.calculateNq(), self.N]
        self._check_params(params, want, "VerifyInverse")
        return self.engine().check_inverse(inputs["f"], inputs["fq"], inputs["quotientI"], inputs["remainderI"], mod_p=mod_p)

    # ---- index.js:201-206 ----------------------------------------------------------------
    def calculateNq(self) -> int:
        return math.ceil(math.log2(self.q * self.q * self.N))

    def calculateNp(self) -> int:
        return math.ceil(math.log2(self.p * self.p * self.N))
