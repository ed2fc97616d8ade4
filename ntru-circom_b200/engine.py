"""Thin Python owner of one ``ntru_ctx`` (one GPU): numpy host buffers and raw device pointers.

All arithmetic happens in libntru_b200.so; this file only marshals buffers.
"""
from __future__ import annotations

import ctypes
from typing import Optional

import numpy as np

from . import _lib
from ._lib import NtruError


def _ptr(a) -> Optional[int]:
    """Address of a numpy array / torch tensor / int / None."""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    raise TypeError(f"cannot take the address of {type(a)}")


def _host(a, dtype, shape) -> np.ndarray:
    """C-contiguous numpy view of the exact dtype/shape the ABI expects (copies only if needed)."""
    if hasattr(a, "numpy") and not isinstance(a, np.ndarray):
        a = a.numpy()          # CPU torch tensor (possibly pinned): zero-copy
    a = np.ascontiguousarray(a, dtype=dtype)
    if a.shape != tuple(shape):
        raise IndexError(f"RangeError: expected shape {tuple(shape)}, got {a.shape}")
    return a


class Engine:
    """One context of the CUDA engine bound to one device."""

    def __init__(self, N: int, p: int, q: int, device: int = 0):
        self.lib = _lib.load()
        self.N, self.p, self.q = int(N), int(p), int(q)
        h = ctypes.c_void_p()
        rc = self.lib.ntru_create(ctypes.byref(h), self.N, self.p, self.q, int(device))
        if rc != _lib.NTRU_OK:
            raise NtruError(rc, {_lib.NTRU_E_CUDA: "no usable CUDA device (this engine has no CPU fallback)",
                                 _lib.NTRU_E_PARAM: "unsupported parameters N/p/q"}.get(
                                     rc, self.lib.ntru_strerror(rc).decode()))
        self._h = h
        self.device = int(device)
        self.pitch = int(self.lib.ntru_pitch(h))

    # -- plumbing ------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self.lib.ntru_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != _lib.NTRU_OK:
            raise NtruError(rc, self.lib.ntru_last_error(self._h).decode() or self.lib.ntru_strerror(rc).decode())

    def set_option(self, key: int, value: int):
        self._check(self.lib.ntru_set_option(self._h, key, value))

    def set_path(self, path: int):
        self.set_option(_lib.NTRU_OPT_PATH, path)

    def set_dec1_form(self, form: int):
        """tcgen05 schedule, first decrypt product at 256 < q <= 2048: 0 auto (fp16), 1 byte limbs, 2 fp16 tiles."""
        self.set_option(_lib.NTRU_OPT_DEC1_FORM, int(form))

    def set_schedule(self, cyc_plus_hi: bool):
        """tcgen05 schedule with the quotient witness: lo + hi phases (default) or the round-1 cyc + hi order."""
        self.set_option(_lib.NTRU_OPT_SCHEDULE, 1 if cyc_plus_hi else 0)

    def set_epilogue(self, mode: int):
        """tcgen05 schedule: 0 auto, 1 two epilogue groups (one per TMEM buffer), 2 one group on every phase."""
        self.set_option(_lib.NTRU_OPT_EPILOGUE, int(mode))

    def set_imma_form(self, generic: bool):
        """IMMA schedule: False = the kernel compiled for this N where there is one, True = the N bucket's generic kernel."""
        self.set_option(_lib.NTRU_OPT_IMMA_FORM, 1 if generic else 0)

    @property
    def launch_count(self) -> int:
        return int(self.lib.ntru_launch_count(self._h))

    @property
    def last_path(self) -> int:
        return int(self.lib.ntru_last_path(self._h))

    def set_timing(self, on: bool):
        self.set_option(_lib.NTRU_OPT_TIMING, 1 if on else 0)

    def timing_reset(self):
        self._check(self.lib.ntru_timing_reset(self._h))

    def timing_read(self) -> dict:
        """{kind: (total_ms, launches)} of the kernels launched since timing_reset (synchronises)."""
        out = {}
        for i, name in enumerate(_lib.KERNEL_KINDS):
            ms, n = ctypes.c_double(0), ctypes.c_uint64(0)
            self._check(self.lib.ntru_timing_read(self._h, i, ctypes.byref(ms), ctypes.byref(n)))
            if n.value:
                out[name] = (ms.value, int(n.value))
        return out

    def stream(self) -> int:
        return int(self.lib.ntru_stream(self._h) or 0)

    def set_stream(self, cuda_stream: int):
        self._check(self.lib.ntru_set_stream(self._h, cuda_stream))

    def sync(self):
        self._check(self.lib.ntru_sync(self._h))

    # -- keys ------------------------------------------------------------------------
    def set_public_key(self, h):
        h = _host(h, np.uint16, (self.N,))
        self._check(self.lib.ntru_set_public_key(self._h, _ptr(h)))

    def set_private_key(self, f, fp):
        f = _host(f, np.int8, (self.N,))
        fp = _host(fp, np.uint8, (self.N,))
        self._check(self.lib.ntru_set_private_key(self._h, _ptr(f), _ptr(fp)))

    # -- host-buffer batches (packed rows) ------------------------------------------------
    def encrypt_batch(self, r, m, *, h=None, witness=True, out=None, dr=None, return_r=False):
        """r, m: (B,N).  h: None (context key) or (B,N) distinct keys.  Returns dict of numpy arrays.

        r=None: the device draws r like index.js:89 (needs dr, here or through set_dr) from its keyed ChaCha20
        generator; return_r=True adds the r that was used (inputs.r, index.js:97) under "r"."""
        N = self.N
        m_arr = np.asarray(m)
        B = m_arr.shape[0]
        if r is not None:
            r = _host(np.ascontiguousarray(r, dtype=np.uint8), np.uint8, (B, N))
        elif dr is not None:
            self.set_dr(dr)
        wide = m_arr.dtype.itemsize > 1 and m_arr.size and int(m_arr.max(initial=0)) > 255
        m_arr = _host(m_arr, np.uint16 if wide else np.uint8, (B, N))
        out = out or {}
        value = out.get("value", np.empty((B, N), dtype=np.uint16))
        quo = out.get("quotientE", np.empty((B, N + 1), dtype=np.uint16)) if witness else None
        rem = out.get("remainderE", np.empty((B, N + 1), dtype=np.uint16)) if witness else None
        r_out = out.get("r", np.empty((B, N), dtype=np.uint8)) if (return_r or r is None) else None
        if h is not None:
            if wide:
                raise NtruError(_lib.NTRU_E_UNSUPPORTED, "wide messages with per-row keys")
            h = _host(h, np.uint16, (B, N))
            rc = self.lib.ntru_encrypt_batch_keys(self._h, B, _ptr(h), _ptr(r), _ptr(m_arr), _ptr(value),
                                                  _ptr(quo), _ptr(rem), _ptr(r_out))
        elif wide:
            rc = self.lib.ntru_encrypt_batch_wide(self._h, B, _ptr(r), _ptr(m_arr), _ptr(value), _ptr(quo),
                                                  _ptr(rem), _ptr(r_out))
        else:
            rc = self.lib.ntru_encrypt_batch(self._h, B, _ptr(r), _ptr(m_arr), _ptr(value), _ptr(quo), _ptr(rem),
                                             _ptr(r_out))
        self._check(rc)
        res = {"value": value, "quotientE": quo, "remainderE": rem}
        if r_out is not None:
            res["r"] = r_out
        return res

    def decrypt_batch(self, e, *, f=None, fp=None, witness=True, out=None):
        N = self.N
        e = np.ascontiguousarray(e, dtype=np.uint16)
        B = e.shape[0]
        e = _host(e, np.uint16, (B, N))
        out = out or {}
        value = out.get("value", np.empty((B, N), dtype=np.uint8))
        q1 = out.get("quotient1", np.empty((B, N + 1), dtype=np.uint16)) if witness else None
        r1 = out.get("remainder1", np.empty((B, N + 1), dtype=np.uint16)) if witness else None
        q2 = out.get("quotient2", np.empty((B, N + 1), dtype=np.uint8)) if witness else None
        r2 = out.get("remainder2", np.empty((B, N + 1), dtype=np.uint8)) if witness else None
        if f is not None or fp is not None:
            f = _host(f, np.int8, (B, N))
            fp = _host(fp, np.uint8, (B, N))
            rc = self.lib.ntru_decrypt_batch_keys(self._h, B, _ptr(f), _ptr(fp), _ptr(e), _ptr(value), _ptr(q1),
                                                  _ptr(r1), _ptr(q2), _ptr(r2))
        else:
            rc = self.lib.ntru_decrypt_batch(self._h, B, _ptr(e), _ptr(value), _ptr(q1), _ptr(r1), _ptr(q2),
                                             _ptr(r2))
        self._check(rc)
        return {"value": value, "quotient1": q1, "remainder1": r1, "quotient2": q2, "remainder2": r2}

    # -- the same two calls with every array as BN254 field elements on the wire (packOutput form) ------------
    def packed_elems(self, mod_q: bool, width: int) -> int:
        """Field elements per row of an array of `width` coefficients: packOutput(q - 1 or p - 1, width, .).outputSize."""
        return int(self.lib.ntru_packed_elems(self._h, 1 if mod_q else 0, int(width)))

    def _fe(self, arr, mod_q, width, B):
        return _host(np.ascontiguousarray(arr, dtype=np.uint32), np.uint32, (B, self.packed_elems(mod_q, width), 8))

    def encrypt_batch_packed(self, r, m, *, witness=True, out=None, dr=None, return_r=False):
        """encrypt_batch with r, m and every result as rows of field elements, (B, elems, 8) uint32 words:
        row = packOutput(maxVal, width, coefficients).expected (index.js:572-596), maxVal = p - 1 for r / m and q - 1
        for value / quotientE / remainderE.  Bits are packed and unpacked on the device."""
        N = self.N
        m = np.ascontiguousarray(m, dtype=np.uint32)
        B = m.shape[0]
        m = self._fe(m, False, N, B)
        if r is not None:
            r = self._fe(r, False, N, B)
        elif dr is not None:
            self.set_dr(dr)
        out = out or {}
        value = out.get("value", np.empty((B, self.packed_elems(True, N), 8), dtype=np.uint32))
        quo = out.get("quotientE", np.empty((B, self.packed_elems(True, N + 1), 8), dtype=np.uint32)) if witness else None
        rem = out.get("remainderE", np.empty((B, self.packed_elems(True, N + 1), 8), dtype=np.uint32)) if witness else None
        r_out = out.get("r", np.empty((B, self.packed_elems(False, N), 8), dtype=np.uint32)) if (return_r or r is None) else None
        self._check(self.lib.ntru_encrypt_batch_packed(self._h, B, _ptr(r), _ptr(m), _ptr(value), _ptr(quo), _ptr(rem), _ptr(r_out)))
        res = {"value": value, "quotientE": quo, "remainderE": rem}
        if r_out is not None:
            res["r"] = r_out
        return res

    def decrypt_batch_packed(self, e, *, witness=True, out=None):
        """decrypt_batch with e and every result as rows of field elements (maxVal = q - 1 for e / quotient1 /
        remainder1, p - 1 for value / quotient2 / remainder2)."""
        N = self.N
        e = np.ascontiguousarray(e, dtype=np.uint32)
        B = e.shape[0]
        e = self._fe(e, True, N, B)
        out = out or {}
        value = out.get("value", np.empty((B, self.packed_elems(False, N), 8), dtype=np.uint32))
        q1 = out.get("quotient1", np.empty((B, self.packed_elems(True, N + 1), 8), dtype=np.uint32)) if witness else None
        r1 = out.get("remainder1", np.empty((B, self.packed_elems(True, N + 1), 8), dtype=np.uint32)) if witness else None
        q2 = out.get("quotient2", np.empty((B, self.packed_elems(False, N + 1), 8), dtype=np.uint32)) if witness else None
        r2 = out.get("remainder2", np.empty((B, self.packed_elems(False, N + 1), 8), dtype=np.uint32)) if witness else None
        self._check(self.lib.ntru_decrypt_batch_packed(self._h, B, _ptr(e), _ptr(value), _ptr(q1), _ptr(r1), _ptr(q2), _ptr(r2)))
        return {"value": value, "quotient1": q1, "remainder1": r1, "quotient2": q2, "remainder2": r2}

    def verify_keys_batch(self, f, fq, fp, g):
        """verifyKeysInputs (index.js:141-197) for B keys: the quotientI / remainderI of the three
        multiply + divide-by-(1 - x^N) pairs (fq case and h case mod q, fp case mod p)."""
        N = self.N
        f = np.ascontiguousarray(f, dtype=np.int8)
        B = f.shape[0]
        f = _host(f, np.int8, (B, N))
        fq = _host(fq, np.uint16, (B, N))
        fp = _host(fp, np.uint8, (B, N))
        g = _host(g, np.int8, (B, N))
        out = {k: np.empty((B, N + 1), dtype=np.uint8 if k.endswith("_fp") else np.uint16)
               for k in ("quotient_fq", "remainder_fq", "quotient_fp", "remainder_fp", "quotient_h", "remainder_h")}
        self._check(self.lib.ntru_verify_keys_batch(self._h, B, _ptr(f), _ptr(fq), _ptr(fp), _ptr(g),
                                                    *[_ptr(out[k]) for k in ("quotient_fq", "remainder_fq", "quotient_fp",
                                                                             "remainder_fp", "quotient_h", "remainder_h")]))
        return out

    def keygen_batch(self, f, g):
        """loadPrivateKeyF + generatePublicKeyH for B keys (index.js:30-79): f, g ternary (B, N).  Returns fixed-length
        fq, fp, h and the validity mask (f invertible modulo 2 and modulo p)."""
        N = self.N
        f = np.ascontiguousarray(f, dtype=np.int8)
        B = f.shape[0]
        f = _host(f, np.int8, (B, N))
        g = _host(g, np.int8, (B, N))
        fq = np.empty((B, N), dtype=np.uint16)
        fp = np.empty((B, N), dtype=np.uint8)
        h = np.empty((B, N), dtype=np.uint16)
        valid = np.empty(B, dtype=np.uint8)
        self._check(self.lib.ntru_keygen_batch(self._h, B, _ptr(f), _ptr(g), _ptr(fq), _ptr(fp), _ptr(h), _ptr(valid)))
        return {"fq": fq, "fp": fp, "h": h, "valid": valid.astype(bool)}

    def keygen_dev(self, B, f, g, fq, fp, h, valid):
        """keygen_batch on device rows (pitch self.pitch; f, g int8, fq, h uint16, fp and valid bytes), asynchronous on
        the context's stream."""
        self._check(self.lib.ntru_keygen_dev(self._h, B, _ptr(f), _ptr(g), _ptr(fq), _ptr(fp), _ptr(h), _ptr(valid)))

    def generate_keys_dev(self, B, df, dg, f, g, fq, fp, h, seed=None):
        """generatePrivateKeyF + generateNewPublicKeyGH (index.js:51-79) for B keys into device rows: f, g drawn by the
        context's ChaCha20 generator (weights (df, df - 1) and (dg, dg)), non-invertible f redrawn on the device.
        seed: as in sample_r_dev (tests / benchmarks only)."""
        if seed is not None:
            self.set_rng_key(seed_key(seed), self.rng_next_row)
        self._check(self.lib.ntru_generate_keys_dev(self._h, B, int(df), int(dg), _ptr(f), _ptr(g), _ptr(fq), _ptr(fp),
                                                    _ptr(h)))

    def muldiv_dev(self, B, x, y, mod_p, quotient=None, remainder=None):
        """multiplyPolynomials(x, y, mod) + dividePolynomials(., 1 - x^N, mod), device-resident rows."""
        self._check(self.lib.ntru_muldiv_dev(self._h, B, _ptr(x), _ptr(y), int(bool(mod_p)), _ptr(quotient), _ptr(remainder)))

    # -- witness checks: VerifyEncrypt / VerifyDecrypt / VerifyInverse (ntru.circom:155-256), one verdict byte per row ------
    def _key(self, a, dtype, B):
        """A key array of a check: (N,) is one row shared by every witness, (B, N) one row per witness."""
        a = np.asarray(a)
        shared = a.ndim == 1
        return _host(a, dtype, (self.N,) if shared else (B, self.N)), shared

    def check_encrypt(self, h, r, m, quotientE, remainderE):
        """Verdicts (B,) uint8 of NTRU_CHECK_* bits for B VerifyEncrypt witnesses: r (B, N) bytes, m (B, N) uint16,
        quotientE / remainderE (B, N + 1) uint16; h (N,) shared or (B, N)."""
        N = self.N
        r = np.asarray(r)
        B = r.shape[0]
        h, shared = self._key(h, np.uint16, B)
        r = _host(r, np.uint8, (B, N))
        m = _host(m, np.uint16, (B, N))
        quo = _host(quotientE, np.uint16, (B, N + 1))
        rem = _host(remainderE, np.uint16, (B, N + 1))
        verdict = np.empty(B, dtype=np.uint8)
        self._check(self.lib.ntru_check_encrypt_batch(self._h, B, _ptr(h), int(shared), _ptr(r), _ptr(m), _ptr(quo), _ptr(rem),
                                                      _ptr(verdict)))
        return verdict

    def check_decrypt(self, f, fp, e, quotient1, remainder1, quotient2, remainder2):
        """Verdicts for B VerifyDecrypt witnesses: f (uint16, -1 as q - 1) and fp (bytes), both (N,) shared or (B, N);
        e (B, N) uint16; quotient1 / remainder1 (B, N + 1) uint16, quotient2 / remainder2 (B, N + 1) bytes."""
        N = self.N
        e = np.asarray(e)
        B = e.shape[0]
        f, shared = self._key(f, np.uint16, B)
        fp, fp_shared = self._key(fp, np.uint8, B)
        if shared != fp_shared:
            raise ValueError("f and fp must both be one shared row or both be one row per witness")
        e = _host(e, np.uint16, (B, N))
        q1 = _host(quotient1, np.uint16, (B, N + 1))
        r1 = _host(remainder1, np.uint16, (B, N + 1))
        q2 = _host(quotient2, np.uint8, (B, N + 1))
        r2 = _host(remainder2, np.uint8, (B, N + 1))
        verdict = np.empty(B, dtype=np.uint8)
        self._check(self.lib.ntru_check_decrypt_batch(self._h, B, _ptr(f), _ptr(fp), int(shared), _ptr(e), _ptr(q1), _ptr(r1),
                                                      _ptr(q2), _ptr(r2), _ptr(verdict)))
        return verdict

    def check_inverse(self, x, y, quotientI, remainderI, mod_p=False):
        """Verdicts for B VerifyInverse witnesses: x (B, N) uint16; modulo q, y (B, N) and quotientI / remainderI
        (B, N + 1) uint16; modulo p (mod_p=True, the fp case) the same as bytes."""
        N = self.N
        x = np.asarray(x)
        B = x.shape[0]
        t = np.uint8 if mod_p else np.uint16
        x = _host(x, np.uint16, (B, N))
        y = _host(y, t, (B, N))
        quo = _host(quotientI, t, (B, N + 1))
        rem = _host(remainderI, t, (B, N + 1))
        verdict = np.empty(B, dtype=np.uint8)
        self._check(self.lib.ntru_check_inverse_batch(self._h, B, int(bool(mod_p)), _ptr(x), _ptr(y), _ptr(quo), _ptr(rem),
                                                      _ptr(verdict)))
        return verdict

    def check_encrypt_dev(self, B, h, key_stride, r, m, quotientE, remainderE, verdict):
        """check_encrypt on device rows (pitch self.pitch), asynchronous; key_stride 0 (one h row) or self.pitch."""
        self._check(self.lib.ntru_check_encrypt_dev(self._h, B, _ptr(h), int(key_stride), _ptr(r), _ptr(m), _ptr(quotientE),
                                                    _ptr(remainderE), _ptr(verdict)))

    def check_decrypt_dev(self, B, f, fp, key_stride, e, quotient1, remainder1, quotient2, remainder2, verdict):
        self._check(self.lib.ntru_check_decrypt_dev(self._h, B, _ptr(f), _ptr(fp), int(key_stride), _ptr(e), _ptr(quotient1),
                                                    _ptr(remainder1), _ptr(quotient2), _ptr(remainder2), _ptr(verdict)))

    def check_inverse_dev(self, B, mod_p, x, y, quotientI, remainderI, verdict):
        self._check(self.lib.ntru_check_inverse_dev(self._h, B, int(bool(mod_p)), _ptr(x), _ptr(y), _ptr(quotientI),
                                                    _ptr(remainderI), _ptr(verdict)))

    # -- packOutput / unpackInput (index.js:572-620) on device rows --------------------------------------
    def pack_geometry(self, max_val: int, data_len: int):
        v = [ctypes.c_int() for _ in range(4)]
        self._check(self.lib.ntru_pack_geometry(int(max_val), int(data_len), *[ctypes.byref(x) for x in v]))
        return tuple(x.value for x in v)     # maxInputBits, inputsPerOutput, arrLen, outputSize

    def pack_output_dev(self, B, data, elem_bytes, data_len, pitch, max_val, out):
        self._check(self.lib.ntru_pack_output_dev(self._h, B, _ptr(data), int(elem_bytes), int(data_len), int(pitch), int(max_val),
                                                  _ptr(out)))

    def unpack_input_dev(self, B, data, n_elems, max_val, packed_bits, out, elem_bytes, pitch):
        self._check(self.lib.ntru_unpack_input_dev(self._h, B, _ptr(data), int(n_elems), int(max_val), int(packed_bits), _ptr(out),
                                                   int(elem_bytes), int(pitch)))

    def pack_output(self, max_val: int, data):
        """packOutput (index.js:572-596) for B host rows: data (B, dataLen) uint8 / uint16 -> (B, outputSize, 8) uint32
        words of BN254 field elements (32 bytes each, little-endian)."""
        data = np.ascontiguousarray(data)
        if data.dtype not in (np.uint8, np.uint16):
            raise TypeError("pack_output takes uint8 or uint16 rows")
        B, n = data.shape
        outs = self.pack_geometry(max_val, n)[3]
        out = np.empty((B, outs, 8), dtype=np.uint32)
        self._check(self.lib.ntru_pack_output(self._h, B, _ptr(data), data.dtype.itemsize, n, int(max_val), _ptr(out)))
        return out

    def unpack_input(self, max_val: int, packed_bits: int, packed, dtype=np.uint16):
        """unpackInput (index.js:598-620) for B host rows of field elements (B, nElems, 8) uint32 -> coefficients."""
        packed = np.ascontiguousarray(packed, dtype=np.uint32)
        B, n_elems = packed.shape[0], packed.shape[1]
        bits = max(1, int(max_val).bit_length())
        out = np.empty((B, (packed_bits // bits) * n_elems), dtype=dtype)
        self._check(self.lib.ntru_unpack_input(self._h, B, _ptr(packed), n_elems, int(max_val), int(packed_bits), _ptr(out),
                                               out.dtype.itemsize))
        return out

    def sum_allreduce(self, e):
        """Column sums mod q over the host rows of EVERY rank of the exchange (this rank alone without one)."""
        e = np.ascontiguousarray(e, dtype=np.uint16)
        B = e.shape[0]
        e = _host(e, np.uint16, (B, self.N))
        out = np.empty(self.N, dtype=np.uint16)
        self._check(self.lib.ntru_sum_allreduce(self._h, B, _ptr(e) if B else None, _ptr(out)))
        return out

    def sum(self, e):
        e = np.ascontiguousarray(e, dtype=np.uint16)
        B = e.shape[0]
        e = _host(e, np.uint16, (B, self.N))
        out = np.empty(self.N, dtype=np.uint16)
        self._check(self.lib.ntru_sum(self._h, B, _ptr(e), _ptr(out)))
        return out

    # -- device-resident batches (pitched rows; arguments: torch CUDA tensors or raw pointers) --------
    def encrypt_dev(self, B, r, m, value=None, quotientE=None, remainderE=None, h_rows=None):
        self._check(self.lib.ntru_encrypt_dev(self._h, B, _ptr(h_rows), _ptr(r), _ptr(m), _ptr(value),
                                              _ptr(quotientE), _ptr(remainderE)))

    def decrypt_dev(self, B, e, value=None, quotient1=None, remainder1=None, quotient2=None, remainder2=None,
                    f_rows=None, fp_rows=None):
        self._check(self.lib.ntru_decrypt_dev(self._h, B, _ptr(f_rows), _ptr(fp_rows), _ptr(e), _ptr(value),
                                              _ptr(quotient1), _ptr(remainder1), _ptr(quotient2),
                                              _ptr(remainder2)))

    def sum_partial_dev(self, B, e, partial):
        self._check(self.lib.ntru_sum_partial_dev(self._h, B, _ptr(e), _ptr(partial)))

    def sum_finalize_dev(self, partial, out):
        self._check(self.lib.ntru_sum_finalize_dev(self._h, _ptr(partial), _ptr(out)))

    # ---- cross-GPU sum over peer memory (include/ntru_b200.h: ntru_xchg_*, ntru_sum_allreduce_dev) ----
    def xchg_create(self, world: int, rank: int) -> bytes:
        """Allocates this rank's exchange window; returns its 64-byte CUDA IPC handle (all-gather it)."""
        buf = (ctypes.c_ubyte * 64)()
        self._check(self.lib.ntru_xchg_create(self._h, int(world), int(rank), buf))
        return bytes(buf)

    def xchg_connect(self, handles: bytes):
        """handles: world x 64 bytes, rank-major."""
        buf = (ctypes.c_ubyte * len(handles)).from_buffer_copy(handles)
        self._check(self.lib.ntru_xchg_connect(self._h, buf))

    def sum_allreduce_dev(self, B, e, out):
        """out[k] = column sums mod q over every rank's rows (local rows only when no exchange is connected)."""
        self._check(self.lib.ntru_sum_allreduce_dev(self._h, B, _ptr(e) if B else None, _ptr(out)))

    def sample_r_dev(self, B, dr, row0, r, seed=None):
        """generateCustomArray(N, dr, dr).map(-1 -> 2) into device rows for the global row numbers [row0, row0 + B),
        drawn by the context's ChaCha20 generator.  seed (tests / benchmarks only): first replaces the context's
        OS-entropy key by seed_key(seed), which makes the rows reproducible -- and predictable."""
        if seed is not None:
            self.set_rng_key(seed_key(seed), self.rng_next_row)
        self._check(self.lib.ntru_sample_r_dev(self._h, B, int(dr), int(row0), _ptr(r)))

    # ---- device generator for r (include/ntru_b200.h: ntru_set_rng_key) ----
    def set_dr(self, dr: int):
        self.set_option(_lib.NTRU_OPT_DR, int(dr))

    def set_rng_key(self, key: bytes, first_row: int = 0):
        """Replaces the OS-entropy key of the device generator (32 bytes) and sets the next row number."""
        if len(key) != 32:
            raise ValueError("the ChaCha20 key is 32 bytes")
        buf = (ctypes.c_ubyte * 32).from_buffer_copy(bytes(key))
        self._check(self.lib.ntru_set_rng_key(self._h, buf, int(first_row)))

    @property
    def rng_next_row(self) -> int:
        return int(self.lib.ntru_rng_next_row(self._h))

    def xchg_destroy(self):
        """Collective (sync + barrier over all ranks first): frees the exchange windows; raises if a peer had timed out."""
        self._check(self.lib.ntru_xchg_destroy(self._h))


# ---- host copy of the device generator (csrc/generic_kernels.cu: chacha20_block, k_sample_ternary) ------------------
# For the key holder's audit replay of device-drawn r and for the parity tests; never used to produce r in the product.
_M32 = 0xFFFFFFFF


def seed_key(seed: int) -> bytes:
    """32-byte key made of a small integer seed (tests / benchmarks: reproducible, NOT secret)."""
    return int(seed).to_bytes(32, "little")


def chacha20_block(key: bytes, counter: int, nonce: int):
    """ChaCha20 block function, D. J. Bernstein's layout: 32-byte key, 64-bit block counter, 64-bit nonce.
    Returns the 16 keystream words (uint32).  RFC 8439's 32-bit counter / 96-bit nonce is the same state with
    counter = ctr | nonce_word0 << 32 and nonce = nonce_word1 | nonce_word2 << 32."""
    k = [int.from_bytes(key[4 * i:4 * i + 4], "little") for i in range(8)]
    st = [0x61707865, 0x3320646E, 0x79622D32, 0x6B206574, *k,
          counter & _M32, (counter >> 32) & _M32, nonce & _M32, (nonce >> 32) & _M32]
    x = list(st)

    def rotl(v, n):
        return ((v << n) & _M32) | (v >> (32 - n))

    def qr(a, b, c, d):
        x[a] = (x[a] + x[b]) & _M32; x[d] = rotl(x[d] ^ x[a], 16)
        x[c] = (x[c] + x[d]) & _M32; x[b] = rotl(x[b] ^ x[c], 12)
        x[a] = (x[a] + x[b]) & _M32; x[d] = rotl(x[d] ^ x[a], 8)
        x[c] = (x[c] + x[d]) & _M32; x[b] = rotl(x[b] ^ x[c], 7)

    for _ in range(10):
        qr(0, 4, 8, 12); qr(1, 5, 9, 13); qr(2, 6, 10, 14); qr(3, 7, 11, 15)
        qr(0, 5, 10, 15); qr(1, 6, 11, 12); qr(2, 7, 8, 13); qr(3, 4, 9, 14)
    return [(a + b) & _M32 for a, b in zip(x, st)]


def sampler_draws(key: bytes, row: int, count: int):
    """The first `count` 32-bit draws of global row number `row`: what the device feeds, in order, to the Fisher-Yates
    steps i = N-1, N-2, ... of generateCustomArray (index.js:476-485), for r as for the key polynomials f and g."""
    out = []
    blk = 0
    while len(out) < count:
        out.extend(chacha20_block(key, blk, row))
        blk += 1
    return out[:count]
