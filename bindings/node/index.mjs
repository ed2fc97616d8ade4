// Drop-in for the hot path of numtel/ntru-circom's index.js over the N-API shim (ntru_napi.c).
// NOT RUN IN THIS REPOSITORY'S IMAGE (no node).  Usage in the reference repository:
//     import NTRUReference, * as ref from './index.js';          // the reference, unchanged
//     import { accelerate } from 'ntru-b200/bindings/node/index.mjs';
//     const NTRU = accelerate(NTRUReference, ref);                // same class, GPU encryptBits/decryptBits
// Key generation, inversion and every helper stay the reference's own JavaScript (north_star).
import { createRequire } from 'node:module';
const native = createRequire(import.meta.url)('./ntru_b200.node');

const OPT_DR = 5;   // NTRU_OPT_DR (include/ntru_b200.h)

export function accelerate(NTRUReference, ref) {
  const { trimPolynomial, expandArray, generateCustomArray } = ref;
  return class NTRU extends NTRUReference {
    #ctx = null; #pub = null; #priv = null;
    #engine() {
      if (!this.#ctx) {
        this.#ctx = native.create(this.N, this.p, this.q, this.device ?? 0);
        native.setOption(this.#ctx, OPT_DR, this.dr);   // the device draws r itself when none is injected
      }
      return this.#ctx;
    }
    #loadPublic() {
      const ctx = this.#engine();
      if (this.#pub !== this.h) {                      // TypeError on h === null, like index.js:90
        native.setPublicKey(ctx, Uint16Array.from(expandArray(this.h, this.N, 0)));
        this.#pub = this.h;
      }
      return ctx;
    }
    #loadPrivate() {
      const ctx = this.#engine();
      if (this.#priv !== this.f) {
        native.setPrivateKey(ctx, Int8Array.from(expandArray(this.f, this.N, 0)), Uint8Array.from(expandArray(this.fp, this.N, 0)));
        this.#priv = this.f;
      }
      return ctx;
    }
    // m reduced into [0, q) like addPolynomials does (index.js:241); a byte array when every coefficient fits one,
    // otherwise the wide (uint16) entry point -- a coefficient >= 256 must NOT wrap modulo 256
    #message(mExp) {
      const q = this.q;
      const red = mExp.map(x => ((x % q) + q) % q);
      return red.some(x => x > 255) ? Uint16Array.from(red) : Uint8Array.from(red);
    }
    // index.js:87-110.  Without `r` the device draws it (generateCustomArray(N, dr, dr), -1 -> p-1, index.js:89) from
    // its entropy-keyed ChaCha20 generator; `r` is the injection seam the reference lacks.
    encryptBits(m, r = null) {
      const ctx = this.#loadPublic();
      const mExp = expandArray(m, this.N, 0);          // RangeError when m.length > N (index.js:98)
      const out = native.encryptBatch(ctx, 1, r === null ? null : Uint8Array.from(r), this.#message(mExp));
      const remainderE = Array.from(out.remainderE);
      return {
        value: trimPolynomial(remainderE),
        inputs: { r: Array.from(out.r), m: mExp, h: expandArray(this.h, this.N, 0), quotientE: Array.from(out.quotientE), remainderE },
        params: [this.q, this.calculateNq(), this.N],
      };
    }
    // index.js:111-140
    decryptBits(e) {
      const ctx = this.#loadPrivate();
      const eExp = expandArray(e, this.N, 0);          // RangeError when e.length > N (index.js:126)
      const q = this.q;
      const out = native.decryptBatch(ctx, 1, Uint16Array.from(eExp, x => ((x % q) + q) % q));
      const remainder2 = Array.from(out.remainder2);
      return {
        value: trimPolynomial(remainder2),
        inputs: {
          f: expandArray(this.f.map(x => x === -1 ? q - 1 : x), this.N, 0), fp: expandArray(this.fp, this.N, 0), e: eExp,
          quotient1: Array.from(out.quotient1), remainder1: Array.from(out.remainder1),
          quotient2: Array.from(out.quotient2), remainder2,
        },
        params: [this.q, this.calculateNq(), this.p, this.calculateNp(), this.N],
      };
    }
    // index.js:141-197: the three multiply + divide pairs run on the GPU, checks and witness assembly as upstream
    verifyKeysInputs() {
      for (const [k, label] of [['f', 'private key F'], ['fq', 'private key Fq'], ['fp', 'private key Fp'], ['g', 'private key G']])
        if (!this[k]) throw new Error(`missing ${label}`);
      if (!this.h) throw new Error('missing public key H');
      const { q, p, N } = this, nq = this.calculateNq(), np = this.calculateNp();
      const ex = a => expandArray(a, N, 0);
      const o = native.verifyKeysBatch(this.#engine(), 1, Int8Array.from(ex(this.f)), Uint16Array.from(ex(this.fq)),
                                       Uint8Array.from(ex(this.fp)), Int8Array.from(ex(this.g)));
      const fmodq = this.f.map(x => x === -1 ? q - 1 : x), fmodp = this.f.map(x => x === -1 ? p - 1 : x);
      const fqp = this.fq.map(x => x * p), g = this.g.map(x => x === -1 ? q - 1 : x);
      const rem = a => trimPolynomial(Array.from(a));
      if (rem(o.remainderFq).length !== 1 && o.remainderFq[0] !== 1) throw new Error('invalid fq');   // sic, index.js:159
      if (rem(o.remainderFp).length !== 1 && o.remainderFp[0] !== 1) throw new Error('invalid fp');
      const hRem = rem(o.remainderH);
      if (this.h.reduce((out, cur, i) => out || hRem[i] !== cur, false)) throw new Error('invalid h');
      const c = (params, a, b, qI, rI) => ({ params, inputs: { f: ex(a), fq: ex(b), quotientI: Array.from(qI), remainderI: Array.from(rI) } });
      return {
        fq: c([q, nq, N], fmodq, this.fq, o.quotientFq, o.remainderFq),
        fp: c([p, np, N], fmodp, this.fp, o.quotientFp, o.remainderFp),
        h: c([q, nq, N], g, fqp, o.quotientH, o.remainderH),
      };
    }
    // engine-native unit of work: B rows per call, typed arrays in and out (fixed length, un-trimmed).
    // r: Uint8Array(B x N) or null (device-drawn, returned as .r); m: Uint8Array, or Uint16Array for coefficients
    // above 255; hs / fs, fps: one key per row.
    encryptBitsBatch(B, r, m, hs = null) { return native.encryptBatch(hs ? this.#engine() : this.#loadPublic(), B, r, m, hs); }
    decryptBitsBatch(B, e, fs = null, fps = null) { return native.decryptBatch(fs ? this.#engine() : this.#loadPrivate(), B, e, fs, fps); }
    // the same two with every array as rows of BN254 field elements on the wire -- row = packOutput(maxVal, width,
    // coefficients).expected as 8 little-endian uint32 words per element, maxVal = q - 1 for the arrays modulo q and
    // p - 1 for r, m and the arrays modulo p: what CombineArray / UnpackArray take, and two thirds of the bytes
    encryptBitsBatchPacked(B, r, m) { return native.encryptBatchPacked(this.#loadPublic(), B, r, m); }
    decryptBitsBatchPacked(B, e) { return native.decryptBatchPacked(this.#loadPrivate(), B, e); }
    sumCiphertexts(B, e) { return trimPolynomial(Array.from(native.sum(this.#engine(), B, e))); }
    // packOutput / unpackInput (index.js:572-620) for B rows at once; field elements as 8 little-endian uint32 words
    packOutputBatch(B, maxVal, data, dataLen) { return native.packOutput(this.#engine(), B, maxVal, data, dataLen); }
    unpackInputBatch(B, maxVal, packedBits, data, nElems, wide = true) {
      return native.unpackInput(this.#engine(), B, maxVal, packedBits, data, nElems, wide);
    }
    // cross-GPU sum (one NTRU instance = one rank = one GPU; the caller moves the 64-byte handles between its worker
    // processes and passes a barrier before xchgDestroy)
    xchgCreate(world, rank) { return native.xchgCreate(this.#engine(), world, rank); }
    xchgConnect(handles, world) { native.xchgConnect(this.#engine(), handles, world); }
    xchgDestroy() { native.xchgDestroy(this.#engine()); }
    sumCiphertextsAllRanks(B, e) { return trimPolynomial(Array.from(native.sumAllreduce(this.#engine(), B, e))); }
    // B key pairs: f, g drawn here like generatePrivateKeyF / generateNewPublicKeyGH do (index.js:51-71), inverses,
    // lifting and h in the engine; rows whose f is not invertible come back with valid = 0 (redraw them)
    generateKeysBatch(B) {
      const f = new Int8Array(B * this.N), g = new Int8Array(B * this.N);
      for (let b = 0; b < B; b++) {
        f.set(generateCustomArray(this.N, this.df, this.df - 1), b * this.N);
        g.set(generateCustomArray(this.N, this.dg, this.dg), b * this.N);
      }
      return { f, g, ...native.keygenBatch(this.#engine(), B, f, g) };
    }
    // witness checks (VerifyEncrypt / VerifyDecrypt / VerifyInverse) for B witnesses: inputs under the reference's key
    // names as flat typed arrays of B rows (h, f, fp may be one row of N), params as the reference emits them.
    // Returns Uint8Array(B) verdicts: bit 1 satisfied, 2 canonical (what dividePolynomials returns), 4 not evaluated.
    #checkParams(params, want, what) {
      if (params.length !== want.length || params.some((x, i) => Number(x) !== want[i]))
        throw new Error(`${what} params ${params} do not match this instance's ${want}`);
    }
    verifyEncryptBatch(B, inputs, params) {
      this.#checkParams(params, [this.q, this.calculateNq(), this.N], 'VerifyEncrypt');
      const { h, r, m, quotientE, remainderE } = inputs;
      return native.checkEncryptBatch(this.#engine(), B, h, h.length === this.N, r, m, quotientE, remainderE);
    }
    verifyDecryptBatch(B, inputs, params) {
      this.#checkParams(params, [this.q, this.calculateNq(), this.p, this.calculateNp(), this.N], 'VerifyDecrypt');
      const { f, fp, e, quotient1, remainder1, quotient2, remainder2 } = inputs;
      return native.checkDecryptBatch(this.#engine(), B, f, fp, f.length === this.N, e, quotient1, remainder1, quotient2, remainder2);
    }
    verifyInverseBatch(B, inputs, params) {
      const modP = Number(params[0]) === this.p;
      this.#checkParams(params, modP ? [this.p, this.calculateNp(), this.N] : [this.q, this.calculateNq(), this.N], 'VerifyInverse');
      const { f, fq, quotientI, remainderI } = inputs;
      return native.checkInverseBatch(this.#engine(), B, modP, f, fq, quotientI, remainderI);
    }
    close() { if (this.#ctx) { native.destroy(this.#ctx); this.#ctx = null; this.#pub = this.#priv = null; } }
  };
}
