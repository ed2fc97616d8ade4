"""ntru-circom_b200 -- B200-native batched NTRU engine behind the API of numtel/ntru-circom.

Importable as ``ntru_circom_b200`` (see the alias module at the repository root; a
hyphen cannot appear in an ``import`` statement).  The default export of the
reference, ``class NTRU``, and its named function exports are re-exported here.
"""
from .ntru import NTRU
from .engine import Engine, chacha20_block, sampler_draws, seed_key
from . import wire
from ._lib import (NtruError, PATH_AUTO, PATH_CUDA_CORE, PATH_TENSOR, PATH_IMMA, NTRU_CHECK_SATISFIED, NTRU_CHECK_CANONICAL,
                   NTRU_CHECK_DOMAIN)
from .poly import (addPolynomials, bigintToBits, bitsToBigInt, bitsToString, degree, dividePolynomials,
                   expandArray, expandArrayToMultiple, extendedEuclideanAlgorithm, generateCustomArray,
                   modInverse, multiplyPolynomials, multiplyPolynomialsByScalar, packOutput, polyInv,
                   stringToBits, subtractPolynomials, trimPolynomial, unpackInput)

__all__ = [
    "NTRU", "Engine", "NtruError", "wire", "PATH_AUTO", "PATH_CUDA_CORE", "PATH_TENSOR", "PATH_IMMA",
    "NTRU_CHECK_SATISFIED", "NTRU_CHECK_CANONICAL", "NTRU_CHECK_DOMAIN", "chacha20_block", "sampler_draws", "seed_key",
    "addPolynomials", "bigintToBits", "bitsToBigInt", "bitsToString", "degree", "dividePolynomials",
    "expandArray", "expandArrayToMultiple", "extendedEuclideanAlgorithm", "generateCustomArray",
    "modInverse", "multiplyPolynomials", "multiplyPolynomialsByScalar", "packOutput", "polyInv",
    "stringToBits", "subtractPolynomials", "trimPolynomial", "unpackInput",
]
