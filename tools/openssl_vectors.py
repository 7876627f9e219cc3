#!/usr/bin/env python3
"""Writes tests/golden/openssl_ed448_x448.npz: Ed448 public keys, signatures and verdicts and X448 outputs on seeded
random inputs, computed by OpenSSL (through the `cryptography` package).  RFC 8032 and RFC 7748 fix these bytes, so they
are what the reference (otrv4/libgoldilocks) returns on the same inputs; the tests compare the oracle, the host simulator
and the product with them without needing the reference's sources.

Verdicts follow OpenSSL, which rejects S >= q; the reference accepts S + q (tests/util.py verify_corpus kind 5), so the
tests leave that kind out of the comparison.  The tests read only the .npz; run this once where `cryptography` exists.
"""
import os
import sys

import numpy as np
from cryptography.exceptions import InvalidSignature
from cryptography.hazmat.primitives.asymmetric import ed448, x448

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import util  # noqa: E402
from libgoldilocks_b200.capi import pack_messages  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "openssl_ed448_x448.npz")
N = 384


class OpenSSL:
    """the two signer calls util.verify_corpus makes, one element at a time"""

    @staticmethod
    def ed448_derive_public_key(sk):
        return np.stack([np.frombuffer(ed448.Ed448PrivateKey.from_private_bytes(bytes(s)).public_key().public_bytes_raw(), np.uint8) for s in sk])

    @staticmethod
    def ed448_sign(sk, pk, msgs):
        return np.stack([np.frombuffer(ed448.Ed448PrivateKey.from_private_bytes(bytes(s)).sign(m), np.uint8) for s, m in zip(sk, msgs)])


def verify(sig, pk, msg):
    try:
        ed448.Ed448PublicKey.from_public_bytes(bytes(pk)).verify(bytes(sig), msg)
        return -1
    except (InvalidSignature, ValueError):
        return 0


def main():
    sig, pk, msgs, kinds = util.verify_corpus(OpenSSL, "golden/openssl", N)
    status = np.array([verify(s, p, m) for s, p, m in zip(sig, pk, msgs)], np.int32)
    arena, off = pack_messages(msgs)
    u = util.stream_bytes("golden/openssl/u", N * 56).reshape(N, 56)
    k = util.stream_bytes("golden/openssl/k", N * 56).reshape(N, 56)
    xo = np.stack([np.frombuffer(x448.X448PrivateKey.from_private_bytes(bytes(b)).exchange(x448.X448PublicKey.from_public_bytes(bytes(a))), np.uint8)
                   for a, b in zip(u, k)])
    sk = util.stream_bytes("golden/openssl/sk", N * 57).reshape(N, 57)       # the keys verify_corpus signed with
    np.savez(OUT, sk=sk, sig=sig, pk=pk, arena=arena, off=off, kinds=kinds, status=status, x448_u=u, x448_k=k, x448_out=xo)
    print("wrote", os.path.relpath(OUT, ROOT), os.path.getsize(OUT), "bytes; verdicts: %d accepted of %d" % ((status == -1).sum(), N))


if __name__ == "__main__":
    main()
