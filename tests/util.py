"""Shared test helpers: library loaders, deterministic input streams, golden vectors, edge cases.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg import this module; it is the
one place that loads anything under oracle/.
"""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
import sys
sys.path.insert(0, ROOT)
from libgoldilocks_b200.capi import BatchLib  # noqa: E402

P = 2**448 - 2**224 - 1
Q = 2**446 - 0x8335dc163bb124b65129c96fde933d8d723a70aadc873d6d54a7bb0d

_cache = {}


def _load(key, path, build=None):
    if key not in _cache:
        if not os.path.exists(path) and build:
            subprocess.run(build, cwd=ROOT, check=True)
        _cache[key] = BatchLib(path) if os.path.exists(path) else None
    return _cache[key]


def oracle_lib():
    lib = _load("oracle", os.path.join(ROOT, "oracle", "liboracle.so"), ["make", "-C", "oracle", "oracle"])
    assert lib is not None, "oracle/liboracle.so failed to build"
    return lib


def ref_lib(arch="x86_64"):
    """the original libgoldilocks as `make -C oracle ref REF=<its source tree>` built it; None when it was not built"""
    return _load("ref_" + arch, os.path.join(ROOT, "oracle", "_ref", "libgoldilocks_ref_%s.so" % arch))


def checker_lib():
    return ref_lib() or oracle_lib()


def hostsim_lib():
    lib = _load("sim", os.path.join(ROOT, "tests", "hostsim", "_hostsim.so"), ["make", "hostsim"])
    assert lib is not None
    return lib


def set_threads(lib, t):
    for name in ("refb_set_threads", "oracle_set_threads", "hostsim_set_threads"):
        if lib.has(name):
            getattr(lib.lib, name)(C.c_int(int(t)))


def golden_vectors():
    with open(os.path.join(ROOT, "tests", "golden", "reference_vectors.json")) as f:
        return json.load(f)


def openssl_golden():
    """Ed448 / X448 outputs of OpenSSL on seeded inputs (tools/openssl_vectors.py)"""
    with np.load(os.path.join(ROOT, "tests", "golden", "openssl_ed448_x448.npz")) as z:
        return {k: z[k] for k in z.files}


def stream_bytes(label, n):
    """n bytes of the SHAKE256 stream keyed by "b200-goldilocks/<label>/448" (SURVEY.md 8(d))."""
    return np.frombuffer(hashlib.shake_256(("b200-goldilocks/%s/448" % label).encode()).digest(int(n)), dtype=np.uint8).copy()


def le(x, nbytes=56):
    return np.frombuffer(int(x).to_bytes(nbytes, "little"), dtype=np.uint8)


def from_le(row):
    return int.from_bytes(bytes(row), "little")


def field_edge_values():
    """56-byte strings the field tests always include (SURVEY.md 8(d) C1 edge block)."""
    vals = [0, 1, 2, P - 1, P, P + 1, 2**224 - 1, 2**224, 2**224 + 1, 2**448 - 1, 2**447, (P - 1) // 2, (P + 1) // 2,
            2**448 - 2**224, sum(0xfffffff << (28 * i) for i in range(0, 16, 2)), sum(0xfffffff << (28 * i) for i in range(1, 16, 2))]
    return np.stack([le(v) for v in vals])


def field_inputs(label, n):
    """n random 56-byte strings followed by the edge block squared out against itself"""
    e = field_edge_values()
    a = np.concatenate([stream_bytes(label + "/a", n * 56).reshape(n, 56), np.repeat(e, len(e), axis=0)])
    b = np.concatenate([stream_bytes(label + "/b", n * 56).reshape(n, 56), np.tile(e, (len(e), 1))])
    return a, b


def scalar_edge_bytes():
    adj = (2**450 - 1) % Q
    vals = [0, 1, 2, Q - 1, Q - 2, (Q - adj) % Q, (Q - adj + 1) % Q, (Q - adj - 1) % Q, (Q + 1) // 2, 2**445, 2**446 - 1 - (2**446 - Q)]
    return np.stack([le(v % Q) for v in vals])


def coords(lib, pts):
    """canonical X|Y|Z|T bytes (4 x 56) of packed point structs: limbs are radix 2^56, any weakly reduced value"""
    pts = np.ascontiguousarray(pts, dtype=np.uint8).reshape(-1, 4, 8, 8)
    limbs = pts.view("<u8").reshape(-1, 4, 8)
    out = np.empty((len(limbs), 4, 56), np.uint8)
    for i in range(len(limbs)):
        for c in range(4):
            v = sum(int(limbs[i, c, k]) << (56 * k) for k in range(8)) % P
            out[i, c] = le(v)
    return out.reshape(len(limbs), 224)


def coords_fast(lib, pts):
    """same as coords() through the checker's C helper when it has one"""
    for name in ("refb_point_coords_batch", "oracle_point_coords_batch"):
        if lib.has(name):
            pts = np.ascontiguousarray(pts, dtype=np.uint8).reshape(-1, 256)
            out = np.empty((len(pts), 224), np.uint8)
            getattr(lib.lib, name)(C.c_void_p(out.ctypes.data), C.c_void_p(pts.ctypes.data), C.c_size_t(len(pts)))
            return out
    return coords(lib, pts)


def random_points(chk, label, n):
    return chk.from_hash_uniform(stream_bytes(label, n * 112).reshape(n, 112))


def random_scalars(chk, label, n):
    return chk.scalar_decode_long(stream_bytes(label, n * 56).reshape(n, 56), 56)


def verify_corpus(signer, label, n, msg_len=None, corrupt_every=8):
    """keys, messages, signatures (made by `signer`) with every `corrupt_every`-th entry corrupted in
    one of the ways SURVEY.md 8(d) C4 lists; returns (sig, pk, msgs, kinds) -- kinds[i] = 0 for untouched."""
    sk = stream_bytes(label + "/sk", n * 57).reshape(n, 57)
    if msg_len is None:
        lens = stream_bytes(label + "/len", n).astype(np.int64)
    else:
        lens = np.full(n, msg_len, np.int64)
    blob = stream_bytes(label + "/msg", int(lens.sum()) + 1)
    offs = np.concatenate([[0], np.cumsum(lens)])
    msgs = [bytes(blob[offs[i]:offs[i + 1]]) for i in range(n)]
    pk = signer.ed448_derive_public_key(sk)
    sig = signer.ed448_sign(sk, pk, msgs)
    kinds = np.zeros(n, np.int32)
    sel = stream_bytes(label + "/sel", 2 * n)
    for i in range(0, n, corrupt_every):
        kind = 1 + (i // corrupt_every) % 6
        kinds[i] = kind
        bit = 1 << (sel[2 * i] & 7)
        pos = int(sel[2 * i + 1])
        if kind == 1:
            sig[i, pos % 57] ^= bit                      # bit flip in R
        elif kind == 2:
            sig[i, 57 + pos % 56] ^= bit                 # bit flip in S
        elif kind == 3:
            pk[i, pos % 57] ^= bit                       # bit flip in A
        elif kind == 4:
            m = bytearray(msgs[i]) or bytearray(b"\0")
            m[pos % len(m)] ^= bit
            msgs[i] = bytes(m)                           # message changed (or grown from empty)
        elif kind == 5:
            s = from_le(sig[i, 57:114]) + Q              # S + q: still ACCEPTED by the reference (no range check)
            sig[i, 57:114] = le(s, 57)
        elif kind == 6:
            pk[i, :] = le(1, 57)                         # y = 1: rejected by the reference's decoder
    return sig, pk, msgs, kinds
