"""X448 peer sets (goldilocks_b200_x448_peerset_*, goldilocks_x448_peerset_batch[_dev]): every output byte and status must be
what goldilocks_x448 returns for the same (peer u, scalar), for honest peers (comb tables), peers with torsion, twist and
non-canonical u (ladder or comb, whichever the set picked), edge scalars and out-of-range peer indices."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import util
from util import le, stream_bytes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = 2**448 - 2**224 - 1
Q = 2**446 - 0x8335dc163bb124b65129c96fde933d8d723a70aadc873d6d54a7bb0d
A = 156326
SUCCESS, FAILURE = -1, 0


def _sqrt(a):
    """a square root of a mod p, or None (p = 3 mod 4)"""
    a %= P
    r = pow(a, (P + 1) // 4, P)
    return r if r * r % P == a else None


def _rhs(u):
    return (u * u * u + A * u * u + u) % P


def _m_add(p1, p2):
    """affine addition on curve448 (v^2 = u^3 + A u^2 + u); None is the point at infinity"""
    if p1 is None:
        return p2
    if p2 is None:
        return p1
    (u1, v1), (u2, v2) = p1, p2
    if u1 == u2:
        if (v1 + v2) % P == 0:
            return None
        lam = (3 * u1 * u1 + 2 * A * u1 + 1) * pow(2 * v1, P - 2, P) % P
    else:
        lam = (v2 - v1) * pow(u2 - u1, P - 2, P) % P
    u3 = (lam * lam - A - u1 - u2) % P
    return u3, (lam * (u1 - u3) - v1) % P


def _twist_us(label, count):
    """random u whose v^2 is not a square: points of the twist, which goldilocks_x448 accepts like any other 56 bytes"""
    out, j = [], 0
    while len(out) < count:
        u = util.from_le(stream_bytes("%s/%d" % (label, j), 56)) % P
        j += 1
        if _sqrt(_rhs(u)) is None:
            out.append(u)
    return out


def corner_peers(chk, label, honest=18):
    """(peers (m,56), kinds): honest keys, the same keys plus torsion, twist points, edge and non-canonical u"""
    sk = stream_bytes(label + "/sk", honest * 56).reshape(honest, 56)
    pk = chk.x448_derive_public_key(sk)
    rows, kinds = [r for r in pk], ["honest"] * honest
    v4 = _sqrt(A - 2)
    torsion = [(0, 0)] + ([(P - 1, v4), (P - 1, P - v4)] if v4 is not None else [])
    for k, row in enumerate(pk[:3]):
        u = util.from_le(row)
        pt = (u, _sqrt(_rhs(u)))
        for t in torsion:
            s = _m_add(pt, t)
            if s is not None:
                rows.append(le(s[0])); kinds.append("torsion")
    for u in _twist_us(label + "/twist", 4):
        rows.append(le(u)); kinds.append("twist")
    for u in (0, 1, P - 1, 5):
        rows.append(le(u)); kinds.append("edge")
    for u in (P, P + 1, P + 5, 2**448 - 1):
        rows.append(le(u)); kinds.append("noncanonical")
    small = next(u for u in range(6, 1000) if _sqrt(_rhs(u)) is not None)   # a curve point small enough that u + p fits 56 bytes
    rows.append(le(small + P)); kinds.append("noncanonical")
    return np.stack(rows).astype(np.uint8), kinds


def corner_scalars(label, n):
    k = stream_bytes(label + "/k", n * 56).reshape(n, 56)
    edge = [np.zeros(56, np.uint8), np.full(56, 0xff, np.uint8), le(4 * Q), le(4 * Q + 4)]   # 4q: the comb lands on the identity
    for j, e in enumerate(edge):
        k[j::17] = e
    return k


def corner_indices(label, n, m):
    idx = (util.from_le(stream_bytes(label + "/i", 8)) % max(m, 1)) * np.ones(n, np.uint32)       # constant
    rnd = np.frombuffer(stream_bytes(label + "/r", 4 * n), np.uint32) % np.uint32(max(m, 1))
    idx[n // 4:] = rnd[n // 4:]                                                                      # random
    for j, bad in enumerate((m, m + 1000, 2**32 - 1)):                                              # out of range
        idx[5 + j::23] = bad
    return idx


def expected(chk, peers, idx, k):
    m = len(peers)
    ok = idx < m
    base = peers[np.where(ok, idx, 0)] if m else np.zeros((len(idx), 56), np.uint8)
    out, st = chk.x448(base, k)
    out[~ok] = 0
    st[~ok] = FAILURE
    return out, st


def check_set(lib, chk, peers, idx, k, label):
    h = lib.x448_peerset_create(peers)
    try:
        assert lib.x448_peerset_size(h) == len(peers)
        got, st = lib.x448_peerset(h, idx, k)
        want, wst = expected(chk, peers, idx, k)
        bad = np.nonzero((got != want).any(axis=1) | (st != wst))[0]
        assert len(bad) == 0, "%s: %d mismatches, first at %d (peer index %d)" % (label, len(bad), bad[0], idx[bad[0]])
        return h
    except BaseException:
        lib.x448_peerset_destroy(h)
        raise


def run_corners(lib, chk, n, label):
    peers, kinds = corner_peers(chk, label)
    sizes = {0: peers[:0], 1: peers[:1], 7: peers[::5][:7], len(peers): peers}
    for m, ps in sizes.items():
        k = corner_scalars("%s/%d" % (label, m), n)
        idx = corner_indices("%s/%d" % (label, m), n, m)
        lib.x448_peerset_destroy(check_set(lib, chk, ps, idx, k, "%s m=%d" % (label, m)))
    return peers, kinds


# ---- CPU tier: the device functors compiled for the host (tests/hostsim/peerset.cpp) -------------------------------------
@pytest.fixture(scope="module")
def psim():
    """the peer-set entry points on the host simulator: tests/hostsim/_hostsim_peerset.so (`make hostsim`)"""
    from libgoldilocks_b200.capi import BatchLib
    path = os.path.join(ROOT, "tests", "hostsim", "_hostsim_peerset.so")
    if not os.path.exists(path):
        subprocess.run(["make", "-C", ROOT, "hostsim"], check=True)
    return BatchLib(path)


def test_peerset_matches_x448_on_the_host_simulator(psim, chk):
    util.set_threads(psim, os.cpu_count() or 4)
    peers, kinds = run_corners(psim, chk, 200, "ps/sim")
    assert len(peers) == 40


def test_peerset_flags_route_honest_peers_to_the_comb(psim, chk):
    """the comb is not a formality: honest keys take their table, u = 0 / p - 1 / p and twist points keep the ladder"""
    import ctypes as C
    peers, kinds = corner_peers(chk, "ps/flags")
    h = psim.x448_peerset_create(peers)
    try:
        flags = np.zeros(len(peers), np.int32)
        psim.lib.hostsim_x448_peerset_flags(flags.ctypes.data_as(C.c_void_p), h)
    finally:
        psim.x448_peerset_destroy(h)
    us = [util.from_le(r) % P for r in peers]
    for u, kind, f in zip(us, kinds, flags):
        on_curve = _sqrt(_rhs(u)) not in (None, 0)
        want = SUCCESS if (on_curve and u not in (0, P - 1)) else FAILURE
        assert f == want, "u = %#x (%s): flag %d, want %d" % (u, kind, f, want)
    assert all(f == SUCCESS for f, kind in zip(flags, kinds) if kind == "honest")
    assert sum(f == FAILURE for f in flags) >= 6


def test_peerset_scalar_constant_is_eight(psim, chk):
    """X448(u, k) = encode_like_x448((k / 8) Q): checked on the base point, where the ladder's answer is also the
    Ed448 key derivation's (x448_derive_public_key halves once, the peer set three times)"""
    k = corner_scalars("ps/eight", 64)
    h = psim.x448_peerset_create(le(5)[None])
    try:
        got, st = psim.x448_peerset(h, np.zeros(64, np.uint32), k)
    finally:
        psim.x448_peerset_destroy(h)
    want = chk.x448_derive_public_key(k)
    nz = (want != 0).any(axis=1)
    assert (got[nz] == want[nz]).all() and (st[nz] == SUCCESS).all()


def test_peerset_matches_cryptography(psim, chk):
    x448 = pytest.importorskip("cryptography.hazmat.primitives.asymmetric.x448")
    from cryptography.hazmat.primitives import serialization
    raw = serialization.Encoding.Raw, serialization.PublicFormat.Raw
    peers_sk = stream_bytes("ps/crypto/sk", 8 * 56).reshape(8, 56)
    peers = chk.x448_derive_public_key(peers_sk)
    k = stream_bytes("ps/crypto/k", 24 * 56).reshape(24, 56)
    idx = np.arange(24, dtype=np.uint32) % 8
    h = psim.x448_peerset_create(peers)
    try:
        got, st = psim.x448_peerset(h, idx, k)
    finally:
        psim.x448_peerset_destroy(h)
    for i in range(24):
        priv = x448.X448PrivateKey.from_private_bytes(bytes(k[i]))
        assert priv.public_key().public_bytes(*raw) == bytes(chk.x448_derive_public_key(k[i:i + 1])[0])
        shared = priv.exchange(x448.X448PublicKey.from_public_bytes(bytes(peers[idx[i]])))
        assert bytes(got[i]) == shared and st[i] == SUCCESS


def test_peerset_kernel_passes_the_sass_audit():
    """tools/ct_audit.py on the shipped SASS audits the peer-set kernel in its group of extension kernels: no secret-dependent
    branch and no secret-dependent global / local / constant address, with the scalar secret and the peer index public"""
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ct_audit.py"), "--no-write"], capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert "extensions: all 1 secret-handling kernels PASS" in r.stdout
    assert any(line.split()[:2] == ["SlotX448Peer", "PASS"] for line in r.stdout.splitlines())


# ---- GPU tier --------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_peerset_matches_x448_on_the_gpu(gpu, chk):
    run_corners(gpu, chk, 1 << 12, "ps/gpu")


@pytest.mark.gpu
def test_peerset_million_elements_against_1024_honest_peers(gpu, chk):
    n, m = 1 << 20, 1024
    util.set_threads(chk, os.cpu_count() or 4)
    peers = chk.x448_derive_public_key(stream_bytes("ps/big/sk", m * 56).reshape(m, 56))
    k = stream_bytes("ps/big/k", n * 56).reshape(n, 56)
    idx = np.frombuffer(stream_bytes("ps/big/i", 4 * n), np.uint32) % np.uint32(m)
    gpu.x448_peerset_destroy(check_set(gpu, chk, peers, idx, k, "2^20 x 1024 peers"))


@pytest.mark.gpu
def test_peerset_dev_equals_host_call(gpu, chk):
    import torch
    from libgoldilocks_b200.engine import DeviceEngine
    eng = DeviceEngine()
    peers, _ = corner_peers(chk, "ps/dev")
    n = 5000
    k = corner_scalars("ps/dev", n)
    idx = corner_indices("ps/dev", n, len(peers))
    h = gpu.x448_peerset_create(peers)
    try:
        want, wst = gpu.x448_peerset(h, idx, k)
        out = torch.empty((n, 56), dtype=torch.uint8, device="cuda")
        st = torch.empty(n, dtype=torch.int32, device="cuda")
        eng.x448_peerset(out, st, h, torch.from_numpy(idx.view(np.int32)).cuda(), torch.from_numpy(k).cuda())
        torch.cuda.synchronize()
        assert (out.cpu().numpy() == want).all() and (st.cpu().numpy() == wst).all()
        eng.x448_peerset(out[:0], st[:0], h, torch.from_numpy(idx.view(np.int32)).cuda(), torch.from_numpy(k).cuda())   # n = 0 succeeds
    finally:
        gpu.x448_peerset_destroy(h)


@pytest.mark.gpu
def test_peerset_from_another_device_fails(gpu, chk):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    peers = chk.x448_derive_public_key(stream_bytes("ps/dev2/sk", 4 * 56).reshape(4, 56))
    k = stream_bytes("ps/dev2/k", 8 * 56).reshape(8, 56)
    prev = torch.cuda.current_device()
    torch.cuda.set_device(1)
    try:
        h = gpu.x448_peerset_create(peers)
    finally:
        torch.cuda.set_device(prev)
    try:
        with pytest.raises(RuntimeError, match="another device"):
            gpu.x448_peerset(h, np.zeros(8, np.uint32), k)
    finally:
        gpu.x448_peerset_destroy(h)


def _kernel_ms(gpu, fn, reps=5):
    """best-of-reps sum of the per-launch CUDA-event times of one call (goldilocks_b200_profile)"""
    import ctypes as C
    L = gpu.lib
    L.goldilocks_b200_profile.restype = None
    L.goldilocks_b200_profile_read.restype = C.c_size_t
    names = C.create_string_buffer(64 * 256)
    ms = (C.c_float * 256)()
    fn()
    best = None
    for _ in range(reps):
        L.goldilocks_b200_profile(C.c_int(1))
        fn()
        L.goldilocks_b200_profile(C.c_int(0))
        cnt = L.goldilocks_b200_profile_read(names, ms, C.c_size_t(256))
        t = sum(ms[j] for j in range(cnt))
        best = t if best is None else min(best, t)
    return best


@pytest.mark.gpu
def test_peerset_time_independent_of_the_scalar(gpu, chk):
    """as test_secret_paths_time_independent_of_the_scalar: all-zero, all-ones, one-bit and random scalars at 2^18 lanes take
    the same kernel time within 2 %, against one peer and against 1024 (random order)"""
    n = 1 << 18
    pats = {"zero": np.zeros((n, 56), np.uint8), "ones": np.full((n, 56), 0xff, np.uint8), "random": stream_bytes("ps/ct/r", n * 56).reshape(n, 56)}
    bit = np.zeros((n, 56), np.uint8)
    bit[:, 30] = 0x10
    pats["one_bit"] = bit
    for m in (1, 1024):
        peers = chk.x448_derive_public_key(stream_bytes("ps/ct/sk%d" % m, m * 56).reshape(m, 56))
        idx = np.frombuffer(stream_bytes("ps/ct/i", 4 * n), np.uint32) % np.uint32(m)
        h = gpu.x448_peerset_create(peers)
        try:
            times = {p: _kernel_ms(gpu, lambda s=s: gpu.x448_peerset(h, idx, s)) for p, s in pats.items()}
        finally:
            gpu.x448_peerset_destroy(h)
        lo, hi = min(times.values()), max(times.values())
        print("[ct-timing] x448_peerset m=%-5d %s  spread %.2f %%" % (m, {p: round(v, 3) for p, v in times.items()}, 100 * (hi - lo) / lo))
        assert hi <= 1.02 * lo, "m=%d: kernel time depends on the scalar pattern: %s" % (m, times)
