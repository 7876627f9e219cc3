"""Decaf peer sets (goldilocks_b200_decaf_peerset_*, goldilocks_448_direct_scalarmul_peerset_batch[_dev]): every output byte and
status must be what goldilocks_448_direct_scalarmul returns for the same (peer encoding, scalar, allow_identity, short_circuit):
valid peers, the identity, non-canonical and low-bit encodings, random strings that fail to decode, out-of-range peer indices
(which behave like 56 bytes that do not decode), edge scalars, and batches in constant, sorted, reversed and random order."""
import os
import re
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
SUCCESS, FAILURE = -1, 0
UNDECODABLE = np.full(56, 0xff, np.uint8)   # 2^448 - 1 >= p: what an out-of-range index stands for


def corner_peers(chk, label):
    """(encodings (40,56), kinds): valid encodings of random points, the identity, s >= p, the low bit set, random strings"""
    pts = util.random_points(chk, label + "/pts", 24)
    enc = chk.point_encode(pts)
    rows, kinds = [r for r in enc[:20]], ["valid"] * 20
    rows.append(np.zeros(56, np.uint8)); kinds.append("identity")
    for s in (P, P + 1, 2**448 - 1):
        rows.append(le(s)); kinds.append("noncanonical")
    for r in enc[20:24]:
        r = r.copy(); r[0] |= 1
        rows.append(r); kinds.append("lowbit")
    for r in stream_bytes(label + "/rnd", 12 * 56).reshape(12, 56):
        rows.append(r); kinds.append("random")
    return np.stack(rows).astype(np.uint8), kinds, pts[:20]


SUBSETS = {0: [], 1: [0], 7: [0, 20, 21, 24, 25, 28, 35]}   # the 7-peer set mixes every kind


def corner_scalars(chk, label, n):
    s = util.random_scalars(chk, label + "/k", n)
    e = util.scalar_edge_bytes()
    for j, row in enumerate(e):
        s[j::29] = row
    return s


def corner_indices(label, n, m):
    """constant, sorted, reversed and random quarters, with out-of-range indices m, m + 1000 and 2^32 - 1 throughout"""
    mm = max(m, 1)
    q = n // 4
    idx = np.empty(n, np.uint32)
    idx[:q] = util.from_le(stream_bytes(label + "/c", 8)) % mm
    idx[q:2 * q] = np.sort(np.frombuffer(stream_bytes(label + "/s", 4 * q), np.uint32) % np.uint32(mm))
    idx[2 * q:3 * q] = np.sort(np.frombuffer(stream_bytes(label + "/v", 4 * q), np.uint32) % np.uint32(mm))[::-1]
    idx[3 * q:] = np.frombuffer(stream_bytes(label + "/r", 4 * (n - 3 * q)), np.uint32) % np.uint32(mm)
    for j, bad in enumerate((m, m + 1000, 2**32 - 1)):
        idx[7 + j::31] = bad
    return idx


def expected(ref_lib, peers, idx, sc, allow, short, prefill=0xa5):
    """goldilocks_448_direct_scalarmul_batch of `ref_lib` on peers[idx], 0xff * 56 standing in for idx >= m"""
    ext = np.concatenate([peers.reshape(-1, 56), UNDECODABLE[None]])
    base = ext[np.minimum(idx, len(peers)).astype(np.int64)]
    return ref_lib.direct_scalarmul(base, sc, allow, short, prefill=prefill)


def check_set(lib, ref_lib, chk, peers, kinds, pts, idx, sc, allow, label):
    """one set, both short_circuit settings: bytes and statuses against ref_lib's direct_scalarmul, valid peers against the
    checker's encode(scalarmul), and against the original reference build where it is present"""
    h = lib.decaf_peerset_create(peers, allow)
    try:
        assert lib.decaf_peerset_size(h) == len(peers)
        for short in (False, True):
            got, st = lib.decaf_peerset(h, idx, sc, short, prefill=0xa5)
            want, wst = expected(ref_lib, peers, idx, sc, allow, short)
            bad = np.nonzero((got != want).any(axis=1) | (st != wst))[0]
            assert len(bad) == 0, "%s allow=%s short=%s: %d mismatches, first at %d (peer index %d)" % (label, allow, short, len(bad), bad[0], idx[bad[0]])
            if chk.has("goldilocks_448_direct_scalarmul_batch"):
                r, rst = expected(chk, peers, idx, sc, allow, short)
                assert (got == r).all() and (st == rst).all(), "%s: differs from the reference build" % label
            valid = np.array([i < len(peers) and kinds[i] == "valid" for i in idx])
            if valid.any():
                w = chk.point_encode(chk.point_scalarmul(pts[idx[valid].astype(np.int64)], sc[valid]))
                assert (got[valid] == w).all() and (st[valid] == SUCCESS).all(), "%s: valid peers vs encode(scalarmul)" % label
    finally:
        lib.decaf_peerset_destroy(h)


def run_corners(lib, ref_lib, chk, n, label):
    peers, kinds, pts = corner_peers(chk, label)
    sets = dict(SUBSETS)
    sets[len(peers)] = list(range(len(peers)))
    for m, rows in sets.items():
        rows = np.array(rows, np.int64)
        ps, ks = peers[rows] if m else peers[:0], [kinds[r] for r in rows]
        pp = np.zeros((m, 256), np.uint8)
        for j, r in enumerate(rows):
            if kinds[r] == "valid":
                pp[j] = pts[r]
        sc = corner_scalars(chk, "%s/%d" % (label, m), n)
        idx = corner_indices("%s/%d" % (label, m), n, m)
        for allow in (False, True):
            check_set(lib, ref_lib, chk, ps, ks, pp, idx, sc, allow, "%s m=%d" % (label, m))
    return peers, kinds


# ---- the math: the comb multiplies by the same integer as the signed-window multiplication -------------------------------
def _adj_from_source():
    with open(os.path.join(ROOT, "libgoldilocks_b200", "csrc", "consts.cuh")) as f:
        words = re.search(r"GOLD_CONST_SC_ADJ \{([^}]*)\}", f.read()).group(1).split(",")
    return sum(int(w.strip().rstrip("u"), 16) << (32 * j) for j, w in enumerate(words))


def _window_multiplier(s1x):
    """s_window_mainloop: 90 signed 5-bit digits 2b - 31 of s1x (s_window_digit) times 32^k"""
    return sum((2 * ((s1x >> (5 * k)) & 31) - 31) * 32**k for k in range(90))


def _comb_multiplier(s1x):
    """s_comb_scalarmul_table: each of the 5 x 5 x 18 teeth adds +2^pos (bit set) or -2^pos; positions >= 446 read 0"""
    total = 0
    for i in range(18):
        for j in range(5):
            for k in range(5):
                pos = i + 18 * (k + 5 * j)
                bit = (s1x >> pos) & 1 if pos < 446 else 0
                total += (2 * bit - 1) << pos
    return total


def test_comb_and_window_multiply_by_the_same_integer(chk):
    """Both kernels recode the scalar with sc_recode_signed, s' = (s + adj) / 2 mod q with adj = (2^450 - 1) mod q, and add up
    signed digits that cover the same 450 bit positions.  So both multiply the point by the same integer 2 s' - (2^450 - 1),
    congruent to s mod q: no torsion difference arises for the decaf encoding to remove, whatever the point's 4-torsion part."""
    adj = _adj_from_source()
    assert adj == (2**450 - 1) % Q
    inv2 = pow(2, -1, Q)
    scalars = [util.from_le(r) for r in util.scalar_edge_bytes()] + [util.from_le(r) for r in util.random_scalars(chk, "dps/int", 64)]
    for s in scalars + [0, 1, Q - 1]:
        s1x = (s + adj) * inv2 % Q
        mw, mc = _window_multiplier(s1x), _comb_multiplier(s1x)
        assert mw == mc == 2 * s1x - (2**450 - 1)
        assert mc % Q == s % Q


# ---- CPU tier: the device functors compiled for the host (tests/hostsim/decaf_peerset.cpp) -------------------------------------
@pytest.fixture(scope="module")
def psim():
    """the decaf peer-set entry points on the host simulator: tests/hostsim/_hostsim_decaf_peerset.so (`make hostsim`)"""
    from libgoldilocks_b200.capi import BatchLib
    path = os.path.join(ROOT, "tests", "hostsim", "_hostsim_decaf_peerset.so")
    if not os.path.exists(path):
        subprocess.run(["make", "-C", ROOT, "hostsim"], check=True)
    lib = BatchLib(path)
    util.set_threads(lib, os.cpu_count() or 4)
    return lib


def test_decaf_peerset_matches_direct_scalarmul_on_the_host_simulator(psim, sim, chk):
    util.set_threads(sim, os.cpu_count() or 4)
    peers, kinds = run_corners(psim, sim, chk, 400, "dps/sim")
    assert len(peers) == 40


def test_decaf_peerset_edge_scalars_against_every_peer_kind(psim, sim, chk):
    """every edge scalar (0, 1, q - 1, the recoding's carry points, ...) against every one of the 40 peers"""
    peers, kinds, pts = corner_peers(chk, "dps/edge")
    e = util.scalar_edge_bytes()
    idx = np.repeat(np.arange(len(peers), dtype=np.uint32), len(e))
    sc = np.tile(e, (len(peers), 1))
    pp = np.zeros((len(peers), 256), np.uint8)
    pp[:20] = pts
    for allow in (False, True):
        check_set(psim, sim, chk, peers, kinds, pp, idx, sc, allow, "edge scalars")


def test_decaf_peerset_flags(psim, chk):
    """the per-peer statuses are the decoder's under the set's allow_identity, and the extra entry m is FAILURE"""
    import ctypes as C
    peers, kinds, _ = corner_peers(chk, "dps/flags")
    for allow in (False, True):
        h = psim.decaf_peerset_create(peers, allow)
        try:
            flags = np.zeros(len(peers) + 1, np.int32)
            psim.lib.hostsim_decaf_peerset_flags(flags.ctypes.data_as(C.c_void_p), h)
        finally:
            psim.decaf_peerset_destroy(h)
        _, want = chk.point_decode(peers, allow)
        assert (flags[:-1] == want).all() and flags[-1] == FAILURE
        by_kind = {k: {int(f) for f, kk in zip(flags, kinds) if kk == k} for k in set(kinds)}
        assert by_kind["valid"] == {SUCCESS} and by_kind["noncanonical"] == {FAILURE} and by_kind["lowbit"] == {FAILURE}
        assert by_kind["identity"] == {SUCCESS if allow else FAILURE}
        assert FAILURE in by_kind["random"]


def test_decaf_peerset_order_does_not_change_the_results(psim, chk):
    """the call sorts by peer internally: a shuffled batch gives the shuffled results of the sorted one"""
    peers, _, _ = corner_peers(chk, "dps/perm")
    n = 96
    idx = np.sort(np.frombuffer(stream_bytes("dps/perm/i", 4 * n), np.uint32) % np.uint32(len(peers) + 2))
    sc = corner_scalars(chk, "dps/perm", n)
    perm = np.random.default_rng(7).permutation(n)
    h = psim.decaf_peerset_create(peers, True)
    try:
        a, sa = psim.decaf_peerset(h, idx, sc, True, prefill=0xa5)
        b, sb = psim.decaf_peerset(h, idx[perm], sc[perm], True, prefill=0xa5)
        assert (a[perm] == b).all() and (sa[perm] == sb).all()
        z, sz = psim.decaf_peerset(h, idx[:0], sc[:0])   # n = 0
        assert z.shape == (0, 56) and sz.shape == (0,)
    finally:
        psim.decaf_peerset_destroy(h)


def test_decaf_peerset_kernel_passes_the_sass_audit():
    """tools/ct_audit.py on the shipped SASS audits SlotDecafPeer as an extension kernel: no secret-dependent branch and no
    secret-dependent global / local / constant address, with the scalars secret and the set, indices and order public"""
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ct_audit.py"), "--no-write", "--only", "SlotDecafPeer"],
                       capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert any(line.split()[:2] == ["SlotDecafPeer", "PASS"] for line in r.stdout.splitlines())


# ---- GPU tier --------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_decaf_peerset_matches_direct_scalarmul_on_the_gpu(gpu, chk):
    util.set_threads(chk, os.cpu_count() or 4)
    run_corners(gpu, gpu, chk, 1 << 12, "dps/gpu")


@pytest.mark.gpu
def test_decaf_peerset_million_scalars_against_1024_peers(gpu, chk):
    """2^20 scalars against 1024 peers (valid, plus every fourth one a string that fails to decode) in random order"""
    n, m = 1 << 20, 1024
    peers = chk.point_encode(util.random_points(chk, "dps/big/p", m))
    peers[::4] = stream_bytes("dps/big/bad", (m // 4) * 56).reshape(m // 4, 56)
    sc = gpu.scalar_decode_long(stream_bytes("dps/big/k", n * 56).reshape(n, 56), 56)
    idx = np.frombuffer(stream_bytes("dps/big/i", 4 * n), np.uint32) % np.uint32(m + 8)   # a few out of range
    h = gpu.decaf_peerset_create(peers, False)
    try:
        for short in (False, True):
            got, st = gpu.decaf_peerset(h, idx, sc, short, prefill=0xa5)
            want, wst = expected(gpu, peers, idx, sc, False, short)
            assert (got == want).all() and (st == wst).all()
            assert (st == FAILURE).sum() > n // 8
    finally:
        gpu.decaf_peerset_destroy(h)


@pytest.mark.gpu
def test_decaf_peerset_sorted_and_shuffled_batches_agree(gpu, chk):
    n, m = 1 << 16, 300
    peers = chk.point_encode(util.random_points(chk, "dps/shuf/p", m))
    sc = gpu.scalar_decode_long(stream_bytes("dps/shuf/k", n * 56).reshape(n, 56), 56)
    idx = np.sort(np.frombuffer(stream_bytes("dps/shuf/i", 4 * n), np.uint32) % np.uint32(m))
    perm = np.random.default_rng(11).permutation(n)
    h = gpu.decaf_peerset_create(peers, False)
    try:
        a, sa = gpu.decaf_peerset(h, idx, sc)
        b, sb = gpu.decaf_peerset(h, idx[perm], sc[perm])
    finally:
        gpu.decaf_peerset_destroy(h)
    assert (a[perm] == b).all() and (sa[perm] == sb).all()


@pytest.mark.gpu
def test_decaf_peerset_dev_equals_host_call(gpu, chk):
    import torch
    from libgoldilocks_b200.engine import DeviceEngine
    eng = DeviceEngine()
    peers, _, _ = corner_peers(chk, "dps/dev")
    n = 5000
    sc = corner_scalars(chk, "dps/dev", n)
    idx = corner_indices("dps/dev", n, len(peers))
    h = gpu.decaf_peerset_create(peers, True)
    try:
        scratch = torch.empty(eng.decaf_peerset_scratch_bytes(n), dtype=torch.uint8, device="cuda")
        d_idx, d_sc = torch.from_numpy(idx.view(np.int32)).cuda(), torch.from_numpy(sc).cuda()
        for short in (False, True):
            want, wst = gpu.decaf_peerset(h, idx, sc, short, prefill=0xa5)
            out = torch.full((n, 56), 0xa5, dtype=torch.uint8, device="cuda")
            st = torch.empty(n, dtype=torch.int32, device="cuda")
            eng.decaf_peerset(out, st, h, d_idx, d_sc, scratch, short)
            torch.cuda.synchronize()
            assert (out.cpu().numpy() == want).all() and (st.cpu().numpy() == wst).all()
        eng.decaf_peerset(out[:0], st[:0], h, d_idx, d_sc, scratch)   # n = 0 succeeds
    finally:
        gpu.decaf_peerset_destroy(h)


@pytest.mark.gpu
def test_decaf_peerset_from_another_device_fails(gpu, chk):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    peers = chk.point_encode(util.random_points(chk, "dps/dev2/p", 4))
    sc = util.random_scalars(chk, "dps/dev2/k", 8)
    prev = torch.cuda.current_device()
    torch.cuda.set_device(1)
    try:
        h = gpu.decaf_peerset_create(peers)
    finally:
        torch.cuda.set_device(prev)
    try:
        with pytest.raises(RuntimeError, match="another device"):
            gpu.decaf_peerset(h, np.zeros(8, np.uint32), sc)
    finally:
        gpu.decaf_peerset_destroy(h)


def _kernel_ms(gpu, fn, name, reps=5):
    """best-of-reps CUDA-event time of the launches of one call whose name contains `name` (goldilocks_b200_profile)"""
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
        t = sum(ms[j] for j in range(cnt) if name in names.raw[64 * j:64 * (j + 1)].split(b"\0")[0].decode())
        best = t if best is None else min(best, t)
    return best


@pytest.mark.gpu
def test_decaf_peerset_time_independent_of_the_scalar(gpu, chk):
    """as test_peerset_time_independent_of_the_scalar: zero, q - 1, one-bit and random scalars at 2^18 lanes take the same
    comb-kernel time within 2 %, against one peer and against 1024 (random order)"""
    n = 1 << 18
    one_bit = np.zeros((n, 56), np.uint8)
    one_bit[:, 30] = 0x10
    pats = {"zero": np.zeros((n, 56), np.uint8), "q-1": np.tile(le(Q - 1), (n, 1)), "one_bit": one_bit,
            "random": gpu.scalar_decode_long(stream_bytes("dps/ct/r", n * 56).reshape(n, 56), 56)}
    for m in (1, 1024):
        peers = chk.point_encode(util.random_points(chk, "dps/ct/p%d" % m, m))
        idx = np.frombuffer(stream_bytes("dps/ct/i", 4 * n), np.uint32) % np.uint32(m)
        h = gpu.decaf_peerset_create(peers)
        try:
            times = {p: _kernel_ms(gpu, lambda s=s: gpu.decaf_peerset(h, idx, s), "SlotDecafPeer") for p, s in pats.items()}
        finally:
            gpu.decaf_peerset_destroy(h)
        lo, hi = min(times.values()), max(times.values())
        print("[ct-timing] decaf_peerset m=%-5d %s  spread %.2f %%" % (m, {p: round(v, 3) for p, v in times.items()}, 100 * (hi - lo) / lo))
        assert hi <= 1.02 * lo, "m=%d: kernel time depends on the scalar pattern: %s" % (m, times)
