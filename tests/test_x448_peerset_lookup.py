"""X448 against a peer set by the peer's bytes (goldilocks_x448_peerset_lookup_batch[_dev]): every output byte and status must be
what goldilocks_x448 returns for (base i, scalar i), whether base i is in the set or not, and peer_index[i] the lowest set index
whose 56 bytes equal base i, or m.  Sets of 0, 1, 7 and all corner peers (honest, torsion, twist, edge, non-canonical) and a set
with duplicate peers; batches that mix hits on every kind with misses (fresh honest keys, twist points, u in {0, 1, p - 1}, the
u + p and u - p encodings of set members); NULL peer_index; n = 0; and batches in any order."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import util
from util import le, stream_bytes
from test_x448_peerset import P, SUCCESS, _kernel_ms, _twist_us, corner_peers, corner_scalars, expected

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def lookup_index(peers, base):
    """the lowest set index whose 56 bytes equal each base row, or m: a dict over the set's bytes"""
    first = {}
    for t, row in enumerate(peers):
        first.setdefault(bytes(row), t)
    return np.array([first.get(bytes(r), len(peers)) for r in base], np.uint32)


def lookup_batch(chk, label, peers, n):
    """n base rows: two thirds hits spread over every row of the set (each row at least once when n >= m), the rest misses --
    fresh honest keys, twist points, u in {0, 1, p - 1} and the other encoding (u + p or u - p) of every set member that has one.
    A "miss" that happens to be in the set (u = 0 in the corner set) is a hit: lookup_index decides."""
    m = len(peers)
    fresh = chk.x448_derive_public_key(stream_bytes(label + "/fresh", 8 * 56).reshape(8, 56))
    other = [le(u) for u in _twist_us(label + "/twist", 4)] + [le(u) for u in (0, 1, P - 1)]
    for row in peers:
        u = util.from_le(row)
        if u + P < 2**448:
            other.append(le(u + P))
        if u >= P:
            other.append(le(u - P))
    misses = np.concatenate([fresh, np.stack(other).astype(np.uint8)])
    sel = np.frombuffer(stream_bytes(label + "/sel", 4 * n), np.uint32).astype(np.int64)
    base = misses[sel % len(misses)].copy()
    if m:
        hit = sel % 3 != 0
        base[hit] = peers[(sel[hit] // 3) % m]
        base[:min(m, n)] = peers[:min(m, n)]
    return base


def check_lookup(lib, chk, peers, base, k, label):
    """the lookup call on a fresh set against the checker's goldilocks_x448 and the dict's indices; returns (out, status, index)"""
    h = lib.x448_peerset_create(peers)
    try:
        got, st, idx = lib.x448_peerset_lookup(h, base, k, return_index=True)
    finally:
        lib.x448_peerset_destroy(h)
    want_idx = lookup_index(peers, base)
    bad = np.nonzero(idx != want_idx)[0]
    assert len(bad) == 0, "%s: %d wrong peer indices, first at %d (%d, want %d)" % (label, len(bad), bad[0], idx[bad[0]], want_idx[bad[0]])
    want, wst = chk.x448(base, k)
    bad = np.nonzero((got != want).any(axis=1) | (st != wst))[0]
    assert len(bad) == 0, "%s: %d mismatches, first at %d (peer index %d)" % (label, len(bad), bad[0], idx[bad[0]])
    return got, st, idx


def corner_sets(chk, label):
    """the sets of the peer-set tests (0, 1, 7 and all corner peers) and one with duplicate peers"""
    peers, kinds = corner_peers(chk, label)
    dup = np.concatenate([peers[[3, 0, 3]], peers[20:26], peers[[0]], peers[20:22]]).astype(np.uint8)
    return {"m=0": peers[:0], "m=1": peers[:1], "m=7": peers[::5][:7], "all": peers, "duplicates": dup}, kinds


def run_corners(lib, chk, n, label):
    sets, kinds = corner_sets(chk, label)
    assert set(kinds) == {"honest", "torsion", "twist", "edge", "noncanonical"}
    for name, ps in sets.items():
        base = lookup_batch(chk, "%s/%s" % (label, name), ps, n)
        k = corner_scalars("%s/%s" % (label, name), n)
        _, _, idx = check_lookup(lib, chk, ps, base, k, "%s %s" % (label, name))
        if len(ps):
            assert (idx < len(ps)).sum() >= min(len(ps), n) and (idx == len(ps)).any(), name   # both paths taken
    return sets


# ---- CPU tier: the device functors compiled for the host (tests/hostsim/peerset_lookup.cpp) ------------------------------
@pytest.fixture(scope="module")
def psim():
    """the peer-set entry points and the lookup call on the host simulator: tests/hostsim/_hostsim_peerset_lookup.so (`make hostsim`)"""
    from libgoldilocks_b200.capi import BatchLib
    path = os.path.join(ROOT, "tests", "hostsim", "_hostsim_peerset_lookup.so")
    if not os.path.exists(path):
        subprocess.run(["make", "-C", ROOT, "hostsim"], check=True)
    lib = BatchLib(path)
    util.set_threads(lib, os.cpu_count() or 4)
    return lib


def test_lookup_matches_x448_on_the_host_simulator(psim, chk):
    run_corners(psim, chk, 160, "psl/sim")


def test_lookup_hits_agree_with_the_index_form(psim, chk):
    """a hit computes what the index form computes for the looked-up index; the index form's misses are its zeros"""
    sets, _ = corner_sets(chk, "psl/idx")
    peers = sets["all"]
    n = 120
    base, k = lookup_batch(chk, "psl/idx", peers, n), corner_scalars("psl/idx", n)
    h = psim.x448_peerset_create(peers)
    try:
        got, st, idx = psim.x448_peerset_lookup(h, base, k, return_index=True)
        ig, ist = psim.x448_peerset(h, idx, k)
    finally:
        psim.x448_peerset_destroy(h)
    want, wst = expected(chk, peers, idx, k)
    assert (ig == want).all() and (ist == wst).all()
    hit = idx < len(peers)
    assert hit.any() and (~hit).any()
    assert (got[hit] == ig[hit]).all() and (st[hit] == ist[hit]).all()


def test_lookup_other_encoding_of_a_set_member_misses(psim, chk):
    """u + p is the same u to goldilocks_x448 but other bytes to the lookup: it misses, takes the ladder and still gives the
    result of the member it encodes"""
    small = next(u for u in range(6, 1000) if pow((u * u * u + 156326 * u * u + u) % P, (P - 1) // 2, P) == 1)
    peers = le(small)[None]
    k = corner_scalars("psl/enc", 34)
    base = np.stack([le(small), le(small + P)] * 17).astype(np.uint8)
    got, st, idx = check_lookup(psim, chk, peers, base, k, "u + p")
    assert (idx == np.tile([0, 1], 17)).all()
    want_hit, wst_hit = chk.x448(np.repeat(le(small)[None], 34, axis=0), k)
    assert (got == want_hit).all() and (st == wst_hit).all() and (st == SUCCESS).any()


def test_lookup_without_index_and_with_n_zero(psim, chk):
    sets, _ = corner_sets(chk, "psl/null")
    peers = sets["m=7"]
    n = 40
    base, k = lookup_batch(chk, "psl/null", peers, n), corner_scalars("psl/null", n)
    h = psim.x448_peerset_create(peers)
    try:
        got, st = psim.x448_peerset_lookup(h, base, k)
        got2, st2, _ = psim.x448_peerset_lookup(h, base, k, return_index=True)
        e_out, e_st, e_idx = psim.x448_peerset_lookup(h, base[:0], k[:0], return_index=True)
    finally:
        psim.x448_peerset_destroy(h)
    assert (got == got2).all() and (st == st2).all()
    assert e_out.shape == (0, 56) and len(e_st) == 0 and len(e_idx) == 0
    h = psim.x448_peerset_create(peers[:0])   # an empty set with n = 0
    try:
        e_out, e_st = psim.x448_peerset_lookup(h, base[:0], k[:0])
    finally:
        psim.x448_peerset_destroy(h)
    assert e_out.shape == (0, 56) and len(e_st) == 0


def test_lookup_permuted_batch_gives_permuted_outputs(psim, chk):
    sets, _ = corner_sets(chk, "psl/perm")
    peers = sets["all"]
    n = 96
    base, k = lookup_batch(chk, "psl/perm", peers, n), corner_scalars("psl/perm", n)
    perm = np.argsort(np.frombuffer(stream_bytes("psl/perm/p", 4 * n), np.uint32), kind="stable")
    h = psim.x448_peerset_create(peers)
    try:
        got, st, idx = psim.x448_peerset_lookup(h, base, k, return_index=True)
        pg, pst, pidx = psim.x448_peerset_lookup(h, base[perm], k[perm], return_index=True)
    finally:
        psim.x448_peerset_destroy(h)
    assert (pg == got[perm]).all() and (pst == st[perm]).all() and (pidx == idx[perm]).all()


def test_lookup_kernel_passes_the_sass_audit():
    """tools/ct_audit.py audits the lookup kernel as its own group of extension kernels, with the scalar secret and the tables,
    flags, bytes, indices and order public; the reference group is unchanged"""
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ct_audit.py"), "--no-write"], capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert "X448 peer-set lookup extensions: all 1 secret-handling kernels PASS" in r.stdout
    assert "reference API: all 15 secret-handling kernels PASS" in r.stdout
    assert any(line.split()[:2] == ["SlotX448PeerLookup", "PASS"] for line in r.stdout.splitlines())


# ---- GPU tier --------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_lookup_matches_x448_on_the_gpu(gpu, chk):
    run_corners(gpu, chk, 1 << 12, "psl/gpu")


def honest_corpus(chk, label, n, m, miss_every=32):
    """n scalars against m honest peers in random order, every miss_every-th element (or none) a fresh key outside the set"""
    util.set_threads(chk, os.cpu_count() or 4)
    peers = chk.x448_derive_public_key(stream_bytes(label + "/sk", m * 56).reshape(m, 56))
    idx = np.frombuffer(stream_bytes(label + "/i", 4 * n), np.uint32) % np.uint32(m)
    base = peers[idx]
    if miss_every:
        q = n // miss_every
        base[::miss_every][:q] = chk.x448_derive_public_key(stream_bytes(label + "/miss", q * 56).reshape(q, 56))
    return peers, base


@pytest.mark.gpu
def test_lookup_million_elements_against_1024_peers_with_misses(gpu, chk):
    n, m = 1 << 20, 1024
    peers, base = honest_corpus(chk, "psl/big", n, m)
    k = stream_bytes("psl/big/k", n * 56).reshape(n, 56)
    _, _, idx = check_lookup(gpu, chk, peers, base, k, "2^20 x 1024 peers, 1/32 misses")
    assert (idx == m).sum() == n // 32


@pytest.mark.gpu
def test_lookup_dev_equals_host_call_on_two_streams(gpu, chk):
    import torch
    from libgoldilocks_b200.engine import DeviceEngine
    eng = DeviceEngine()
    sets, _ = corner_sets(chk, "psl/dev")
    peers = sets["all"]
    n = 5000
    base_a, k_a = lookup_batch(chk, "psl/dev/a", peers, n), corner_scalars("psl/dev/a", n)
    base_b, k_b = lookup_batch(chk, "psl/dev/b", peers, n), corner_scalars("psl/dev/b", n)
    h = gpu.x448_peerset_create(peers)
    try:
        want_a, wst_a, widx_a = gpu.x448_peerset_lookup(h, base_a, k_a, return_index=True)
        want_b, wst_b = gpu.x448_peerset_lookup(h, base_b, k_b)
        cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        db_a, dk_a, db_b, dk_b = cuda(base_a), cuda(k_a), cuda(base_b), cuda(k_b)
        nbytes = eng.x448_peerset_scratch_bytes(n)
        assert nbytes >= 20 * n
        sc_a = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        sc_b = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        out_a = torch.empty((n, 56), dtype=torch.uint8, device="cuda"); st_a = torch.empty(n, dtype=torch.int32, device="cuda")
        out_b = torch.empty((n, 56), dtype=torch.uint8, device="cuda"); st_b = torch.empty(n, dtype=torch.int32, device="cuda")
        idx_a = torch.empty(n, dtype=torch.int32, device="cuda")
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        s1.wait_stream(torch.cuda.current_stream()); s2.wait_stream(torch.cuda.current_stream())
        for _ in range(2):
            with torch.cuda.stream(s1):
                eng.x448_peerset_lookup(out_a, st_a, idx_a, h, db_a, dk_a, sc_a)
            with torch.cuda.stream(s2):
                eng.x448_peerset_lookup(out_b, st_b, None, h, db_b, dk_b, sc_b)
        torch.cuda.synchronize()
        assert (out_a.cpu().numpy() == want_a).all() and (st_a.cpu().numpy() == wst_a).all()
        assert (idx_a.cpu().numpy().view(np.uint32) == widx_a).all()
        assert (out_b.cpu().numpy() == want_b).all() and (st_b.cpu().numpy() == wst_b).all()
        eng.x448_peerset_lookup(out_a[:0], st_a[:0], None, h, db_a, dk_a, sc_a)   # n = 0 succeeds
        torch.cuda.synchronize()
    finally:
        gpu.x448_peerset_destroy(h)
    want, wst = chk.x448(base_a, k_a)
    assert (want == want_a).all() and (wst == wst_a).all()


@pytest.mark.gpu
def test_lookup_empty_set_with_n_zero(gpu, chk):
    import torch
    from libgoldilocks_b200.engine import DeviceEngine
    eng = DeviceEngine()
    h = gpu.x448_peerset_create(np.zeros((0, 56), np.uint8))
    try:
        out, st, idx = gpu.x448_peerset_lookup(h, np.zeros((0, 56), np.uint8), np.zeros((0, 56), np.uint8), return_index=True)
        assert out.shape == (0, 56) and len(st) == 0 and len(idx) == 0
        e = torch.empty((0, 56), dtype=torch.uint8, device="cuda")
        eng.x448_peerset_lookup(e, torch.empty(0, dtype=torch.int32, device="cuda"), None, h, e, e,
                                torch.empty(max(eng.x448_peerset_scratch_bytes(0), 1), dtype=torch.uint8, device="cuda"))
        torch.cuda.synchronize()
    finally:
        gpu.x448_peerset_destroy(h)


@pytest.mark.gpu
def test_lookup_from_another_device_fails(gpu, chk):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    peers = chk.x448_derive_public_key(stream_bytes("psl/dev2/sk", 4 * 56).reshape(4, 56))
    k = stream_bytes("psl/dev2/k", 8 * 56).reshape(8, 56)
    prev = torch.cuda.current_device()
    torch.cuda.set_device(1)
    try:
        h = gpu.x448_peerset_create(peers)
    finally:
        torch.cuda.set_device(prev)
    try:
        with pytest.raises(RuntimeError, match="another device"):
            gpu.x448_peerset_lookup(h, peers[np.arange(8) % 4], k)
    finally:
        gpu.x448_peerset_destroy(h)


@pytest.mark.gpu
def test_lookup_time_independent_of_the_scalar(gpu, chk):
    """as test_peerset_time_independent_of_the_scalar: all-zero, all-ones, one-bit and random scalars at 2^18 lanes take the same
    kernel time (lookup, sort and the slot kernel) within 2 %, against one peer, 1024 peers in random order, and 1024 peers with
    1/32 misses"""
    n = 1 << 18
    pats = {"zero": np.zeros((n, 56), np.uint8), "ones": np.full((n, 56), 0xff, np.uint8), "random": stream_bytes("psl/ct/r", n * 56).reshape(n, 56)}
    bit = np.zeros((n, 56), np.uint8)
    bit[:, 30] = 0x10
    pats["one_bit"] = bit
    for m, miss_every in ((1, 0), (1024, 0), (1024, 32)):
        peers, base = honest_corpus(chk, "psl/ct/%d" % m, n, m, miss_every)
        h = gpu.x448_peerset_create(peers)
        try:
            times = {p: _kernel_ms(gpu, lambda s=s: gpu.x448_peerset_lookup(h, base, s)) for p, s in pats.items()}
        finally:
            gpu.x448_peerset_destroy(h)
        lo, hi = min(times.values()), max(times.values())
        print("[ct-timing] x448_peerset_lookup m=%-5d misses 1/%s %s  spread %.2f %%" % (m, miss_every or "-", {p: round(v, 3) for p, v in times.items()},
                                                                                      100 * (hi - lo) / lo))
        assert hi <= 1.02 * lo, "m=%d: kernel time depends on the scalar pattern: %s" % (m, times)
