"""Verification by public-key bytes against a key set (goldilocks_ed448_verify_keyset_lookup_batch[_dev]): every status must be
what goldilocks_ed448_verify returns for (signature i, pubkey i, message i), whether key i is in the set or not, and key_index[i]
the lowest set index whose 57 bytes equal key i, or m.  Sets of 0, 1, 7 and 40 keys in both table layouts, with duplicate keys, a
key that does not decode (y = 1) and random bytes; batches that mix hits, misses, near misses (a set key with byte 0 or the sign
bit changed) and corrupted R, S and messages under hit keys; prehashed with a 255-byte context; fewer than 64 misses (stand-alone
miss path) and 64 or more with repeated unknown keys (grouped miss path); n = 0; and batches in any order."""
import os

import numpy as np
import pytest

import util
from util import stream_bytes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEFAULT_POLICY = 32 << 30     # goldilocks_b200_keyset_policy's default: sets of 2^16 keys are flat
N_SIGNERS = 48                # signers 0..34 can be in a set, 35..47 never are


def signers(chk, label):
    sk = stream_bytes(label + "/sk", N_SIGNERS * 57).reshape(N_SIGNERS, 57)
    return sk, chk.ed448_derive_public_key(sk)


def key_set(pk, label, m):
    """m keys: signer keys, duplicates, y = 1 (does not decode) and random bytes mixed in"""
    y1 = util.le(1, 57)[None]
    junk = stream_bytes(label + "/junk", 2 * 57).reshape(2, 57)
    if m == 0:
        return np.zeros((0, 57), np.uint8)
    if m == 1:
        return pk[:1].copy()
    if m == 7:
        return np.concatenate([pk[[0, 1]], pk[[0]], y1, junk[:1], pk[[2, 3]]]).astype(np.uint8)
    assert m == 40
    return np.concatenate([pk[:32], pk[[5]], y1, pk[[0]], junk, pk[32:35]]).astype(np.uint8)


def batch(chk, label, keys, sk, pk, n, prehashed=False, context=b""):
    """(sig, pubkey, msgs): signatures by random signers, then misuse threaded through: keys of the set that are not signer keys
    (y = 1, random bytes), near misses of set keys, and corrupted R, S and messages"""
    who = stream_bytes(label + "/who", n).astype(np.int64) % N_SIGNERS
    lens = stream_bytes(label + "/len", n).astype(np.int64) % 80
    blob = stream_bytes(label + "/msg", int(lens.sum()) + 1)
    offs = np.concatenate([[0], np.cumsum(lens)])
    msgs = [bytes(blob[offs[i]:offs[i + 1]]) for i in range(n)]
    sig = chk.ed448_sign(sk[who], pk[who], msgs, prehashed=prehashed, context=context)
    pub = pk[who].copy()
    sel = stream_bytes(label + "/sel", n)
    for i in range(n):
        kind = i % 11
        if kind == 1 and len(keys):
            pub[i] = keys[sel[i] % len(keys)]              # any key of the set, decodable or not: a hit
        elif kind == 3:
            pub[i, 0] ^= 1 << (sel[i] & 7)                 # near miss: byte 0
        elif kind == 5:
            pub[i, 56] ^= 0x80                             # near miss: the sign bit
        elif kind == 7:
            sig[i, sel[i] % 57] ^= 1 << (sel[i] & 7)       # R
        elif kind == 8:
            sig[i, 57 + sel[i] % 56] ^= 1 << (sel[i] & 7)  # S
        elif kind == 9:
            m = bytearray(msgs[i]) or bytearray(b"\0")
            m[sel[i] % len(m)] ^= 1
            msgs[i] = bytes(m)
    return sig, pub, msgs


def index_reference(keys, pub):
    lowest = {}
    for j in range(len(keys) - 1, -1, -1):
        lowest[keys[j].tobytes()] = j
    return np.array([lowest.get(p.tobytes(), len(keys)) for p in pub], np.uint32)


def check(lib, chk, keys, sig, pub, msgs, label, prehashed=False, context=b""):
    h = lib.keyset_create(keys)
    try:
        st, idx = lib.ed448_verify_keyset_lookup(h, sig, pub, msgs, prehashed=prehashed, context=context, return_index=True)
    finally:
        lib.keyset_destroy(h)
    want = chk.ed448_verify(sig, pub, msgs, prehashed=prehashed, context=context)
    bad = np.nonzero(st != want)[0]
    assert len(bad) == 0, "%s: %d statuses differ, first at %d" % (label, len(bad), bad[0])
    ref_idx = index_reference(keys, pub)
    assert (idx == ref_idx).all(), "%s: key_index differs" % label
    return st, idx


def run_cases(lib, chk, n, label, layout):
    sk, pk = signers(chk, label)
    for m in (0, 1, 7, 40):
        keys = key_set(pk, label, m)
        sig, pub, msgs = batch(chk, "%s/%d" % (label, m), keys, sk, pk, n)
        st, idx = check(lib, chk, keys, sig, pub, msgs, "%s m=%d %s" % (label, m, layout))
        hits = idx < m
        if m == 40:
            assert hits.any() and (~hits).sum() >= 64, "the case must take both paths, the misses grouped"
            assert (st[hits] == -1).any() and (st[hits] == 0).any() and (st[~hits] == -1).any()


# ---- CPU tier: the device functors compiled for the host (tests/hostsim/keyset_lookup.cpp) --------------------------------------
@pytest.fixture(scope="module")
def ksim():
    """the lookup call on the host simulator: tests/hostsim/_hostsim_keyset_lookup.so (`make hostsim`)"""
    from libgoldilocks_b200.capi import BatchLib
    path = os.path.join(ROOT, "tests", "hostsim", "_hostsim_keyset_lookup.so")
    if not os.path.exists(path):
        pytest.skip("tests/hostsim/_hostsim_keyset_lookup.so is not built (make hostsim)")
    return BatchLib(path)


@pytest.fixture(params=["flat", "compact"])
def layout(request, ksim):
    ksim.keyset_policy(DEFAULT_POLICY if request.param == "flat" else 0)
    yield request.param
    ksim.keyset_policy(DEFAULT_POLICY)


@pytest.fixture
def threads(ksim, chk):
    util.set_threads(ksim, os.cpu_count() or 4)
    util.set_threads(chk, os.cpu_count() or 4)


def test_lookup_matches_verify_on_the_host_simulator(ksim, chk, layout, threads):
    run_cases(ksim, chk, 320, "ksl/sim", layout)


def test_lookup_prehashed_with_long_context(ksim, chk, layout, threads):
    sk, pk = signers(chk, "ksl/ph")
    keys = key_set(pk, "ksl/ph", 40)
    ctx = bytes(stream_bytes("ksl/ph/ctx", 255))
    sig, pub, msgs = batch(chk, "ksl/ph", keys, sk, pk, 200, prehashed=True, context=ctx)
    st, _ = check(ksim, chk, keys, sig, pub, msgs, "prehashed " + layout, prehashed=True, context=ctx)
    assert (st == -1).any()


def test_lookup_few_misses_and_empty_batch(ksim, chk, layout, threads):
    """fewer than 64 misses: the stand-alone miss path; n = 0 succeeds"""
    sk, pk = signers(chk, "ksl/few")
    keys = key_set(pk, "ksl/few", 7)
    sig, pub, msgs = batch(chk, "ksl/few", keys, sk, pk, 40)
    _, idx = check(ksim, chk, keys, sig, pub, msgs, "n=40 " + layout)
    assert 0 < (idx == 7).sum() < 64
    h = ksim.keyset_create(keys)
    try:
        st, idx = ksim.ed448_verify_keyset_lookup(h, sig[:0], pub[:0], [], return_index=True)
        assert st.shape == (0,) and idx.shape == (0,)
    finally:
        ksim.keyset_destroy(h)


def test_lookup_order_does_not_change_the_results(ksim, chk, layout, threads):
    sk, pk = signers(chk, "ksl/perm")
    keys = key_set(pk, "ksl/perm", 40)
    sig, pub, msgs = batch(chk, "ksl/perm", keys, sk, pk, 160)
    perm = np.random.default_rng(5).permutation(len(sig))
    h = ksim.keyset_create(keys)
    try:
        a, ia = ksim.ed448_verify_keyset_lookup(h, sig, pub, msgs, return_index=True)
        b, ib = ksim.ed448_verify_keyset_lookup(h, sig[perm], pub[perm], [msgs[i] for i in perm], return_index=True)
    finally:
        ksim.keyset_destroy(h)
    assert (a[perm] == b).all() and (ia[perm] == ib).all()


# ---- GPU tier --------------------------------------------------------------------------------------------------------------
@pytest.fixture(params=["flat", "compact"])
def gpu_layout(request, gpu):
    gpu.keyset_policy(DEFAULT_POLICY if request.param == "flat" else 0)
    yield request.param
    gpu.keyset_policy(DEFAULT_POLICY)


@pytest.mark.gpu
def test_lookup_matches_verify_on_the_gpu(gpu, chk, gpu_layout):
    util.set_threads(chk, os.cpu_count() or 4)
    run_cases(gpu, chk, 1 << 12, "ksl/gpu", gpu_layout)
    sk, pk = signers(chk, "ksl/gpu/ph")
    keys = key_set(pk, "ksl/gpu/ph", 40)
    ctx = bytes(stream_bytes("ksl/gpu/ph/ctx", 255))
    sig, pub, msgs = batch(chk, "ksl/gpu/ph", keys, sk, pk, 1 << 12, prehashed=True, context=ctx)
    check(gpu, chk, keys, sig, pub, msgs, "prehashed " + gpu_layout, prehashed=True, context=ctx)
    sig, pub, msgs = batch(chk, "ksl/gpu/few", keys, sk, pk, 40)
    check(gpu, chk, keys, sig, pub, msgs, "n=40 " + gpu_layout)


@pytest.mark.gpu
def test_lookup_bench_corpus_in_any_order(gpu, gpu_layout):
    """the benchmark's shape: 2^20 signatures by the reference under 2^16 keys x 16, one in eight corrupted, the 2^16 intact keys as
    the set.  The statuses are goldilocks_ed448_verify_batch's, i.e. the corpus' own expectations, in corpus order and shuffled."""
    import bench
    n = 1 << 20
    signer, _ = bench.reference_signer()
    sig, pk, arena, off, expect = bench.make_corpus(signer, n, "ksl/bench")
    keys = pk[1::16].copy()
    want = gpu.ed448_verify(sig, pk, (arena, off))
    assert (want == expect).all()
    h = gpu.keyset_create(keys)
    try:
        st, idx = gpu.ed448_verify_keyset_lookup(h, sig, pk, (arena, off), return_index=True)
        assert (st == expect).all()
        assert (idx == index_reference(keys, pk)).all()
        perm = np.random.default_rng(3).permutation(n)
        lens = (off[1:] - off[:-1])[perm]
        off_p = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
        arena_p = np.concatenate([arena[int(off[i]):int(off[i + 1])] for i in perm] + [np.zeros(1, np.uint8)])
        st_p = gpu.ed448_verify_keyset_lookup(h, sig[perm], pk[perm], (arena_p, off_p))
        assert (st_p == expect[perm]).all()
    finally:
        gpu.keyset_destroy(h)


def _dev(a, dtype=None):
    import torch
    return torch.from_numpy(np.array(a if dtype is None else a.view(dtype))).cuda()


@pytest.mark.gpu
def test_lookup_dev_forms_equal_host_calls(gpu, chk, gpu_layout):
    import torch
    from libgoldilocks_b200.capi import pack_messages
    from libgoldilocks_b200.engine import DeviceEngine
    eng = DeviceEngine()
    sk, pk = signers(chk, "ksl/dev")
    keys = key_set(pk, "ksl/dev", 40)
    n = 3000
    ctx = bytes(stream_bytes("ksl/dev/ctx", 17))
    sig, pub, msgs = batch(chk, "ksl/dev", keys, sk, pk, n, context=ctx)
    arena, off = pack_messages(msgs)
    h = gpu.keyset_create(keys)
    try:
        want, want_idx = gpu.ed448_verify_keyset_lookup(h, sig, pub, (arena, off), context=ctx, return_index=True)
        scratch = torch.empty(eng.keyset_scratch_bytes(n, int(off[-1])), dtype=torch.uint8, device="cuda")
        d_sig, d_pk, d_msg, d_off, d_ctx = _dev(sig), _dev(pub), _dev(arena), _dev(off, np.int64), _dev(np.frombuffer(ctx, np.uint8))
        st = torch.full((n,), 7, dtype=torch.int32, device="cuda")
        d_idx = torch.full((n,), 7, dtype=torch.int32, device="cuda")
        eng.ed448_verify_keyset_lookup(st, d_idx, h, d_sig, d_pk, d_msg, d_off, scratch, ctx=d_ctx, ctx_len=len(ctx))
        torch.cuda.synchronize()
        assert (st.cpu().numpy() == want).all()
        assert (d_idx.cpu().numpy().view(np.uint32) == want_idx).all()
        st.fill_(7)
        eng.ed448_verify_keyset_lookup(st, None, h, d_sig, d_pk, d_msg, d_off, scratch, ctx=d_ctx, ctx_len=len(ctx))
        torch.cuda.synchronize()
        assert (st.cpu().numpy() == want).all()
        # the index form: device-resident against goldilocks_ed448_verify_keyset_batch
        want_ks = gpu.ed448_verify_keyset(h, want_idx, sig, (arena, off), context=ctx)
        st.fill_(7)
        eng.ed448_verify_keyset(st, h, _dev(want_idx, np.int32), d_sig, d_msg, d_off, scratch, ctx=d_ctx, ctx_len=len(ctx))
        torch.cuda.synchronize()
        assert (st.cpu().numpy() == want_ks).all()
        assert (want_ks[want_idx < len(keys)] == want[want_idx < len(keys)]).all()
        eng.ed448_verify_keyset_lookup(st[:0], None, h, d_sig, d_pk, d_msg, d_off, scratch)   # n = 0 succeeds
        eng.ed448_verify_keyset(st[:0], h, d_idx, d_sig, d_msg, d_off, scratch)
    finally:
        gpu.keyset_destroy(h)


@pytest.mark.gpu
def test_lookup_empty_set_is_verify_batch(gpu, chk, gpu_layout):
    sk, pk = signers(chk, "ksl/empty")
    sig, pub, msgs = batch(chk, "ksl/empty", pk[:0], sk, pk, 700)
    h = gpu.keyset_create(np.zeros((0, 57), np.uint8))
    try:
        st, idx = gpu.ed448_verify_keyset_lookup(h, sig, pub, msgs, return_index=True)
        assert (st == gpu.ed448_verify(sig, pub, msgs)).all() and (idx == 0).all()
        st, idx = gpu.ed448_verify_keyset_lookup(h, sig[:0], pub[:0], [], return_index=True)
        assert st.shape == (0,)
    finally:
        gpu.keyset_destroy(h)


@pytest.mark.gpu
def test_lookup_from_another_device_fails(gpu, chk):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    sk, pk = signers(chk, "ksl/dev2")
    sig, pub, msgs = batch(chk, "ksl/dev2", pk[:4], sk, pk, 8)
    prev = torch.cuda.current_device()
    torch.cuda.set_device(1)
    try:
        h = gpu.keyset_create(pk[:4])
    finally:
        torch.cuda.set_device(prev)
    try:
        with pytest.raises(RuntimeError, match="another device"):
            gpu.ed448_verify_keyset_lookup(h, sig, pub, msgs)
    finally:
        gpu.keyset_destroy(h)
