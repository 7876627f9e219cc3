"""GPU tier: the product library (libgoldilocks_b200.so, through its C ABI) against the checker,
the reference's golden vectors, and size-independent properties at BASELINE.json's full 2^20 sizes."""
import os

import numpy as np
import pytest

import parity
import util
from util import ROOT, stream_bytes

pytestmark = pytest.mark.gpu
FULL = 1 << 20


@pytest.fixture(scope="module", autouse=True)
def _threads(chk):
    util.set_threads(chk, os.cpu_count() or 1)


def test_tables(gpu, chk):
    parity.check_tables(gpu, chk)


def test_field_full(gpu, chk):
    """config 1: 2^20 random + edge pairs, bit-exact against the checker"""
    parity.check_field(gpu, chk, FULL)
    parity.check_field_isr(gpu, chk, 1 << 14)


def test_points_edge_and_glue(gpu, chk):
    """identity / mixed representatives, negate, eq, valid (the 2^20 coordinate comparison is test_points_all_2_20)"""
    parity.check_points(gpu, chk, 1 << 14)


def test_niels_mixed_additions(gpu, chk):
    """row a9 directly (goldilocks.c:271-380): all four coordinates of every mixed addition / conversion, by value and on the slot
    machine, against the reference's formulas restated on integers, and as group elements against its exported point_add / point_sub"""
    parity.check_niels(gpu, chk, 5000)


def test_codec_elligator(gpu, chk):
    parity.check_codec(gpu, chk, 1 << 14)
    parity.check_elligator_inverse(gpu, chk, 1 << 12)


def test_scalars(gpu, chk):
    parity.check_scalars(gpu, chk, 1 << 16)


def test_comb(gpu, chk):
    parity.check_comb(gpu, chk, 1 << 14)


def test_scalarmul(gpu, chk):
    parity.check_scalarmul(gpu, chk, 1 << 11)


def test_widened(gpu, chk):
    parity.check_widened(gpu, chk, 1 << 10)


def test_x448(gpu, chk, vectors):
    parity.check_x448(gpu, chk, 1 << 12)
    parity.check_x448_vectors(gpu, vectors, iters=1000)


def test_eddsa_vectors(gpu, vectors):
    parity.check_eddsa_vectors(gpu, vectors)


def test_openssl_golden(gpu):
    parity.check_openssl_golden(gpu, util.openssl_golden())


def test_eddsa_random(gpu, chk):
    parity.check_eddsa_random(gpu, chk, 1 << 12)


def test_eddsa_repeated_keys(gpu, chk):
    """per-key tables (device-side key grouping): mixed multiplicities, more groups than tables (all pairs: the
    table budget of n/4 + 1 overflows and the rest must fall back to stand-alone verification), one key for the
    whole batch, and a batch just at the grouping threshold"""
    parity.check_eddsa_grouped(gpu, chk, 1 << 12)
    parity.check_eddsa_grouped(gpu, chk, 1 << 11, label="c4g/pairs", per_key=(2,))
    parity.check_eddsa_grouped(gpu, chk, 44 * 40, label="c4g/44", per_key=(44,))            # 30 columns x 3 rows (slot_algos.cuh vsh_pick)
    parity.check_eddsa_grouped(gpu, chk, 3000, label="c4g/one-signer", per_key=(3000,))    # 90 columns, no doublings
    parity.check_eddsa_grouped(gpu, chk, 1 << 10, label="c4g/one", per_key=(3, 1 << 10))
    parity.check_eddsa_grouped(gpu, chk, 64, label="c4g/min", per_key=(4, 1, 9))
    parity.check_eddsa_grouped(gpu, chk, 512, label="c4g/ctx", prehashed=True, context=b"\x01" * 255)
    parity.check_eddsa_grouped(gpu, chk, 300, label="c4g/ctx2", context=b"repeated keys")


def test_eddsa_keyset(gpu, chk):
    """per-key tables that outlive a call (goldilocks_b200_keyset_*)"""
    parity.check_eddsa_keyset(gpu, chk, 1 << 12)
    parity.check_eddsa_keyset(gpu, chk, 700, nkeys=300, label="c4k/many")
    parity.check_eddsa_keyset(gpu, chk, 40, nkeys=5, label="c4k/few")


def test_eddsa_corner_cases(gpu, chk):
    """torsion in R and A, small-order and undecodable R, non-canonical R: the square-root-free R check against the reference"""
    parity.check_eddsa_adversarial(gpu, chk)


def test_eddsa_rlc(gpu, chk):
    """random-linear-combination batch verification (goldilocks_ed448_verify_rlc_batch): all-valid batches are decided by
    the batch equation, undecodable entries are rejected up front, a single bad signature sends the call to the
    per-signature path; digit widths 3 .. 7, one key for the whole batch, all keys distinct, below the threshold"""
    parity.check_eddsa_rlc(gpu, chk, 1 << 12)
    parity.check_eddsa_rlc(gpu, chk, 300, label="c4r/small")
    parity.check_eddsa_rlc(gpu, chk, 1 << 11, label="c4r/one", per_key=(1 << 11,))
    parity.check_eddsa_rlc(gpu, chk, 1 << 10, label="c4r/distinct", per_key=(1,))
    sig, pk, msgs, kinds = util.verify_corpus(chk, "c4r/tiny", 40)       # fewer than 64: the ordinary path, fast = 0
    st, fast = gpu.ed448_verify_rlc(sig, pk, msgs)
    parity.eq(st, chk.ed448_verify(sig, pk, msgs), "ed448_verify_rlc below the threshold")
    assert fast == 0
    st, fast = gpu.ed448_verify_rlc(np.zeros((0, 114), np.uint8), np.zeros((0, 57), np.uint8), [])
    assert st.shape == (0,)


def test_eddsa_rlc_chunks(gpu, chk):
    """goldilocks_ed448_verify_rlc_batch when the whole-batch equation fails: the per-chunk equations localise the bad signatures
    (fast = 2) and only the failing chunks are re-verified -- statuses are the reference's.  Chunks of 64 signatures so that a
    small batch has many: a short last chunk, key groups that straddle chunk boundaries, bad signatures in the first, a middle and
    the last chunk, an undecodable R (rejected up front: its chunk still holds), then most chunks bad (fast = 0) and the
    skip-and-reprobe policy that follows."""
    os.environ["GOLDILOCKS_B200_RLC_CHUNK"] = "64"
    try:
        gpu.rlc_policy(0)
        n = 64 * 40 + 17
        sk = stream_bytes("c4rc/sk", n * 57).reshape(n, 57)
        for g0 in range(0, n - 24, 100):                                  # repeated keys: groups of 24 straddle the 64-signature chunks
            sk[g0:g0 + 24] = sk[g0]
        lens = stream_bytes("c4rc/len", n).astype(np.int64) % 70
        blob = stream_bytes("c4rc/msg", int(lens.sum()) + 1)
        offs = np.concatenate([[0], np.cumsum(lens)])
        msgs = [bytes(blob[offs[i]:offs[i + 1]]) for i in range(n)]
        pk = chk.ed448_derive_public_key(sk)
        sig = chk.ed448_sign(sk, pk, msgs)
        st, fast = gpu.ed448_verify_rlc(sig, pk, msgs)
        assert fast == 1 and (st == -1).all()
        bad = sig.copy()
        for i in (3, 64 * 7 + 5, 64 * 7 + 60, n - 2):
            bad[i, 60 + i % 50] ^= 4                                      # wrong S in the first, a middle (twice) and the last (short) chunk
        bad[64 * 11 + 9, :57] = util.le(1, 57)                            # undecodable R: rejected up front, chunk 11 still holds
        st, fast = gpu.ed448_verify_rlc(bad, pk, msgs)
        parity.eq(st, chk.ed448_verify(bad, pk, msgs), "rlc chunks: localised fallback")
        assert fast == 2 and (st == 0).sum() == 5
        worse = sig.copy()
        worse[::40, 70] ^= 1                                              # more than half of the chunks fail: per-signature path over everything
        gpu.rlc_policy(4)
        st, fast = gpu.ed448_verify_rlc(worse, pk, msgs)
        parity.eq(st, chk.ed448_verify(worse, pk, msgs), "rlc chunks: most chunks bad")
        assert fast == 0
        seen = [gpu.ed448_verify_rlc(sig, pk, msgs)[1] for _ in range(4)]
        assert seen == [0, 0, 0, 1], "after a hopeless call three calls skip the equation, the fourth tries again: %s" % seen
    finally:
        del os.environ["GOLDILOCKS_B200_RLC_CHUNK"]
        gpu.rlc_policy(16)


def test_eddsa_rlc_device_pointers(gpu, chk):
    """goldilocks_ed448_verify_rlc_batch_dev on torch tensors: same statuses and fast-path flag as the host-pointer call"""
    import torch
    from libgoldilocks_b200.engine import DeviceEngine
    from libgoldilocks_b200.capi import pack_messages
    eng = DeviceEngine()
    dev = torch.device("cuda")
    n = 777
    gpu.rlc_policy(16)
    sig, pk, msgs, kinds = util.verify_corpus(chk, "c4r/dev", n + 1, corrupt_every=n + 1)   # only entry 0 is corrupted: dropped
    sig, pk, msgs = sig[1:].copy(), pk[1:].copy(), msgs[1:]
    arena, off = pack_messages(msgs)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    st = torch.zeros(n, dtype=torch.int32, device=dev)
    d_sig, d_pk, d_msg, d_off = t(sig.reshape(-1)), t(pk.reshape(-1)), t(arena), t(np.asarray(off).view(np.int64))
    assert eng.ed448_verify_rlc(st, d_sig, d_pk, d_msg, d_off) == 1
    assert (st.cpu().numpy() == -1).all()
    bad = sig.copy(); bad[5, 80] ^= 2
    assert eng.ed448_verify_rlc(st, t(bad.reshape(-1)), d_pk, d_msg, d_off) != 1
    parity.eq(st.cpu().numpy(), chk.ed448_verify(bad, pk, msgs), "verify_rlc_batch_dev statuses after the fallback")


def test_decaf_vectors(gpu, vectors):
    parity.check_decaf_vectors(gpu, vectors)


def test_shake(gpu):
    parity.check_shake(gpu)


def test_empty_and_single(gpu):
    z56 = np.zeros((0, 56), np.uint8)
    assert gpu.gf_mul(z56, z56).shape == (0, 56)
    assert gpu.x448(z56, z56)[0].shape == (0, 56)
    assert gpu.ed448_verify(np.zeros((0, 114), np.uint8), np.zeros((0, 57), np.uint8), []).shape == (0,)


def test_legacy_single_element_symbols(gpu, vectors):
    """the reference's own function names, batch of one on the GPU (SURVEY.md 8(b))"""
    import ctypes as C
    L = gpu.lib
    c = vectors["eddsa"][0]
    sk = (C.c_uint8 * 57).from_buffer_copy(bytes.fromhex(c["sk"]))
    pk = (C.c_uint8 * 57)()
    sig = (C.c_uint8 * 114)()
    L.goldilocks_ed448_derive_public_key(pk, sk)
    assert bytes(pk).hex() == c["pk"]
    L.goldilocks_ed448_sign(sig, sk, pk, None, C.c_size_t(0), C.c_uint8(0), None, C.c_uint8(0))
    assert bytes(sig).hex() == c["sig"]
    L.goldilocks_ed448_verify.restype = C.c_int32
    assert L.goldilocks_ed448_verify(sig, pk, None, C.c_size_t(0), C.c_uint8(0), None, C.c_uint8(0)) == -1
    sig[3] ^= 1
    assert L.goldilocks_ed448_verify(sig, pk, None, C.c_size_t(0), C.c_uint8(0), None, C.c_uint8(0)) == 0
    base = (C.c_uint8 * 56)(5)
    out = (C.c_uint8 * 56)()
    L.goldilocks_x448.restype = C.c_int32
    assert L.goldilocks_x448(out, base, base) == -1
    assert bytes(out).hex() == vectors["x448_iter"]["1"]
    zero = (C.c_uint8 * 56)()
    assert L.goldilocks_x448(out, zero, base) == 0 and bytes(out) == bytes(56)


def test_streaming_sha3_and_prehash(gpu, vectors):
    """goldilocks_sha3_* objects (reference shake.c) and Ed448ph through them (eddsa.c:232-251,309-329):
    FIPS 202 outputs from hashlib for every exported parameter set, multi-part update/output, and the
    RFC 8032 Ed448ph vectors through sign_prehash / verify_prehash."""
    import ctypes as C
    import hashlib
    L = gpu.lib
    for f in ("goldilocks_sha3_update", "goldilocks_sha3_output", "goldilocks_sha3_final", "goldilocks_sha3_hash", "goldilocks_ed448_verify_prehash"):
        getattr(L, f).restype = C.c_int32
    L.goldilocks_sha3_default_output_bytes.restype = C.c_size_t
    msg = bytes(stream_bytes("sha3/msg", 1000))
    cases = [("GOLDILOCKS_SHAKE128_params_s", hashlib.shake_128, None), ("GOLDILOCKS_SHAKE256_params_s", hashlib.shake_256, None),
             ("GOLDILOCKS_SHA3_224_params_s", hashlib.sha3_224, 28), ("GOLDILOCKS_SHA3_256_params_s", hashlib.sha3_256, 32),
             ("GOLDILOCKS_SHA3_384_params_s", hashlib.sha3_384, 48), ("GOLDILOCKS_SHA3_512_params_s", hashlib.sha3_512, 64)]
    for sym, href, fixed in cases:
        params = C.c_void_p(C.addressof(C.c_uint8.in_dll(L, sym)))
        for cut in (0, 1, 135, 136, 137, 500, 1000):
            sp = (C.c_uint64 * 26)()
            L.goldilocks_sha3_init(sp, params)
            buf = (C.c_uint8 * 1000).from_buffer_copy(msg)
            assert L.goldilocks_sha3_update(sp, buf, C.c_size_t(cut)) == -1
            rest = (C.c_uint8 * (1000 - cut)).from_buffer_copy(msg[cut:]) if cut < 1000 else None
            assert L.goldilocks_sha3_update(sp, rest, C.c_size_t(1000 - cut)) == -1
            if fixed is None:
                o1, o2 = (C.c_uint8 * 100)(), (C.c_uint8 * 300)()
                assert L.goldilocks_sha3_output(sp, o1, C.c_size_t(100)) == -1
                assert L.goldilocks_sha3_output(sp, o2, C.c_size_t(300)) == -1
                assert bytes(o1) + bytes(o2) == href(msg).digest(400), "%s cut %d" % (sym, cut)
            else:
                assert L.goldilocks_sha3_default_output_bytes(sp) == fixed
                o = (C.c_uint8 * fixed)()
                assert L.goldilocks_sha3_final(sp, o, C.c_size_t(fixed)) == -1
                assert bytes(o) == href(msg).digest(), "%s cut %d" % (sym, cut)
                o2 = (C.c_uint8 * (fixed + 1))()
                L.goldilocks_sha3_update(sp, buf, C.c_size_t(3))
                assert L.goldilocks_sha3_output(sp, o2, C.c_size_t(fixed + 1)) == 0   # more than max_out: FAILURE like the reference
    o = (C.c_uint8 * 64)()
    assert L.goldilocks_sha3_hash(o, C.c_size_t(64), (C.c_uint8 * 1000).from_buffer_copy(msg), C.c_size_t(1000), C.c_void_p(C.addressof(C.c_uint8.in_dll(L, "GOLDILOCKS_SHAKE256_params_s")))) == -1
    assert bytes(o) == hashlib.shake_256(msg).digest(64)
    done = 0
    for c in vectors["eddsa"]:
        if not c["prehashed"]:
            continue
        m = bytes.fromhex(c["msg"]); ctx = bytes.fromhex(c["context"])
        sk = (C.c_uint8 * 57).from_buffer_copy(bytes.fromhex(c["sk"])); pk = (C.c_uint8 * 57).from_buffer_copy(bytes.fromhex(c["pk"]))
        cb = (C.c_uint8 * max(1, len(ctx))).from_buffer_copy(ctx or b"\0")
        h = (C.c_uint64 * 26)()
        L.goldilocks_ed448_prehash_init(h)
        L.goldilocks_sha3_update(h, (C.c_uint8 * max(1, len(m))).from_buffer_copy(m or b"\0"), C.c_size_t(len(m)))
        sig = (C.c_uint8 * 114)()
        L.goldilocks_ed448_sign_prehash(sig, sk, pk, h, cb, C.c_uint8(len(ctx)))
        assert bytes(sig).hex() == c["sig"], "Ed448ph signature"
        assert L.goldilocks_ed448_verify_prehash(sig, pk, h, cb, C.c_uint8(len(ctx))) == -1
        L.goldilocks_sha3_update(h, (C.c_uint8 * 1)(1), C.c_size_t(1))
        assert L.goldilocks_ed448_verify_prehash(sig, pk, h, cb, C.c_uint8(len(ctx))) == 0
        done += 1
    assert done >= 1


def test_spongerng(gpu, chk):
    """goldilocks_spongerng_* (spongerng.c:92-205): a deterministic generator reproduces the reference's stream (the
    reference's own tests draw every input from it, test_goldilocks.cxx:151) -- checked against a hashlib restatement
    and, when the reference build is present, against the reference itself; a non-deterministic one must differ."""
    import ctypes as C
    import hashlib
    L = gpu.lib

    class Model:  # stir = squeeze 32 bytes, re-key with them + input; next = absorb the length, squeeze, stir
        def __init__(self, seed): self.data = b""; self.stir(seed)
        def stir(self, more, skip=0): self.data = hashlib.shake_256(self.data).digest(skip + 32)[skip:] + more
        def next(self, n):
            self.data += n.to_bytes(8, "little")
            out = hashlib.shake_256(self.data).digest(n)
            self.stir(b"", n)
            return out

    seed = b"test_field arithmetic"
    lens = [56, 1, 0, 136, 137, 32, 400, 56]
    prng = (C.c_uint64 * 26)()
    L.goldilocks_spongerng_init_from_buffer(prng, (C.c_uint8 * len(seed)).from_buffer_copy(seed), C.c_size_t(len(seed)), C.c_int(1))
    model = Model(seed)
    ref = None
    if chk.has("goldilocks_spongerng_next"):
        ref = (C.c_uint64 * 26)()
        chk.lib.goldilocks_spongerng_init_from_buffer(ref, (C.c_uint8 * len(seed)).from_buffer_copy(seed), C.c_size_t(len(seed)), C.c_int(1))
    for k, n in enumerate(lens):
        out = (C.c_uint8 * max(1, n))()
        L.goldilocks_spongerng_next(prng, out, C.c_size_t(n))
        want = model.next(n)
        assert bytes(out)[:n] == want, "spongerng_next #%d (%d bytes) vs hashlib model" % (k, n)
        if ref is not None:
            o2 = (C.c_uint8 * max(1, n))()
            chk.lib.goldilocks_spongerng_next(ref, o2, C.c_size_t(n))
            assert bytes(o2)[:n] == want, "reference spongerng_next #%d" % k
        if k == 3:
            extra = b"more entropy"
            L.goldilocks_spongerng_stir(prng, (C.c_uint8 * len(extra)).from_buffer_copy(extra), C.c_size_t(len(extra)))
            model.stir(extra)
            if ref is not None:
                chk.lib.goldilocks_spongerng_stir(ref, (C.c_uint8 * len(extra)).from_buffer_copy(extra), C.c_size_t(len(extra)))
    # non-deterministic: same seed, different streams
    a, b = (C.c_uint64 * 26)(), (C.c_uint64 * 26)()
    oa, ob = (C.c_uint8 * 32)(), (C.c_uint8 * 32)()
    for st, o in ((a, oa), (b, ob)):
        L.goldilocks_spongerng_init_from_buffer(st, (C.c_uint8 * len(seed)).from_buffer_copy(seed), C.c_size_t(len(seed)), C.c_int(0))
        L.goldilocks_spongerng_next(st, o, C.c_size_t(32))
    assert bytes(oa) != bytes(ob)
    L.goldilocks_spongerng_init_from_dev_urandom.restype = C.c_int32
    L.goldilocks_spongerng_init_from_file.restype = C.c_int32
    assert L.goldilocks_spongerng_init_from_dev_urandom(a) == -1
    assert L.goldilocks_spongerng_init_from_file(a, b"/nonexistent/file", C.c_size_t(8), C.c_int(1)) == 0
    assert L.goldilocks_spongerng_init_from_file(a, b"/dev/zero", C.c_size_t(300), C.c_int(1)) == -1
    L.goldilocks_spongerng_next(a, oa, C.c_size_t(32))
    m = Model.__new__(Model); m.data = bytes(300); m.stir(b"")
    assert bytes(oa) == m.next(32), "init_from_file stream"


def test_reference_test_program_passes_on_this_library(gpu):
    """SURVEY.md 8(f)1: the reference's own test/test_goldilocks.cxx, compiled against the reference's public C++
    headers and linked against THIS library (oracle/Makefile: reftest_b200; only NTESTS is lowered), must pass:
    scalar arithmetic, Elligator + inverses, point laws, codecs, X448 / EdDSA vectors, SHAKE objects, SpongeRng --
    every call a batch of one on the GPU."""
    import subprocess
    exe = os.path.join(ROOT, "oracle", "_ref", "reftest_b200")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/reftest_b200 not built (reference sources absent at build time)")
    r = subprocess.run([exe], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=900)
    out = r.stdout.decode(errors="replace")
    log_dir = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(log_dir):
        with open(os.path.join(log_dir, "reftest_b200.log"), "w") as f:
            f.write(out)
    assert r.returncode == 0 and "Passed all tests." in out, out[-3000:]


def test_device_pointer_entry_points_any_alignment(gpu, chk):
    """`*_batch_dev` on torch tensors: the staged field kernel takes its TMA bulk path only for 16-byte aligned, full
    blocks; records that start 8 bytes off (still the documented 8-byte alignment), ragged tails and in-place
    output must give the same bytes through the cooperative path."""
    import torch
    from libgoldilocks_b200.engine import DeviceEngine
    eng = DeviceEngine()
    dev = torch.device("cuda")
    n = 128 * 37 + 5
    a, b = util.field_inputs("dev/gf", n - 256)
    want = chk.gf_mul(a, b)
    for shift in (0, 8):
        ta = torch.zeros(n * 56 + 16, dtype=torch.uint8, device=dev)[shift:shift + n * 56]
        tb = torch.zeros(n * 56 + 16, dtype=torch.uint8, device=dev)[shift:shift + n * 56]
        to = torch.zeros(n * 56 + 16, dtype=torch.uint8, device=dev)[shift:shift + n * 56]
        ta.copy_(torch.from_numpy(a.reshape(-1))); tb.copy_(torch.from_numpy(b.reshape(-1)))
        eng.gf_mul(to, ta, tb)
        assert (to.cpu().numpy().reshape(n, 56) == want).all(), "gf_mul_batch_dev shift %d" % shift
        eng.gf_mul(ta, ta, tb)      # in place
        assert (ta.cpu().numpy().reshape(n, 56) == want).all(), "gf_mul_batch_dev in place, shift %d" % shift
    m = 128 * 5 + 3
    p = util.random_points(chk, "dev/p", m); q = util.random_points(chk, "dev/q", m)
    tp, tq = torch.from_numpy(p.reshape(-1)).to(dev), torch.from_numpy(q.reshape(-1)).to(dev)
    to = torch.empty_like(tp)
    eng.point_add(to, tp, tq)
    assert (util.coords_fast(chk, to.cpu().numpy().reshape(m, 256)) == util.coords_fast(chk, chk.point_add(p, q))).all()
    eng.point_double(tp, tp)        # in place
    assert (util.coords_fast(chk, tp.cpu().numpy().reshape(m, 256)) == util.coords_fast(chk, chk.point_double(p))).all()
    torch.cuda.synchronize()


def _kernel_ms(gpu, fn, reps=5):
    """best-of-`reps` sum of the kernel times of one host-pointer call (the library's per-launch CUDA events)"""
    import ctypes as C
    L = gpu.lib
    L.goldilocks_b200_profile_read.restype = C.c_size_t
    names = C.create_string_buffer(64 * 256); ms = (C.c_float * 256)()
    best = None
    fn()
    for _ in range(reps):
        L.goldilocks_b200_profile(C.c_int(1))
        fn()
        L.goldilocks_b200_profile(C.c_int(0))
        cnt = L.goldilocks_b200_profile_read(names, ms, C.c_size_t(256))
        t = sum(ms[k] for k in range(cnt))
        best = t if best is None else min(best, t)
    return best


def test_secret_paths_time_independent_of_the_scalar(gpu, chk):
    """dynamic side of the constant-time claim (static side: tools/ct_audit.py on the SASS): the kernels of the secret paths
    take the same time for all-zero, all-ones, single-bit and random scalars -- 2^18 lanes each, best of 5, within 2 %.  A
    secret-indexed table or a secret-dependent branch would show up as a cache / divergence difference between the
    degenerate patterns (every lane the same index) and the random one (every lane another)."""
    n = 1 << 18
    pats = {"zero": np.zeros((n, 56), np.uint8), "ones": np.full((n, 56), 0xff, np.uint8), "random": stream_bytes("ct/r", n * 56).reshape(n, 56)}
    bit = np.zeros((n, 56), np.uint8); bit[:, 30] = 0x10
    pats["one_bit"] = bit
    pts = util.random_points(chk, "ct/p", n)
    u = stream_bytes("ct/u", n * 56).reshape(n, 56)
    sk57 = {k: np.concatenate([v, v[:, :1]], axis=1) for k, v in pats.items()}
    msgs = (stream_bytes("ct/m", n * 32), np.arange(n + 1, dtype=np.uint64) * 32)
    pk = gpu.ed448_derive_public_key(sk57["random"])
    report = {}
    for name, call in (("precomputed_scalarmul", lambda s, k: gpu.precomputed_scalarmul(gpu.scalar_decode_long(s, 56))),
                       ("x448", lambda s, k: gpu.x448(u, s)),
                       ("point_scalarmul", lambda s, k: gpu.point_scalarmul(pts, gpu.scalar_decode_long(s, 56))),
                       ("ed448_derive_public_key", lambda s, k: gpu.ed448_derive_public_key(k)),
                       ("ed448_sign", lambda s, k: gpu.ed448_sign(k, pk, msgs))):
        times = {}
        for pat in pats:
            s, k = pats[pat], sk57[pat]
            if name in ("precomputed_scalarmul", "point_scalarmul"):
                sc = gpu.scalar_decode_long(s, 56)
                fn = (lambda sc=sc: gpu.precomputed_scalarmul(sc)) if name == "precomputed_scalarmul" else (lambda sc=sc: gpu.point_scalarmul(pts, sc))
            else:
                fn = lambda s=s, k=k: call(s, k)
            times[pat] = _kernel_ms(gpu, fn)
        report[name] = times
        lo, hi = min(times.values()), max(times.values())
        print("[ct-timing] %-24s %s  spread %.2f %%" % (name, {k: round(v, 3) for k, v in times.items()}, 100 * (hi - lo) / lo))
        assert hi <= 1.02 * lo, "%s: kernel time depends on the scalar pattern: %s" % (name, times)
    out = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(out):
        import json
        with open(os.path.join(out, "ct_timing.json"), "w") as f:
            json.dump(report, f, indent=1)


def test_concurrent_host_threads(gpu, chk):
    """host threads that call at the same time are dealt the three contexts of a device round-robin (abi.cu my_lane): six threads, each
    looping over a different mix of entry points (verify, X448, sign, codec, comb), must all get the single-threaded answers -- with and
    without a device set installed underneath them"""
    import threading
    n = 3000
    sig, pk, msgs, kinds = util.verify_corpus(chk, "thr/v", n)
    u = stream_bytes("thr/u", n * 56).reshape(n, 56); k = stream_bytes("thr/k", n * 56).reshape(n, 56)
    sk = stream_bytes("thr/sk", n * 57).reshape(n, 57)
    h = stream_bytes("thr/h", 20000 * 56).reshape(20000, 56)
    sc = util.random_scalars(chk, "thr/s", n)
    want = {"verify": gpu.ed448_verify(sig, pk, msgs), "x448": gpu.x448(u, k)[0], "pk": gpu.ed448_derive_public_key(sk),
            "enc": gpu.point_encode(gpu.from_hash_nonuniform(h)), "comb": gpu.point_encode(gpu.precomputed_scalarmul(sc))}
    want["sign"] = gpu.ed448_sign(sk, want["pk"], msgs)
    parity.eq(want["verify"], chk.ed448_verify(sig, pk, msgs), "single-threaded verify vs reference")
    errors = []

    def worker(t):
        try:
            for it in range(4):
                which = (t + it) % 5
                if which == 0:
                    parity.eq(gpu.ed448_verify(sig, pk, msgs), want["verify"], "thread %d verify" % t)
                elif which == 1:
                    parity.eq(gpu.x448(u, k)[0], want["x448"], "thread %d x448" % t)
                elif which == 2:
                    parity.eq(gpu.ed448_sign(sk, want["pk"], msgs), want["sign"], "thread %d sign" % t)
                elif which == 3:
                    parity.eq(gpu.point_encode(gpu.from_hash_nonuniform(h)), want["enc"], "thread %d elligator + encode" % t)
                else:
                    parity.eq(gpu.point_encode(gpu.precomputed_scalarmul(sc)), want["comb"], "thread %d comb" % t)
        except Exception as e:  # noqa: BLE001
            errors.append("thread %d: %r" % (t, e))

    for devs in ([], [0, 0]):
        gpu.set_devices(devs)
        try:
            threads = [threading.Thread(target=worker, args=(t,)) for t in range(6)]
            for th in threads:
                th.start()
            for th in threads:
                th.join()
        finally:
            gpu.set_devices([])
        assert not errors, errors


def test_device_set_sharded_equals_unsharded(gpu, chk):
    """goldilocks_b200_set_devices: ONE host-pointer batch cut into contiguous ranges over the device set (csrc/shard.h) gives
    the bytes of the unsharded call for every kind of entry point -- heavy (one range per device: verify incl. key groups
    that straddle a cut, RLC, sign, X448, scalar multiplications) and light (chunks pipelined over three contexts per
    device).  On a one-GPU box the same device is listed three times, which exercises the same partition and workers."""
    import torch
    ndev = torch.cuda.device_count()
    devs = list(range(ndev)) if ndev >= 2 else [0, 0, 0]
    n = 3 * 4096 + 77
    sig, pk, msgs, kinds = util.verify_corpus(chk, "shard/v", n)
    pk[100:4200] = pk[100]                                # one key group across the first cut (its signatures now fail: fine)
    sk = stream_bytes("shard/sk", n * 57).reshape(n, 57)
    u = stream_bytes("shard/u", n * 56).reshape(n, 56); k = stream_bytes("shard/k", n * 56).reshape(n, 56)
    sc = util.random_scalars(chk, "shard/s", n); pts = util.random_points(chk, "shard/p", n)
    big = 1 << 18                                          # light operations: enough traffic for several chunks per lane
    h = stream_bytes("shard/h", big * 56).reshape(big, 56)

    def run():
        out = {}
        out["verify"] = gpu.ed448_verify(sig, pk, msgs)
        out["rlc"] = gpu.ed448_verify_rlc(sig, pk, msgs)[0]
        pkd = gpu.ed448_derive_public_key(sk)
        out["pk"] = pkd
        out["sign"] = gpu.ed448_sign(sk, pkd, msgs, context=b"shard")
        out["x448"], out["x448_st"] = gpu.x448(u, k)
        out["scalarmul"] = gpu.point_encode(gpu.point_scalarmul(pts, sc))
        out["bdsm"] = gpu.point_encode(gpu.base_double_scalarmul_non_secret(sc, pts, sc[::-1].copy()))
        p = gpu.from_hash_nonuniform(h)
        out["elligator"] = util.coords_fast(chk, p)
        out["encode"] = gpu.point_encode(p)
        d, st = gpu.point_decode(out["encode"])
        out["decode"], out["decode_st"] = util.coords_fast(chk, d), st
        out["add"] = util.coords_fast(chk, gpu.point_add(p, d[::-1].copy()))
        out["comb"] = gpu.point_encode(gpu.precomputed_scalarmul(util.random_scalars(chk, "shard/c", big)))
        out["gf_mul"] = gpu.gf_mul(h, h[::-1].copy())
        out["shake"] = gpu.shake256(msgs, 33) if hasattr(gpu, "shake256") else np.zeros(1)
        return out

    assert gpu.get_devices() == []
    base = run()
    parity.eq(base["verify"], chk.ed448_verify(sig, pk, msgs), "unsharded verify vs reference")
    gpu.set_devices(devs)
    try:
        assert gpu.get_devices() == devs
        got = run()
    finally:
        gpu.set_devices([])
    for name in base:
        parity.eq(got[name], base[name], "device set %s: %s" % (devs, name))
    assert gpu.get_devices() == []
    gpu.set_devices([0])                                   # a set of one device: light operations are still pipelined
    try:
        parity.eq(gpu.point_encode(gpu.from_hash_nonuniform(h)), base["encode"], "one-device set: pipelined elligator + encode")
        parity.eq(gpu.ed448_verify(sig, pk, msgs), base["verify"], "one-device set: verify")
    finally:
        gpu.set_devices([])


# ---- the full 2^20 batches of BASELINE.json, every element compared with the compiled reference (all host cores) ----

def _timed(what, t0):
    import time
    print("[full-parity] %s: %.1f s" % (what, time.time() - t0))


def test_points_all_2_20(gpu, chk):
    """config 1 (group half) at 2^20: all four coordinates of point_add / point_sub / point_double against the reference
    (goldilocks.c:178-258) on 2^20 pairs, half of them non-trivial projective representatives"""
    import time
    t0 = time.time()
    n = FULL
    p = util.random_points(chk, "c1full/p", n)
    q = util.random_points(chk, "c1full/q", n)
    p[1::2] = chk.point_add(p[1::2], q[::2])          # Z != 1 inputs
    q[1::2] = chk.point_double(q[1::2])
    c = util.coords_fast
    parity.eq(c(chk, gpu.point_add(p, q)), c(chk, chk.point_add(p, q)), "point_add coords over 2^20")
    parity.eq(c(chk, gpu.point_sub(p, q)), c(chk, chk.point_sub(p, q)), "point_sub coords over 2^20")
    parity.eq(c(chk, gpu.point_double(p)), c(chk, chk.point_double(p)), "point_double coords over 2^20")
    _timed("point add/sub/double 2^20 vs reference", t0)


def test_x448_all_2_20(gpu, chk):
    """config 3 at 2^20: output bytes and status of every element against the reference (goldilocks.c:1006-1076), random u
    (any 56 bytes, so non-canonical u too) and random scalars, the edge block of check_x448 riding along; DH commutes"""
    import time
    t0 = time.time()
    n = FULL
    a = stream_bytes("c3full/a", n * 56).reshape(n, 56)
    b = stream_bytes("c3full/b", n * 56).reshape(n, 56)
    u = stream_bytes("c3full/u", n * 56).reshape(n, 56)
    u[-9:] = parity.x448_inputs(1)[0][-9:]           # 0, 1, p-1, p, p+5, 2^448-1, ...
    o1, s1 = gpu.x448(u, a)
    o2, s2 = chk.x448(u, a)
    parity.eq(s1, s2, "x448 status over 2^20")
    parity.eq(o1, o2, "x448 output over 2^20")
    _timed("x448 2^20 vs reference", t0)
    base = np.zeros((n, 56), np.uint8); base[:, 0] = 5
    pa, sa = gpu.x448(base, a)
    pb, sb = gpu.x448(base, b)
    ab, s3 = gpu.x448(pa, b)
    ba, s4 = gpu.x448(pb, a)
    assert (sa == -1).all() and (sb == -1).all() and (s3 == -1).all() and (s4 == -1).all()
    parity.eq(ab, ba, "x448 DH commutativity over 2^20")


def test_comb_all_2_20(gpu, chk):
    """config 2 at 2^20: decaf encoding of precomputed_scalarmul(k) for every k against the reference
    (goldilocks.c:830-877 then 98-140); comb(a) + comb(b) == comb(a+b)"""
    import time
    t0 = time.time()
    n = FULL
    a = gpu.scalar_decode_long(stream_bytes("c2full/a", n * 56).reshape(n, 56), 56)
    a[-len(util.scalar_edge_bytes()):] = util.scalar_edge_bytes()
    pa = gpu.precomputed_scalarmul(a)
    parity.eq(gpu.point_encode(pa), chk.point_encode(chk.precomputed_scalarmul(a)), "comb decaf encoding over 2^20")
    _timed("comb + encode 2^20 vs reference", t0)
    b = gpu.scalar_decode_long(stream_bytes("c2full/b", n * 56).reshape(n, 56), 56)
    pab = gpu.precomputed_scalarmul(gpu.scalar_add(a, b))
    assert gpu.point_eq(gpu.point_add(pa, gpu.precomputed_scalarmul(b)), pab).all()


def _c4_corpus(signer, label, nk, per, kinds_mod=5):
    """SURVEY 8(d) C4: nk keys x per messages of 32 bytes SIGNED BY `signer` (the reference), 1/8 corrupted"""
    n = nk * per
    sk = stream_bytes(label + "/sk", nk * 57).reshape(nk, 57)
    pk = signer.ed448_derive_public_key(sk)
    sk_all, pk_all = np.repeat(sk, per, axis=0), np.repeat(pk, per, axis=0)
    arena = stream_bytes(label + "/msg", n * 32)
    off = (np.arange(n + 1, dtype=np.uint64) * 32)
    sig = signer.ed448_sign(sk_all, pk_all, (arena, off))
    kinds = np.zeros(n, np.int32)
    kinds[::8] = 1 + (np.arange(n // 8) % kinds_mod)
    sel = stream_bytes(label + "/sel", n)
    i1 = np.flatnonzero(kinds == 1); sig[i1, sel[i1] % 57] ^= 1
    i2 = np.flatnonzero(kinds == 2); sig[i2, 57 + sel[i2] % 56] ^= 2
    i3 = np.flatnonzero(kinds == 3); pk_all[i3, sel[i3] % 57] ^= 4
    i4 = np.flatnonzero(kinds == 4); arena[i4 * 32 + sel[i4] % 32] ^= 8
    for i in np.flatnonzero(kinds == 5)[:4096]:
        sig[i, 57:114] = util.le(util.from_le(sig[i, 57:114]) + util.Q, 57)      # S + q: accepted by the reference
    kinds[np.flatnonzero(kinds == 5)[4096:]] = 0
    return sk_all, pk, sig, pk_all, arena, off, kinds


def test_verify_all_2_20(gpu, chk):
    """config 4 at 2^20, corpus signed by the REFERENCE (SURVEY 8(d)): 2^16 keys x 16 messages, 1/8 corrupted.  All 2^20
    accept bits against goldilocks_ed448_verify of the reference (eddsa.c:253-306), the product's signatures over the
    same 2^20 (key, message) pairs byte for byte against the reference's, and the corruption kinds' expected verdicts"""
    import time
    t0 = time.time()
    sk_all, pk, sig, pk_all, arena, off, kinds = _c4_corpus(chk, "c4full", 1 << 16, 16)
    _timed("reference keygen + sign 2^20", t0)
    t0 = time.time()
    st = gpu.ed448_verify(sig, pk_all, (arena, off))
    want = chk.ed448_verify(sig, pk_all, (arena, off))
    _timed("reference verify 2^20", t0)
    parity.eq(st, want, "verify accept bits over 2^20 vs reference")
    parity.eq(st, np.where((kinds == 0) | (kinds == 5), -1, 0).astype(np.int32), "verify accept bits over 2^20 vs corruption kinds")
    parity.eq(gpu.ed448_derive_public_key(sk_all[::16]), pk, "derive_public_key over 2^16 vs reference")
    clean = kinds == 0                                   # the signatures the corpus left untouched are the reference's own bytes
    arena0, pk0 = stream_bytes("c4full/msg", len(arena)), np.repeat(pk, 16, axis=0)
    parity.eq(gpu.ed448_sign(sk_all, pk0, (arena0, off))[clean], sig[clean], "sign over 2^20 vs reference")


def test_verify_all_2_20_distinct_keys(gpu, chk):
    """the same with 2^20 DISTINCT keys (no per-key table can be shared: every signature takes the stand-alone finish)"""
    import time
    t0 = time.time()
    sk_all, pk, sig, pk_all, arena, off, kinds = _c4_corpus(chk, "c4fulld", 1 << 20, 1)
    st = gpu.ed448_verify(sig, pk_all, (arena, off))
    parity.eq(st, chk.ed448_verify(sig, pk_all, (arena, off)), "verify accept bits over 2^20 distinct keys vs reference")
    parity.eq(st, np.where((kinds == 0) | (kinds == 5), -1, 0).astype(np.int32), "verify accept bits (distinct keys) vs corruption kinds")
    _timed("distinct-key corpus: reference keygen + sign + verify 2^20", t0)


def test_verify_rlc_full(gpu, chk):
    """2^20 valid signatures (2^16 keys x 16 messages): the batch equation accepts them all; with one wrong S, one
    undecodable R and one swapped message among them the statuses are exactly those three rejections"""
    nk, per = 1 << 16, 16
    n = nk * per
    sk = stream_bytes("c4rfull/sk", nk * 57).reshape(nk, 57)
    pk = gpu.ed448_derive_public_key(sk)
    sk_all, pk_all = np.repeat(sk, per, axis=0), np.repeat(pk, per, axis=0)
    arena = stream_bytes("c4rfull/msg", n * 32)
    off = (np.arange(n + 1, dtype=np.uint64) * 32)
    sig = gpu.ed448_sign(sk_all, pk_all, (arena, off))
    gpu.rlc_policy(16)
    st, fast = gpu.ed448_verify_rlc(sig, pk_all, (arena, off))
    assert fast == 1 and (st == -1).all()
    sig[777, :57] = util.le(1, 57)                     # undecodable R: rejected up front, the equation still decides
    st, fast = gpu.ed448_verify_rlc(sig, pk_all, (arena, off))
    assert fast == 1 and st[777] == 0 and (st == -1).sum() == n - 1
    sig[123456, 99] ^= 0x10                            # wrong S
    arena[32 * 999999 + 5] ^= 1                        # another message
    st, fast = gpu.ed448_verify_rlc(sig, pk_all, (arena, off))
    assert fast == 2                                   # localised: 2 of 256 chunks re-verified one signature at a time
    expect = np.full(n, -1, np.int32); expect[[777, 123456, 999999]] = 0
    parity.eq(st, expect, "verify_rlc statuses over 2^20 after the fallback")
    parity.eq(st, gpu.ed448_verify(sig, pk_all, (arena, off)), "verify_rlc vs verify over 2^20")


def test_codec_roundtrip_large(gpu, chk):
    """config 5 shape at 2^21 elements = one GPU's share of BASELINE configs[4] (2^24 over 8 GPUs): Elligator-hashed points
    are valid, encode(decode(encode(P))) is idempotent, one Elligator preimage per point maps back to it, and a sample
    of the encodings is compared with the checker"""
    n = 1 << 21
    h = stream_bytes("c5full/h", n * 56).reshape(n, 56)
    pts = gpu.from_hash_nonuniform(h)
    ser = gpu.point_encode(pts)
    dec, st = gpu.point_decode(ser)
    assert (st == -1).all()
    parity.eq(gpu.point_encode(dec), ser, "encode/decode round trip over 2^21")
    assert gpu.point_eq(dec, pts).all()
    del dec
    which = (np.arange(n) % 8).astype(np.uint32)
    rec, ok = gpu.invert_elligator_nonuniform(pts, which)
    good = ok == -1
    assert good.sum() > n // 8
    assert gpu.point_eq(gpu.from_hash_nonuniform(rec[good]), pts[good]).all(), "from_hash(invert_elligator(P)) != P"
    idx = np.arange(0, n, n // (1 << 13))
    parity.eq(ser[idx], chk.point_encode(chk.from_hash_nonuniform(h[idx])), "elligator+encode sample vs checker")


def test_single_calls_from_many_threads_are_gathered(gpu, chk):
    """goldilocks_b200_coalesce (csrc/coalesce.h): 32 host threads call the reference's own one-element entry points -- verify (three
    different (prehashed, context) domains mixed in one gathering), sign and X448 -- and every call must return what the reference returns for
    it, while the library runs them as a few batches instead of one launch per call"""
    import threading
    T, K = 32, 12
    n = T * K
    doms = [(False, b""), (False, b"gathered"), (True, b"\x07" * 9)]
    sk = stream_bytes("coal/sk", n * 57).reshape(n, 57)
    pk = chk.ed448_derive_public_key(sk)
    msgs = [bytes(stream_bytes("coal/m%d" % i, 64 if doms[i % 3][0] else i % 50)) for i in range(n)]
    sig = np.zeros((n, 114), np.uint8)
    for d, (ph, ctx) in enumerate(doms):
        idx = np.arange(d, n, 3)
        sig[idx] = chk.ed448_sign(sk[idx], pk[idx], [msgs[i] for i in idx], ph, ctx)
    bad = sig.copy()
    bad[::4, 60] ^= 1
    want_v = np.zeros(n, np.int32)
    for d, (ph, ctx) in enumerate(doms):
        idx = np.arange(d, n, 3)
        want_v[idx] = chk.ed448_verify(bad[idx], pk[idx], [msgs[i] for i in idx], ph, ctx)
    assert (want_v == -1).sum() > n // 2 and (want_v == 0).sum() >= n // 5
    u = stream_bytes("coal/u", n * 56).reshape(n, 56); k = stream_bytes("coal/k", n * 56).reshape(n, 56)
    u[5] = 0                                                       # a low-order point: FAILURE and 56 zero bytes
    want_x, want_xs = chk.x448(u, k)
    errors = []

    def worker(t):
        try:
            for j in range(K):
                i = t * K + j
                ph, ctx = doms[i % 3]
                st = gpu.ed448_verify_one(bad[i], pk[i], msgs[i], ph, ctx)
                if st != want_v[i]:
                    errors.append("verify %d: %d, reference %d" % (i, st, want_v[i]))
                s = gpu.ed448_sign_one(sk[i], pk[i], msgs[i], ph, ctx)
                if s != bytes(sig[i]):
                    errors.append("sign %d differs" % i)
                o, st = gpu.x448_one(u[i], k[i])
                if o != bytes(want_x[i]) or st != want_xs[i]:
                    errors.append("x448 %d differs" % i)
        except Exception as e:  # noqa: BLE001
            errors.append("thread %d: %r" % (t, e))

    calls0, batches0, _ = gpu.coalesce_stats()
    gpu.coalesce(300)
    try:
        threads = [threading.Thread(target=worker, args=(t,)) for t in range(T)]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
    finally:
        gpu.coalesce(0)
    assert not errors, errors[:5]
    calls, batches, largest = gpu.coalesce_stats()
    assert calls - calls0 == 3 * n
    assert batches - batches0 < (calls - calls0) // 3 and largest >= 4, (calls - calls0, batches - batches0, largest)
    # switched off again: a call runs alone and still answers
    assert gpu.ed448_verify_one(sig[0], pk[0], msgs[0]) == -1 and gpu.coalesce_stats()[0] == calls


def test_two_verifications_in_flight_on_two_streams(gpu, chk):
    """goldilocks_ed448_verify_batch_dev writes only into the caller's scratch, so two calls on two streams -- each with its own scratch and
    status array, one over a batch of repeated keys, one over distinct keys (half-size stand-alone path) -- may overlap freely and must
    both give the reference's statuses, call after call"""
    import torch
    from libgoldilocks_b200.engine import DeviceEngine
    from libgoldilocks_b200.capi import pack_messages
    eng = DeviceEngine()
    dev = torch.device("cuda")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    jobs = []
    for label, n, per in (("2s/shared", 6000, 12), ("2s/distinct", 5000, 1)):
        nk = (n + per - 1) // per
        sk = stream_bytes(label + "/sk", nk * 57).reshape(nk, 57)[np.arange(n) // per]
        pk = chk.ed448_derive_public_key(sk)
        msgs = [bytes(stream_bytes(label + "/m%d" % i, i % 40)) for i in range(n)]
        sig = chk.ed448_sign(sk, pk, msgs)
        sig[::5, 90] ^= 4
        arena, off = pack_messages(msgs)
        want = chk.ed448_verify(sig, pk, msgs)
        assert (want == 0).sum() == (n + 4) // 5
        jobs.append({"want": want, "st": torch.zeros(n, dtype=torch.int32, device=dev), "args": (t(sig.reshape(-1)), t(pk.reshape(-1)), t(arena), t(np.asarray(off).view(np.int64))),
                     "scratch": torch.empty(eng.verify_scratch_bytes(n), dtype=torch.uint8, device=dev), "stream": torch.cuda.Stream(device=dev)})
    torch.cuda.synchronize()
    for rep in range(3):
        for j in jobs:
            j["st"].zero_()
        torch.cuda.synchronize()
        for _ in range(2):                                           # back to back on each stream, interleaved across the two
            for j in jobs:
                with torch.cuda.stream(j["stream"]):
                    eng.ed448_verify(j["st"], *j["args"], j["scratch"])
        torch.cuda.synchronize()
        for j in jobs:
            parity.eq(j["st"].cpu().numpy(), j["want"], "verify_batch_dev statuses with two calls in flight, round %d" % rep)
