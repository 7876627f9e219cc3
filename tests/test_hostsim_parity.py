"""CPU tier: the CUDA sources' device math compiled for the host (tests/hostsim, with limb-bound
assertions on) against the checker and the reference's golden vectors.  No GPU needed."""
import os

import numpy as np

import parity
import util


def _threads(*libs):
    for lib in libs:
        util.set_threads(lib, os.cpu_count() or 1)


def test_field(sim, chk):
    _threads(sim, chk)
    parity.check_field(sim, chk, 4096)
    parity.check_field_isr(sim, chk, 256)


def test_points(sim, chk):
    parity.check_points(sim, chk, 1024)


def test_niels_mixed_additions(sim, chk):
    """row a9 directly: the mixed additions and conversions of goldilocks.c:271-380, by value and on the slot machine"""
    parity.check_niels(sim, chk, 300)


def test_codec_elligator(sim, chk):
    parity.check_codec(sim, chk, 256)
    parity.check_elligator_inverse(sim, chk, 96)


def test_scalars(sim, chk):
    parity.check_scalars(sim, chk, 1024)


def test_tables(sim, chk):
    parity.check_tables(sim, chk)


def test_comb(sim, chk):
    parity.check_comb(sim, chk, 256)


def test_scalarmul(sim, chk):
    parity.check_scalarmul(sim, chk, 64)


def test_x448(sim, chk, vectors):
    _threads(sim, chk)
    parity.check_x448(sim, chk, 128)
    parity.check_x448_vectors(sim, vectors, iters=1000)


def test_eddsa(sim, chk, vectors):
    _threads(sim, chk)
    parity.check_eddsa_vectors(sim, vectors)
    parity.check_eddsa_random(sim, chk, 192)
    parity.check_eddsa_grouped(sim, chk, 160)                                          # 13 signatures per key table: 15 columns x 6 rows
    parity.check_eddsa_grouped(sim, chk, 80, label="c4g/few", per_key=(2, 3, 1))       # 2.5 per key table: 10 columns x 9 rows (vsh_pick)
    parity.check_eddsa_grouped(sim, chk, 132, label="c4g/44", per_key=(44,))           # 30 columns x 3 rows
    parity.check_eddsa_grouped(sim, chk, 300, label="c4g/300", per_key=(300,))         # one signer: 90 columns, additions only
    parity.check_eddsa_grouped(sim, chk, 380, label="c4g/edge9", per_key=(9, 10, 8, 11))       # averages right at the shape thresholds
    parity.check_eddsa_grouped(sim, chk, 384, label="c4g/edge32", per_key=(32, 31, 33))
    parity.check_eddsa_grouped(sim, chk, 811, label="c4g/edge256", per_key=(256, 300, 255))
    parity.check_eddsa_keyset(sim, chk, 120)
    parity.check_eddsa_adversarial(sim, chk, copies=1)
    parity.check_eddsa_grouped(sim, chk, 96, label="c4g/ctx", prehashed=True, context=b"ctx")


def test_decaf_vectors(sim, vectors):
    parity.check_decaf_vectors(sim, vectors)


def test_shake(sim):
    parity.check_shake(sim)


def test_openssl_golden(sim):
    parity.check_openssl_golden(sim, util.openssl_golden())


def test_widened(sim, chk):
    parity.check_widened(sim, chk, 96)


def test_eddsa_rlc(sim, chk):
    """random-linear-combination batch verification (csrc/rlc.cuh) at several digit widths"""
    import ctypes
    _threads(sim, chk)
    for c in (0, 2, 5, 7):   # 0 = the width the product picks for this n; 7 > log2(32): segments and tree nodes both in play
        sim.lib.hostsim_rlc_config(ctypes.c_int(c), None)
        parity.check_eddsa_rlc(sim, chk, 150 if c else 100, label="c4r/%d" % c)
    sim.lib.hostsim_rlc_config(ctypes.c_int(0), None)
    # tiny batches (the host simulator has no size threshold) and a batch in which every key is undecodable
    import numpy as np
    for n in (1, 2, 5):
        sk = util.stream_bytes("c4r/tiny/sk%d" % n, n * 57).reshape(n, 57)
        pk = chk.ed448_derive_public_key(sk)
        msgs = [bytes(util.stream_bytes("c4r/tiny/m%d.%d" % (n, i), i)) for i in range(n)]
        sig = chk.ed448_sign(sk, pk, msgs)
        st, fast = sim.ed448_verify_rlc(sig, pk, msgs)
        assert fast == 1 and (st == -1).all()
        sig[0, 100] ^= 1
        st, fast = sim.ed448_verify_rlc(sig, pk, msgs)
        assert fast == 0 and st[0] == 0 and (st[1:] == -1).all()
        pk[:] = util.le(1, 57)
        st, fast = sim.ed448_verify_rlc(sig, pk, msgs)
        assert (st == 0).all() and fast == 1     # everything rejected up front; the empty equation holds


def test_eddsa_rlc_chunks(sim, chk):
    """chunked batch equations (branch next/rlc-chunks): every chunk of consecutive signatures has its own verdict, so a bad
    signature sends only its chunk to the per-signature path; statuses are the reference's for every chunk size"""
    import ctypes
    _threads(sim, chk)
    try:
        for csize in (16, 50, 149):
            sim.lib.hostsim_rlc_chunk(ctypes.c_size_t(csize))
            for c in (0, 3):
                sim.lib.hostsim_rlc_config(ctypes.c_int(c), None)
                parity.check_eddsa_rlc(sim, chk, 150, label="c4r/chunk%d.%d" % (csize, c))
    finally:
        sim.lib.hostsim_rlc_chunk(ctypes.c_size_t(0))
        sim.lib.hostsim_rlc_config(ctypes.c_int(0), None)


def test_scalar_folding_reduction_fuzz(sim):
    """sc_reduce_114 / sc_reduce_57 (csrc/sc.cuh: folding at 2^448 = 4c) against Python integers: random values, long runs
    of ones and zeros (carry ripples), multiples of q plus small offsets, values just below the top"""
    import random
    import numpy as np
    _threads(sim)
    rnd = random.Random(448)
    for ln in (57, 114):
        top = 2 ** (8 * ln)
        vals = []
        for t in range(6000):
            r = rnd.random()
            if r < 0.3:
                v = rnd.getrandbits(8 * ln)
            elif r < 0.6:
                v, pos = 0, 0
                while pos < 8 * ln:
                    run = rnd.choice([1, 7, 31, 32, 33, 64, 100, 224])
                    if rnd.random() < 0.5:
                        v |= ((1 << run) - 1) << pos
                    pos += run
                v %= top
            elif r < 0.8:
                v = (rnd.getrandbits(8 * ln - 446) * util.Q + rnd.choice([0, 1, util.Q - 1, rnd.getrandbits(200)])) % top
            else:
                v = (top - 1 - rnd.getrandbits(rnd.randrange(1, 8 * ln))) % top
            vals.append(v)
        ser = np.stack([util.le(v, ln) for v in vals])
        want = np.stack([util.le(v % util.Q, 56) for v in vals])
        parity.eq(sim.scalar_decode_long(ser, ln), want, "scalar_decode_long by folding, len %d" % ln)


def test_half_gcd(sim):
    """sc_half_gcd (csrc/sc.cuh, decision 15): for every c < q it must return u, v with v c == u (mod q), 0 <= u < 2^223 and
    0 < |v| < 2^223 -- checked on Python integers for random scalars and for the inputs that stress Lehmer's batching and the stopping
    rule: all-ones quotients (q times a Fibonacci ratio), c next to q a / b (a huge quotient late in the sequence), c around 2^223 and
    around every power of two, inverses of 223-bit numbers (a remainder right at the stopping point), 0, 1, q - 1."""
    import ctypes as C
    import random
    Q = util.Q
    rnd = random.Random(20260917)
    fa, fb = 1, 1
    for _ in range(330):
        fa, fb = fb, fa + fb
    cs = [0, 1, 2, 3, Q - 1, Q - 2, Q // 2, Q // 2 + 1, Q * fa // fb]
    for a in range(1, 24):
        for b in range(a + 1, 25):
            cs += [Q * a // b, Q * a // b + 1]
    for k in range(1, 223):
        cs += [(1 << 223) + (1 << k), (1 << (223 + k % 200)) - 1]
    for k in range(2, 446):
        cs += [Q >> k, (Q >> k) + 1, Q - (1 << k)]
    for _ in range(200):
        t = rnd.randrange(1 << 222, 1 << 223) | 1
        cs += [pow(t, -1, Q), rnd.randrange(1 << 223) * pow(t, -1, Q) % Q]
    cs += [rnd.randrange(Q) for _ in range(20000)]
    cs = [x % Q for x in cs]
    n = len(cs)
    c = np.frombuffer(b"".join(x.to_bytes(56, "little") for x in cs), np.uint8).reshape(n, 56).copy()
    u = np.zeros((n, 56), np.uint8); v = np.zeros((n, 56), np.uint8); neg = np.zeros(n, np.uint32)
    sim.lib.hostsim_half_gcd(u.ctypes.data_as(C.c_void_p), v.ctypes.data_as(C.c_void_p), neg.ctypes.data_as(C.c_void_p),
                             c.ctypes.data_as(C.c_void_p), C.c_size_t(n))
    for i, x in enumerate(cs):
        uu = int.from_bytes(bytes(u[i]), "little"); vv = int.from_bytes(bytes(v[i]), "little")
        if neg[i]:
            vv = -vv
        assert (vv * x - uu) % Q == 0, "v c != u (mod q) for c = %x" % x
        assert 0 <= uu < (1 << 223) and 0 < abs(vv) < (1 << 223), "bounds for c = %x: %d / %d bits" % (x, uu.bit_length(), abs(vv).bit_length())
