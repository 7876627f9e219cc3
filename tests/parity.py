"""Parity checks shared by the CPU tier (lib = host simulator of the CUDA sources) and the GPU tier
(lib = libgoldilocks_b200.so on a B200).  `chk` is the checker (reference build or oracle).
Every comparison is bit-exact (integer/byte work)."""
import hashlib

import numpy as np

import util
from util import P, Q, le, stream_bytes


def eq(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, "%s: shape %s vs %s" % (what, a.shape, b.shape)
    if not (a == b).all():
        bad = np.argwhere((a != b).reshape(len(a), -1).any(axis=1)).ravel()
        raise AssertionError("%s: %d of %d elements differ, first at %d" % (what, len(bad), len(a), bad[0]))


def check_field(lib, chk, n):
    """BASELINE config 1 (field half): gf_mul/sqr/add/sub/mulw on n random + edge pairs"""
    a, b = util.field_inputs("c1/field", n)
    eq(lib.gf_mul(a, b), chk.gf_mul(a, b), "gf_mul")
    eq(lib.gf_sqr(a), chk.gf_sqr(a), "gf_sqr")
    eq(lib.gf_add(a, b), chk.gf_add(a, b), "gf_add")
    eq(lib.gf_sub(a, b), chk.gf_sub(a, b), "gf_sub")
    for w in (1, 39081, 39082, 156326, (1 << 28) - 1):
        eq(lib.gf_mulw(a[: max(64, n // 8)], w), chk.gf_mulw(a[: max(64, n // 8)], w), "gf_mulw %d" % w)


def check_field_isr(lib, chk, n):
    a, _ = util.field_inputs("c1/isr", n)
    r1, s1 = lib.gf_isr(a)
    r2, s2 = chk.gf_isr(a)
    eq(s1, s2, "gf_isr status")
    eq(r1, r2, "gf_isr value")
    eq(lib.gf_invert(a), chk.gf_invert(a), "gf_invert")


def check_points(lib, chk, n):
    """BASELINE config 1 (group half): all four coordinates of add/sub/double, canonicalised"""
    p = util.random_points(chk, "c1/p", n)
    q = util.random_points(chk, "c1/q", n)
    # also feed non-trivial projective representatives (outputs of earlier group operations)
    p2 = chk.point_add(p, q)
    q2 = chk.point_double(q)
    ident = np.zeros((1, 4, 8), "<u8"); ident[0, 1, 0] = 1; ident[0, 2, 0] = 1
    ident = ident.view(np.uint8).reshape(1, 256)
    pa = np.concatenate([p, p2, ident, p[:1], ident])
    qa = np.concatenate([q, q2, ident, ident, q[:1]])
    c = util.coords_fast
    eq(c(chk, lib.point_add(pa, qa)), c(chk, chk.point_add(pa, qa)), "point_add coords")
    eq(c(chk, lib.point_sub(pa, qa)), c(chk, chk.point_sub(pa, qa)), "point_sub coords")
    eq(c(chk, lib.point_double(pa)), c(chk, chk.point_double(pa)), "point_double coords")
    eq(c(chk, lib.point_negate(pa)), c(chk, chk.point_negate(pa)), "point_negate coords")
    eq(lib.point_eq(pa, qa), chk.point_eq(pa, qa), "point_eq")
    eq(lib.point_eq(pa, pa), chk.point_eq(pa, pa), "point_eq self")
    eq(lib.point_valid(pa), chk.point_valid(pa), "point_valid")
    garbage = stream_bytes("c1/garbage", 8 * 256).reshape(8, 256) & 0x7f
    eq(lib.point_valid(garbage), chk.point_valid(garbage), "point_valid garbage")


def check_niels(lib, chk, n):
    """SURVEY 8(a) row a9, directly: pt_to_pniels / pniels_to_pt / niels_to_pt / add_niels_to_pt / sub_niels_from_pt / add_pniels_to_pt /
    sub_pniels_from_pt (goldilocks.c:271-380).  The reference keeps them static, so the expected coordinates are its formulas restated
    on Python integers below (line for line: the projective representative matters, all four coordinates are compared), and the results
    are tied to the reference itself as group elements through its exported point_add / point_sub.  Both shapes of the product's code:
    by value (ops 0-5) and on the slot machine (ops 6-9)."""
    D2 = (2 * -39082) % P                                   # 2 * TWISTED_D (goldilocks.c:45,286)
    p = util.random_points(chk, "a9/p", n)
    q = util.random_points(chk, "a9/q", n)
    p[1::2] = chk.point_add(p[1::2], q[::2][: len(p[1::2])])  # Z != 1 representatives on both sides
    q[::3] = chk.point_double(q[::3])
    which = (stream_bytes("a9/w", n).astype(np.uint32) * 7 + np.arange(n, dtype=np.uint32)) % 200   # reduced mod 80 by the library
    comb = np.frombuffer(lib.export_comb_table().tobytes(), dtype="<u8").reshape(80, 3, 8)
    comb = [[sum(int(comb[e, j, l]) << (56 * l) for l in range(8)) for j in range(3)] for e in range(80)]
    cp, cq = util.coords_fast(chk, p).reshape(n, 4, 56), util.coords_fast(chk, q).reshape(n, 4, 56)
    P4 = [[util.from_le(c) for c in row] for row in cp]
    Q4 = [[util.from_le(c) for c in row] for row in cq]

    def to_pniels(x, y, z, t):                               # goldilocks.c:280-288
        return (y - x) % P, (x + y) % P, (t * D2) % P, (2 * z) % P

    def pniels_to_pt(a, b, c, z):                            # goldilocks.c:290-301
        eu, ey = (b + a) % P, (b - a) % P
        return (z * ey) % P, (z * eu) % P, (z * z) % P, (ey * eu) % P

    def niels_to_pt(a, b, c):                                # goldilocks.c:303-313
        ey, ex = (b + a) % P, (b - a) % P
        return ex, ey, 1, (ey * ex) % P

    def add_niels(d, e, sub):                                # goldilocks.c:315-359 (before_double = 0)
        x, y, z, t = d
        ea, eb, ec = e
        if sub:
            ea, eb = eb, ea
        a = ea * (y - x) % P
        yy = eb * (x + y) % P
        xx = ec * t % P
        c, b = (a + yy) % P, (yy - a) % P
        if not sub:
            y2, a2 = (z - xx) % P, (xx + z) % P
        else:
            y2, a2 = (z + xx) % P, (z - xx) % P
        return (y2 * b) % P, (a2 * c) % P, (a2 * y2) % P, (b * c) % P

    def add_pniels(d, pn, sub):                              # goldilocks.c:361-380
        x, y, z, t = d
        return add_niels((x, y, z * pn[3] % P, t), pn[:3], sub)

    def pack(rows):
        return np.stack([np.concatenate([util.le(v) for v in r]) for r in rows])

    c = util.coords_fast
    pnq = [to_pniels(*r) for r in Q4]
    want = {0: [pniels_to_pt(*pn) for pn in pnq],
            1: [add_pniels(d, pn, False) for d, pn in zip(P4, pnq)], 2: [add_pniels(d, pn, True) for d, pn in zip(P4, pnq)],
            3: [add_niels(d, comb[w % 80], False) for d, w in zip(P4, which)], 4: [add_niels(d, comb[w % 80], True) for d, w in zip(P4, which)],
            5: [niels_to_pt(*comb[w % 80]) for w in which]}
    want[6], want[7], want[8], want[9] = want[1], want[2], want[3], want[4]
    got = {}
    for op in range(10):
        got[op] = lib.debug_niels(p, q, which, op)
        eq(c(chk, got[op]), pack(want[op]), "niels op %d coordinates" % op)
    # the same results as group elements, against the reference's own exported group law
    eq(chk.point_eq(got[0], q), np.ones(n, bool), "pniels_to_pt(pt_to_pniels(q)) == q")
    eq(chk.point_eq(got[1], chk.point_add(p, q)), np.ones(n, bool), "p + pniels(q) == point_add(p, q)")
    eq(chk.point_eq(got[7], chk.point_sub(p, q)), np.ones(n, bool), "p - pniels(q) == point_sub(p, q) (slot machine)")
    eq(chk.point_eq(chk.point_sub(got[8], got[5]), p), np.ones(n, bool), "(p + comb[e]) - niels_to_pt(comb[e]) == p (slot machine)")
    eq(chk.point_eq(chk.point_add(got[4], got[5]), p), np.ones(n, bool), "(p - comb[e]) + niels_to_pt(comb[e]) == p")
    assert chk.point_valid(got[5]).all() and chk.point_valid(got[9]).all()


def check_codec(lib, chk, n):
    """BASELINE config 5: decaf encode/decode + Elligator"""
    h = stream_bytes("c5/h", n * 112).reshape(n, 112)
    c = util.coords_fast
    pts = chk.from_hash_uniform(h)
    eq(c(chk, lib.from_hash_uniform(h)), c(chk, pts), "from_hash_uniform coords")
    eq(c(chk, lib.from_hash_nonuniform(h[:, :56])), c(chk, chk.from_hash_nonuniform(h[:, :56])), "from_hash_nonuniform coords")
    proj = chk.point_add(pts, chk.point_double(pts[::-1].copy()))
    allp = np.concatenate([pts, proj])
    ser = chk.point_encode(allp)
    eq(lib.point_encode(allp), ser, "point_encode")
    d1, s1 = lib.point_decode(ser)
    d2, s2 = chk.point_decode(ser)
    eq(s1, s2, "point_decode status (valid)")
    assert (s2 == -1).all()
    eq(c(chk, d1), c(chk, d2), "point_decode coords")
    # random strings (about a quarter decode), edge strings, identity with both flags
    rnd = np.concatenate([stream_bytes("c5/rnd", n * 56).reshape(n, 56), util.field_edge_values()])
    rnd[: n // 2, 0] &= 0xfe
    rnd[: n // 2, 55] &= 0x7f
    for allow in (False, True):
        d1, s1 = lib.point_decode(rnd, allow)
        d2, s2 = chk.point_decode(rnd, allow)
        eq(s1, s2, "point_decode status (random, allow_identity=%s)" % allow)
        ok = s2 == -1
        eq(c(chk, d1[ok]), c(chk, d2[ok]), "point_decode coords (random)")
    eq(lib.encode_like_eddsa(allp), chk.encode_like_eddsa(allp), "encode_like_eddsa")
    eq(lib.encode_like_x448(allp), chk.encode_like_x448(allp), "encode_like_x448")
    enc = chk.encode_like_eddsa(allp)
    extra = np.zeros((6, 57), np.uint8)
    extra[0] = le(1, 57); extra[1] = le(P - 1, 57); extra[2] = le(0, 57); extra[3] = le(0, 57); extra[3, 56] = 0x80
    extra[4] = le(P, 57); extra[5] = enc[0]; extra[5, 56] |= 0x01
    flip = enc.copy(); flip[:, 56] ^= 0x80
    rnd57 = stream_bytes("c5/rnd57", n * 57).reshape(n, 57); rnd57[:, 56] &= 0x80
    allenc = np.concatenate([enc, flip, extra, rnd57])
    d1, s1 = lib.decode_like_eddsa(allenc)
    d2, s2 = chk.decode_like_eddsa(allenc)
    eq(s1, s2, "decode_like_eddsa status")
    ok = s2 == -1
    eq(c(chk, d1[ok]), c(chk, d2[ok]), "decode_like_eddsa coords")


def check_elligator_inverse(lib, chk, n):
    """Elligator inverses (elligator.c:104-164): status + bytes for all 8 branches per point, and the round trip
    from_hash(recovered) == point on every success (the reference's own test, test_goldilocks.cxx:291-361)."""
    h = stream_bytes("c5/inv", n * 56).reshape(n, 56)
    ident = np.zeros((1, 256), np.uint8); ident[0, 64] = 1; ident[0, 128] = 1
    pts = np.concatenate([chk.from_hash_nonuniform(h), chk.from_hash_uniform(stream_bytes("c5/inv2", 8 * 112).reshape(8, 112)), ident])
    m = len(pts)
    total_ok = 0
    for base in range(8):
        which = ((np.arange(m) + base) % 8).astype(np.uint32)
        which[::5] += 8 * (1 + base)          # upper bits are ignored on this curve (elligator.c:113-118)
        r1, s1 = lib.invert_elligator_nonuniform(pts, which)
        r2, s2 = chk.invert_elligator_nonuniform(pts, which)
        eq(s1, s2, "invert_elligator_nonuniform status")
        eq(r1, r2, "invert_elligator_nonuniform bytes")
        ok = s2 == -1
        total_ok += int(ok.sum())
        back = lib.from_hash_nonuniform(r1[ok])
        assert lib.point_eq(back, pts[ok]).all(), "from_hash_nonuniform(invert(p)) != p"
        second = stream_bytes("c5/inv3/%d" % base, m * 56).reshape(m, 56)
        u1, t1 = lib.invert_elligator_uniform(pts, second, which)
        u2, t2 = chk.invert_elligator_uniform(pts, second, which)
        eq(t1, t2, "invert_elligator_uniform status")
        eq(u1, u2, "invert_elligator_uniform bytes")
        okk = t2 == -1
        assert lib.point_eq(lib.from_hash_uniform(u1[okk]), pts[okk]).all(), "from_hash_uniform(invert(p)) != p"
    assert total_ok > m, "too few Elligator preimages found"


def check_scalars(lib, chk, n):
    a = np.concatenate([util.random_scalars(chk, "sc/a", n), util.scalar_edge_bytes()])
    b = np.concatenate([util.random_scalars(chk, "sc/b", n), util.scalar_edge_bytes()[::-1]])
    eq(lib.scalar_add(a, b), chk.scalar_add(a, b), "scalar_add")
    eq(lib.scalar_sub(a, b), chk.scalar_sub(a, b), "scalar_sub")
    eq(lib.scalar_mul(a, b), chk.scalar_mul(a, b), "scalar_mul")
    eq(lib.scalar_halve(a), chk.scalar_halve(a), "scalar_halve")
    for ln in (0, 1, 31, 55, 56, 57, 112, 113, 114, 200):
        ser = stream_bytes("sc/long%d" % ln, max(1, 64 * ln)).reshape(64, ln) if ln else np.zeros((4, 0), np.uint8)
        if ln:
            ser[0] = 0xff
        got, want = lib.scalar_decode_long(ser, ln), chk.scalar_decode_long(ser, ln)
        eq(got, want, "scalar_decode_long len %d" % ln)
        for i in range(min(4, len(ser))):
            assert util.from_le(want[i]) == util.from_le(ser[i]) % Q
    # the two EdDSA lengths are reduced by folding at 2^448 = 4c (csrc/sc.cuh): values that make every carry ripple
    c = 2**446 - Q
    for ln in (57, 114):
        top = 2**(8 * ln)
        vals = [0, 1, Q - 1, Q, Q + 1, 2 * Q - 1, 2 * Q, 2**446 - 1, 2**446, 2**448 - 1, 2**448, 2**448 + 1, 2**448 - 4 * c, 2**448 - 4 * c - 1,
                2**448 - 4 * c + 1, top - 1, top - 2**448, top - 2**446, top - Q, (top // Q) * Q, (top // Q) * Q - 1, top - 4 * c, 2**448 + 2**264 - 1,
                2**449 - 1, 2**450 - 4 * c, (2**448 - 1) ^ (2**288 - 1), (2**448 - 1) - 2**300]
        vals += [v ^ ((1 << k) - 1) for v in (top - 1, 2**448 - 1) for k in (31, 32, 33, 224, 287, 288, 289, 415, 416, 446)]
        vals += [(top - 1) // 3, (top - 1) // 5 * 3, (top - 1) - (2**448 - 1), ((top - 1) >> 448 << 448) + 2**448 - 4 * c * ((top - 1) >> 448)]
        vals = [v % top for v in vals if v >= 0]
        ser = np.stack([le(v, ln) for v in vals])
        got = lib.scalar_decode_long(ser, ln)
        for i, v in enumerate(vals):
            assert util.from_le(got[i]) == v % Q, "scalar_decode_long (folding) len %d case %d" % (ln, i)
        eq(got, chk.scalar_decode_long(ser, ln), "scalar_decode_long edge values len %d" % ln)


def check_comb(lib, chk, n):
    """BASELINE config 2: fixed-base comb, compared as decaf and EdDSA encodings"""
    s = np.concatenate([util.random_scalars(chk, "c2/s", n), util.scalar_edge_bytes()])
    got, want = lib.precomputed_scalarmul(s), chk.precomputed_scalarmul(s)
    eq(lib.point_eq(got, want), np.ones(len(s), bool), "comb point_eq")
    eq(chk.point_encode(got), chk.point_encode(want), "comb decaf encoding")
    eq(chk.encode_like_eddsa(got), chk.encode_like_eddsa(want), "comb eddsa encoding")
    assert chk.point_valid(got).all()


def check_scalarmul(lib, chk, n):
    s = np.concatenate([util.random_scalars(chk, "sm/s", n), util.scalar_edge_bytes()])
    t = np.concatenate([util.random_scalars(chk, "sm/t", n), util.scalar_edge_bytes()[::-1]])
    p = util.random_points(chk, "sm/p", len(s))
    got, want = lib.point_scalarmul(p, s), chk.point_scalarmul(p, s)
    eq(chk.point_encode(got), chk.point_encode(want), "point_scalarmul")
    eq(chk.encode_like_eddsa(got), chk.encode_like_eddsa(want), "point_scalarmul eddsa encoding")
    got, want = lib.base_double_scalarmul_non_secret(s, p, t), chk.base_double_scalarmul_non_secret(s, p, t)
    eq(chk.point_encode(got), chk.point_encode(want), "base_double_scalarmul_non_secret")
    q = util.random_points(chk, "sm/q", len(s))
    got, want = lib.point_double_scalarmul(p, s, q, t), chk.point_double_scalarmul(p, s, q, t)
    eq(chk.point_encode(got), chk.point_encode(want), "point_double_scalarmul")


def x448_inputs(n):
    u = stream_bytes("c3/u", n * 56).reshape(n, 56)
    k = stream_bytes("c3/k", n * 56).reshape(n, 56)
    edge_u = np.stack([le(v) for v in (0, 1, P - 1, P, P + 5, 2**448 - 1, 5, P + 1, 2**447)])
    edge_k = stream_bytes("c3/ek", len(edge_u) * 56).reshape(-1, 56)
    return np.concatenate([u, edge_u]), np.concatenate([k, edge_k])


def check_x448(lib, chk, n):
    """BASELINE config 3: X448 incl. the non-canonical / low-order inputs of SURVEY.md 8(a) notes"""
    u, k = x448_inputs(n)
    o1, s1 = lib.x448(u, k)
    o2, s2 = chk.x448(u, k)
    eq(s1, s2, "x448 status")
    eq(o1, o2, "x448 output")
    assert (s2[n:n + 3] == 0).all() and (o2[n:n + 3] == 0).all()      # u in {0,1,p-1}: FAILURE and zeros
    eq(lib.x448_derive_public_key(k), chk.x448_derive_public_key(k), "x448_derive_public_key")
    base = np.zeros((len(k), 56), np.uint8); base[:, 0] = 5
    eq(lib.x448(base, k)[0], chk.x448_derive_public_key(k), "x448(base) == derive_public_key")


def check_x448_vectors(lib, vectors, iters=1000):
    """RFC 7748 iterated ladder (reference test_goldilocks.cxx:546-565)"""
    k = np.zeros((1, 56), np.uint8); k[0, 0] = 5
    u = k.copy()
    for i in range(iters):
        n, st = lib.x448(u, k)
        assert st[0] == -1
        u, k = k, n
        if i == 0:
            assert bytes(k[0]).hex() == vectors["x448_iter"]["1"]
    if iters >= 1000:
        assert bytes(k[0]).hex() == vectors["x448_iter"]["1000"]


def eddsa_case(c):
    msg = bytes.fromhex(c["msg"])
    if c["prehashed"]:
        msg = hashlib.shake_256(msg).digest(64)     # Ed448ph: PH = SHAKE256(msg, 64) (reference ed448.h prehash)
    return (np.frombuffer(bytes.fromhex(c["sk"]), np.uint8)[None], bytes.fromhex(c["pk"]), msg, c["prehashed"],
            bytes.fromhex(c["context"]), bytes.fromhex(c["sig"]))


def check_eddsa_vectors(lib, vectors):
    """RFC 8032 Ed448 x 11: public key, signature bytes, verify (reference test_goldilocks.cxx:501-543)"""
    for t, c in enumerate(vectors["eddsa"]):
        sk, pk, msg, ph, ctx, sig = eddsa_case(c)
        got_pk = lib.ed448_derive_public_key(sk)
        assert bytes(got_pk[0]) == pk, "RFC 8032 case %d: public key" % t
        got_sig = lib.ed448_sign(sk, got_pk, [msg], ph, ctx)
        assert bytes(got_sig[0]) == sig, "RFC 8032 case %d: signature" % t
        assert lib.ed448_verify(got_sig, got_pk, [msg], ph, ctx)[0] == -1, "RFC 8032 case %d: verify" % t
        assert lib.ed448_verify(got_sig, got_pk, [msg + b"x"], ph, ctx)[0] == 0
        assert lib.ed448_verify(got_sig, got_pk, [msg], not ph, ctx)[0] == 0
        assert lib.ed448_verify(got_sig, got_pk, [msg], ph, ctx + b"y")[0] == 0


def check_decaf_vectors(lib, vectors):
    """16 multiples of the base point and 16 Elligator pairs (reference test_goldilocks.cxx:665-680)"""
    want = np.stack([np.frombuffer(bytes.fromhex(x), np.uint8) for x in vectors["base_multiples"]])
    sc = np.zeros((16, 56), np.uint8); sc[:, 0] = np.arange(16)
    eq(lib.point_encode(lib.precomputed_scalarmul(sc)), want, "i*B encodings via comb")
    base, st = lib.point_decode(want[1:2])
    assert st[0] == -1
    acc = np.zeros((1, 4, 8), "<u8"); acc[0, 1, 0] = 1; acc[0, 2, 0] = 1
    acc = acc.view(np.uint8).reshape(1, 256)
    for i in range(16):
        assert bytes(lib.point_encode(acc)[0]) == bytes(want[i]), "%d*B" % i
        acc = lib.point_add(acc, base)
    d, st = lib.point_decode(want, True)
    assert (st == -1).all()
    d, st = lib.point_decode(want, False)
    assert st[0] == 0 and (st[1:] == -1).all()
    one = np.zeros((1, 56), np.uint8); one[0, 0] = 1
    assert lib.point_decode(one, True)[1][0] == 0            # decode rejects [1] (test_goldilocks.cxx:334-341)
    inp = np.stack([np.frombuffer(bytes.fromhex(x), np.uint8) for x in vectors["elligator_inputs"]])
    out = np.stack([np.frombuffer(bytes.fromhex(x), np.uint8) for x in vectors["elligator_outputs"]])
    eq(lib.point_encode(lib.from_hash_nonuniform(inp)), out, "Elligator KATs")
    patho = np.frombuffer(bytes.fromhex(vectors["elli_patho"]), np.uint8)[None]
    assert lib.point_valid(lib.from_hash_nonuniform(patho)).all()


def check_eddsa_random(lib, chk, n, label="c4"):
    """BASELINE config 4 shape: keys x messages with 1/8 corrupted; keygen/sign bytes and accept bits"""
    sig, pk, msgs, kinds = util.verify_corpus(chk, label, n)
    sk = stream_bytes(label + "/sk", n * 57).reshape(n, 57)
    good = kinds == 0
    pk0 = chk.ed448_derive_public_key(sk)
    eq(lib.ed448_derive_public_key(sk), pk0, "ed448_derive_public_key")
    clean_msgs = list(msgs)
    want = chk.ed448_verify(sig, pk, msgs)
    eq(lib.ed448_verify(sig, pk, msgs), want, "ed448_verify status")
    assert (want[good] == -1).all()
    assert (want[kinds == 5] == -1).all(), "S+q must be accepted like the reference"
    assert (want[(kinds != 0) & (kinds != 5)] == 0).all()
    # signing is deterministic: bytes must match for the untouched entries
    idx = np.flatnonzero(good)
    sub_msgs = [clean_msgs[i] for i in idx]
    eq(lib.ed448_sign(sk[idx], pk0[idx], sub_msgs), sig[idx], "ed448_sign bytes")
    for ctx, ph in ((b"ctx", False), (b"", True), (b"\xff" * 255, True)):
        m = min(len(idx), 24)
        s1 = lib.ed448_sign(sk[idx[:m]], pk0[idx[:m]], sub_msgs[:m], ph, ctx)
        eq(s1, chk.ed448_sign(sk[idx[:m]], pk0[idx[:m]], sub_msgs[:m], ph, ctx), "sign ctx/ph")
        eq(lib.ed448_verify(s1, pk0[idx[:m]], sub_msgs[:m], ph, ctx), np.full(m, -1, np.int32), "verify ctx/ph")


def check_eddsa_grouped(lib, chk, n, label="c4g", per_key=(1, 2, 3, 16, 5, 1, 40), prehashed=False, context=b""):
    """Repeated public keys (SURVEY.md 8(f)4): the batch path groups byte-identical keys and verifies them against one
    per-key table; accept bits must still be the reference's, whatever the multiplicities and the order.  Keys come with
    multiplicities cycling through `per_key`, the batch is shuffled, 1/8 of the entries are corrupted (R, S, A, message,
    S+q) and two whole groups use undecodable keys (y = 1 and a non-canonical y >= p)."""
    mult = []
    while sum(mult) < n:
        mult.append(per_key[len(mult) % len(per_key)])
    nk = len(mult)
    key_of = np.repeat(np.arange(nk), mult)[:n]
    sk = stream_bytes(label + "/sk", nk * 57).reshape(nk, 57)
    pk_k = chk.ed448_derive_public_key(sk)
    lens = stream_bytes(label + "/len", n).astype(np.int64) % 70
    blob = stream_bytes(label + "/msg", int(lens.sum()) + 1)
    offs = np.concatenate([[0], np.cumsum(lens)])
    msgs = [bytes(blob[offs[i]:offs[i + 1]]) for i in range(n)]
    pk = pk_k[key_of].copy()
    sig = chk.ed448_sign(sk[key_of], pk, msgs, prehashed, context)
    sel = stream_bytes(label + "/sel", 2 * n)
    for i in range(0, n, 8):
        kind = 1 + (i // 8) % 5
        bit = 1 << (sel[2 * i] & 7); pos = int(sel[2 * i + 1])
        if kind == 1: sig[i, pos % 57] ^= bit
        elif kind == 2: sig[i, 57 + pos % 56] ^= bit
        elif kind == 3: pk[i, pos % 57] ^= bit
        elif kind == 4:
            m = bytearray(msgs[i]) or bytearray(b"\0"); m[pos % len(m)] ^= bit; msgs[i] = bytes(m)
        else: sig[i, 57:114] = le(util.from_le(sig[i, 57:114]) + util.Q, 57)
    bad_groups = [g for g in range(nk) if 3 <= mult[g] <= 16][:2]
    for g, enc in zip(bad_groups, (le(1, 57), le(P + 2, 57))):
        pk[key_of == g] = enc
    perm = np.argsort(stream_bytes(label + "/perm", 4 * n).view("<u4")[:n], kind="stable")
    sig, pk, msgs = sig[perm], pk[perm], [msgs[i] for i in perm]
    want = chk.ed448_verify(sig, pk, msgs, prehashed, context)
    got = lib.ed448_verify(sig, pk, msgs, prehashed, context)
    eq(got, want, "ed448_verify status with repeated public keys")
    if context or prehashed:   # the context and the prehash flag are part of the challenge: without them nothing verifies
        assert (lib.ed448_verify(sig, pk, msgs) == 0).all()
    assert (want == -1).sum() > n // 2 and (want == 0).sum() >= n // 16
    return want


def check_eddsa_keyset(lib, chk, n, nkeys=11, label="c4k"):
    """Key sets (goldilocks_b200_keyset_*): tables of `nkeys` public keys built once, then several batches verified against
    them; status must equal the reference's per-signature verify with pubkeys[key_index[i]], including undecodable keys in
    the set (y = 1, y >= p), corrupted signatures / messages, S + q, and out-of-range key indices (FAILURE).  Both table layouts
    (goldilocks_b200_keyset_policy): the flat one -- a table per digit position, no doublings -- and the compact one."""
    if lib.has("goldilocks_b200_keyset_policy") and not label.endswith("/compact"):
        lib.keyset_policy(0)
        try:
            check_eddsa_keyset(lib, chk, n, nkeys, label + "/compact")
        finally:
            lib.keyset_policy(32 << 30)
    sk = stream_bytes(label + "/sk", nkeys * 57).reshape(nkeys, 57)
    keys = chk.ed448_derive_public_key(sk)
    keys[3] = le(1, 57)
    if nkeys > 7:
        keys[7] = le(P + 2, 57)
    h = lib.keyset_create(keys)
    try:
        for rnd, (ph, ctx) in enumerate(((False, b""), (True, b"keyset ctx"), (False, b"\x02" * 255))):
            kidx = (stream_bytes(label + "/kidx%d" % rnd, n).astype(np.uint32) * 7 + np.arange(n, dtype=np.uint32)) % nkeys
            lens = stream_bytes(label + "/len%d" % rnd, n).astype(np.int64) % 90
            blob = stream_bytes(label + "/msg%d" % rnd, int(lens.sum()) + 1)
            offs = np.concatenate([[0], np.cumsum(lens)])
            msgs = [bytes(blob[offs[i]:offs[i + 1]]) for i in range(n)]
            good_pk = chk.ed448_derive_public_key(sk)
            sig = chk.ed448_sign(sk[kidx], good_pk[kidx], msgs, ph, ctx)
            sel = stream_bytes(label + "/sel%d" % rnd, 2 * n)
            for i in range(0, n, 6):
                kind = (i // 6) % 4
                if kind == 0: sig[i, int(sel[2 * i]) % 57] ^= 1 << (sel[2 * i + 1] & 7)
                elif kind == 1: sig[i, 57 + int(sel[2 * i]) % 56] ^= 1 << (sel[2 * i + 1] & 7)
                elif kind == 2:
                    m = bytearray(msgs[i]) or bytearray(b"\0"); m[0] ^= 0x40; msgs[i] = bytes(m)
                else: sig[i, 57:114] = le(util.from_le(sig[i, 57:114]) + util.Q, 57)
            want = chk.ed448_verify(sig, keys[kidx], msgs, ph, ctx)
            got = lib.ed448_verify_keyset(h, kidx, sig, msgs, ph, ctx)
            eq(got, want, "ed448_verify_keyset status (round %d)" % rnd)
            assert (want == -1).sum() > n // 3 and (want == 0).sum() > n // 8
            bad = kidx.copy(); bad[::5] = nkeys + (np.arange(len(bad[::5])) % 3).astype(np.uint32) * 1000
            got = lib.ed448_verify_keyset(h, bad, sig, msgs, ph, ctx)
            assert (got[::5] == 0).all(), "out-of-range key index must fail"
            keep = np.ones(n, bool); keep[::5] = False
            eq(got[keep], want[keep], "ed448_verify_keyset status next to bad indices")
    finally:
        lib.keyset_destroy(h)


# ---- hand-made signatures around the corner cases of the R check (torsion, y = 0, y = +-1, non-canonical y) -------------
_D = -39081
_BX = 224580040295924300187604334099896036246789641632564134246125461686950415467406032909029192869357953282578032075146446173674602635247710
_BY = 298819210078481492676017930443930673437544040154080242095928241372331506189835876003536878655418784733982303233503462500531545062832660


def _ed_add(p1, p2):
    (x1, y1), (x2, y2) = p1, p2
    t = _D * x1 * x2 * y1 * y2 % P
    return ((x1 * y2 + y1 * x2) * pow(1 + t, P - 2, P) % P, (y1 * y2 - x1 * x2) * pow(1 - t, P - 2, P) % P)


def _ed_mul(k, pt):
    acc = (0, 1)
    while k:
        if k & 1:
            acc = _ed_add(acc, pt)
        pt = _ed_add(pt, pt)
        k >>= 1
    return acc


def _ed_enc(pt):
    b = bytearray(int(pt[1]).to_bytes(57, "little"))
    b[56] |= 0x80 if pt[0] & 1 else 0
    return bytes(b)


def _ed_secret(sk):
    h = bytearray(hashlib.shake_256(bytes(sk)).digest(114)[:57])
    h[0] &= 0xfc; h[55] |= 0x80; h[56] = 0
    return int.from_bytes(h, "little")


def _ed_challenge(r_enc, a_enc, msg):
    return int.from_bytes(hashlib.shake_256(b"SigEd448\0\0" + r_enc + a_enc + msg).digest(114), "little") % util.Q


def check_eddsa_adversarial(lib, chk, copies=3):
    """Signatures built by hand (plain Python Ed448 arithmetic) so that R or A carry 2- and 4-torsion, R is a small-order
    point (y = 0: the degenerate branch of the square-root-free R check; y = +-1: undecodable), R is non-canonical, or the
    low bits of the last byte are set.  Whatever the reference says is the answer; the list is repeated so that the
    grouped path (n >= 64) sees it too, and a short prefix goes through the plain path."""
    B = (_BX, _BY)
    torsion = [(0, 1), (0, P - 1), (1, 0), (P - 1, 0)]
    sigs, pks, msgs = [], [], []
    for t in range(6):
        sk = bytes(stream_bytes("adv/sk%d" % t, 57))
        s = _ed_secret(sk)
        A = _ed_mul(s, B)
        for ti, T in enumerate(torsion):
            for tj, TA in enumerate(torsion if t < 2 else torsion[:1]):
                msg = bytes(stream_bytes("adv/m%d.%d.%d" % (t, ti, tj), 5 + t))
                r = util.from_le(stream_bytes("adv/r%d.%d.%d" % (t, ti, tj), 56)) % util.Q
                a_enc = _ed_enc(_ed_add(A, TA))
                r_enc = _ed_enc(_ed_add(_ed_mul(r, B), T))
                k = _ed_challenge(r_enc, a_enc, msg)
                sigs.append(r_enc + int((r + k * s) % util.Q).to_bytes(57, "little")); pks.append(a_enc); msgs.append(msg)
        a_enc = _ed_enc(A)
        for r_pt, extra in (((1, 0), 0), ((P - 1, 0), 0), ((0, 1), 0), ((0, P - 1), 0), ((1, 0), 1), ((1, 0), 0x40)):
            msg = bytes(stream_bytes("adv/small%d" % t, 9))
            r_enc = bytearray(_ed_enc(r_pt)); r_enc[56] |= extra; r_enc = bytes(r_enc)
            k = _ed_challenge(r_enc, a_enc, msg)
            sigs.append(r_enc + int(k * s % util.Q).to_bytes(57, "little")); pks.append(a_enc); msgs.append(msg)   # r = 0: S B - k A = identity
        for y_nc in (P, P + 1):                                    # non-canonical y: the decoder must refuse
            msg = b"nc"
            r_enc = int(y_nc).to_bytes(57, "little")
            k = _ed_challenge(r_enc, a_enc, msg)
            sigs.append(r_enc + int(k * s % util.Q).to_bytes(57, "little")); pks.append(a_enc); msgs.append(msg)
    sig = np.frombuffer(b"".join(sigs), np.uint8).reshape(-1, 114).copy()
    pk = np.frombuffer(b"".join(pks), np.uint8).reshape(-1, 57).copy()
    sig, pk, msgs = np.tile(sig, (copies, 1)), np.tile(pk, (copies, 1)), msgs * copies
    want = chk.ed448_verify(sig, pk, msgs)
    assert (want == -1).any() and (want == 0).any()
    eq(lib.ed448_verify(sig, pk, msgs), want, "ed448_verify status, hand-made corner cases (grouped path)")
    eq(lib.ed448_verify(sig[:40], pk[:40], msgs[:40]), want[:40], "ed448_verify status, hand-made corner cases (plain path)")
    if lib.has("goldilocks_b200_keyset_create"):
        keys, kidx = np.unique(pk, axis=0, return_inverse=True)
        h = lib.keyset_create(keys)
        try:
            eq(lib.ed448_verify_keyset(h, kidx.reshape(-1), sig, msgs), want, "ed448_verify_keyset status, hand-made corner cases")
        finally:
            lib.keyset_destroy(h)
    if lib.has("goldilocks_ed448_verify_rlc_batch"):
        check_eddsa_rlc_adversarial(lib, chk, sig, pk, msgs, want)
    return want


def check_eddsa_rlc(lib, chk, n, label="c4r", per_key=(1, 2, 3, 16, 5, 1, 40)):
    """Random-linear-combination batch verification (SURVEY.md 8(f)3, goldilocks_ed448_verify_rlc_batch): statuses must
    be the reference's per-signature verdicts, whichever way the call went.
    (a) all signatures valid, repeated keys, S + q mixed in (the reference accepts it): the batch equation must decide
        (fast = 1);
    (b) the same batch with some R / public keys made undecodable: rejected up front, the equation still decides the rest;
    (c) one signature with a wrong S, one with a flipped message bit, one with a decodable but wrong R: the equation must
        fail and the per-signature fallback must find exactly those;
    (d) hand-made torsion / small-order corner cases: whatever the reference says."""
    _rlc_fresh(lib)
    mult = []
    while sum(mult) < n:
        mult.append(per_key[len(mult) % len(per_key)])
    nk = len(mult)
    key_of = np.repeat(np.arange(nk), mult)[:n]
    sk = stream_bytes(label + "/sk", nk * 57).reshape(nk, 57)
    pk_k = chk.ed448_derive_public_key(sk)
    lens = stream_bytes(label + "/len", n).astype(np.int64) % 70
    blob = stream_bytes(label + "/msg", int(lens.sum()) + 1)
    offs = np.concatenate([[0], np.cumsum(lens)])
    msgs = [bytes(blob[offs[i]:offs[i + 1]]) for i in range(n)]
    pk = pk_k[key_of].copy()
    sig = chk.ed448_sign(sk[key_of], pk, msgs)
    for i in range(5, n, 9):
        sig[i, 57:114] = le(util.from_le(sig[i, 57:114]) + util.Q, 57)
    perm = np.argsort(stream_bytes(label + "/perm", 4 * n).view("<u4")[:n], kind="stable")
    sig, pk, msgs = sig[perm], pk[perm], [msgs[i] for i in perm]
    # (a)
    want = chk.ed448_verify(sig, pk, msgs)
    assert (want == -1).all()
    got, fast = lib.ed448_verify_rlc(sig, pk, msgs)
    eq(got, want, "ed448_verify_rlc status, all valid")
    assert fast == 1, "an all-valid batch must be decided by the batch equation"
    # (b)
    sig_b, pk_b = sig.copy(), pk.copy()
    sig_b[3, :57] = le(1, 57)            # R: y = 1, the decoder refuses
    sig_b[10, :57] = le(P + 2, 57)       # R: non-canonical y
    pk_b[17] = le(1, 57)                 # A undecodable (its whole group when the key repeats)
    sig_b[20, 56] |= 0x01                # stray bit in the last byte of R
    want = chk.ed448_verify(sig_b, pk_b, msgs)
    assert (want[[3, 10, 17, 20]] == 0).all()
    got, fast = lib.ed448_verify_rlc(sig_b, pk_b, msgs)
    eq(got, want, "ed448_verify_rlc status, undecodable entries")
    assert (want == 0).sum() == 4
    assert fast == 1, "undecodable entries are rejected up front; the equation decides the rest"
    # (c)
    for kind in range(3):
        sig_c, msgs_c = sig.copy(), list(msgs)
        i = 7 + 11 * kind
        if kind == 0: sig_c[i, 60] ^= 4
        elif kind == 1: msgs_c[i] = msgs_c[i] + b"x"
        else: sig_c[i, :57] = sig[(i + 1) % n, :57]       # someone else's R: decodes, does not match
        want = chk.ed448_verify(sig_c, pk, msgs_c)
        assert want[i] == 0 and (want == -1).sum() == n - 1
        got, fast = lib.ed448_verify_rlc(sig_c, pk, msgs_c)
        eq(got, want, "ed448_verify_rlc status, one bad signature (kind %d)" % kind)
        assert fast != 1, "a bad signature must fail the batch equation"
    # contexts and prehash flag go through the same challenge hash
    m = min(n, 80)
    s1 = chk.ed448_sign(sk[key_of[perm][:m]], pk[:m], msgs[:m], True, b"rlc ctx")
    got, fast = lib.ed448_verify_rlc(s1, pk[:m], msgs[:m], True, b"rlc ctx")
    eq(got, np.full(m, -1, np.int32), "ed448_verify_rlc with context + prehash flag")
    if m >= 64: assert fast == 1
    got, fast = lib.ed448_verify_rlc(s1, pk[:m], msgs[:m])
    assert (got == 0).all() and fast != 1
    return want


def _rlc_fresh(lib):
    """the product remembers a call in which most chunks failed and skips the equation for a while (goldilocks_b200_rlc_policy);
    tests that expect the equation to run start from a clean slate"""
    if lib.has("goldilocks_b200_rlc_policy"):
        lib.rlc_policy(16)


def check_eddsa_rlc_adversarial(lib, chk, sig, pk, msgs, want):
    """the hand-made corner cases of check_eddsa_adversarial through the RLC entry point"""
    _rlc_fresh(lib)
    got, _ = lib.ed448_verify_rlc(sig, pk, msgs)
    eq(got, want, "ed448_verify_rlc status, hand-made corner cases")
    ok = np.flatnonzero(want == -1)
    if len(ok) >= 64:   # the accepted ones alone (torsion on R and A, small-order R): the equation must hold for them
        got, fast = lib.ed448_verify_rlc(sig[ok], pk[ok], [msgs[i] for i in ok])
        eq(got, want[ok], "ed448_verify_rlc status, accepted corner cases only")
        assert fast == 1, "torsion components vanish under the isogeny: the batch equation must hold"


def check_shake(lib, n=40):
    msgs = [bytes(stream_bytes("shake/%d" % i, i * 7)) for i in range(n)] + [b"", b"a" * 135, b"b" * 136, b"c" * 137, b"d" * 272]
    for outlen in (32, 57, 114, 136, 137, 300):
        got = lib.shake256(msgs, outlen)
        for i, m in enumerate(msgs):
            assert bytes(got[i]) == hashlib.shake_256(m).digest(outlen), "shake256 len %d out %d" % (len(m), outlen)


def check_tables(lib, chk):
    eq(lib.export_comb_table(), chk.export_comb_table(), "comb table (15360 B)")
    eq(lib.export_wnaf_table(), chk.export_wnaf_table(), "wNAF base table (6144 B)")


def check_openssl_golden(lib, g):
    """tests/golden/openssl_ed448_x448.npz (tools/openssl_vectors.py): public keys, signatures, verdicts and X448 outputs that
    RFC 8032 / RFC 7748 fix, as OpenSSL computed them on seeded inputs -- the reference's bytes, checked without the reference.
    Verify kind 5 (S + q) is left out: the reference accepts it, OpenSSL does not."""
    intact, kinds, msgs = g["kinds"] == 0, g["kinds"], (g["arena"], g["off"])
    pk = lib.ed448_derive_public_key(g["sk"])
    eq(pk[intact], g["pk"][intact], "ed448_derive_public_key vs OpenSSL")
    eq(lib.ed448_sign(g["sk"], pk, msgs)[intact], g["sig"][intact], "ed448_sign vs OpenSSL")
    st = lib.ed448_verify(g["sig"], g["pk"], msgs)
    eq(st[kinds != 5], g["status"][kinds != 5], "ed448_verify vs OpenSSL")
    out, xs = lib.x448(g["x448_u"], g["x448_k"])
    eq(out, g["x448_out"], "x448 vs OpenSSL")
    assert (xs == -1).all(), "x448 status on random inputs"


def check_widened(lib, chk, n):
    """SURVEY.md 8(f)1: the rest of the reference ABI that sits next to the hot path -- scalar_invert,
    point_dual_scalarmul, direct_scalarmul, precompute + caller-supplied comb tables, key conversions,
    debugging_torque/pscale.  Byte for byte against a checker that exports them (the reference build); against one
    that does not (the C restatement) each result is checked on its own terms instead: Python integers, SHAKE256 from
    hashlib, and identities over the checker's scalarmul and X448, which the golden vectors pin."""
    full = chk.has("goldilocks_448_scalar_invert_batch")
    c = util.coords_fast
    # scalar_invert: random + edge scalars (0 fails, like the reference)
    a = np.concatenate([util.random_scalars(chk, "w/inv", n), util.scalar_edge_bytes()])
    r1, s1 = lib.scalar_invert(a)
    if full:
        r2, s2 = chk.scalar_invert(a)
        eq(s1, s2, "scalar_invert status")
        eq(r1, r2, "scalar_invert value")
    av = [util.from_le(x) % Q for x in a]
    eq(s1, np.array([-1 if v else 0 for v in av], np.int32), "scalar_invert status (0 fails)")
    ok = s1 == -1
    eq(r1[ok], np.stack([le(pow(v, -1, Q)) for v in av if v]), "scalar_invert value vs Python integers")
    one = np.zeros(56, np.uint8); one[0] = 1
    assert (chk.scalar_mul(r1[ok], a[ok]) == one).all()
    # dual scalarmul
    m = max(8, n // 4)
    p = util.random_points(chk, "w/p", m)
    s = np.concatenate([util.random_scalars(chk, "w/s", m - 4), util.scalar_edge_bytes()[:4]])
    t = util.random_scalars(chk, "w/t", m)
    g1, g2 = lib.point_dual_scalarmul(p, s, t)
    if full:
        w1, w2 = chk.point_dual_scalarmul(p, s, t)
        eq(chk.point_encode(g1), chk.point_encode(w1), "dual_scalarmul a1")
        eq(chk.point_encode(g2), chk.point_encode(w2), "dual_scalarmul a2")
    eq(chk.point_encode(g1), chk.point_encode(chk.point_scalarmul(p, s)), "dual_scalarmul a1 == scalarmul")
    eq(chk.point_encode(g2), chk.point_encode(chk.point_scalarmul(p, t)), "dual_scalarmul a2 == scalarmul")
    # direct scalarmul: valid encodings, random strings (most fail), identity
    enc = chk.point_encode(p)
    bad = stream_bytes("w/bad", m * 56).reshape(m, 56)
    ident = np.zeros((1, 56), np.uint8)
    base = np.concatenate([enc, bad, ident])
    sc = np.concatenate([s, t, s[:1]])
    want_enc = chk.point_encode(chk.point_scalarmul(p, s))
    for allow in (False, True):
        for short in (False, True):
            o1, st1 = lib.direct_scalarmul(base, sc, allow, short, prefill=0xa5)
            if full:
                o2, st2 = chk.direct_scalarmul(base, sc, allow, short, prefill=0xa5)
                eq(st1, st2, "direct_scalarmul status allow=%s short=%s" % (allow, short))
                eq(o1, o2, "direct_scalarmul bytes allow=%s short=%s" % (allow, short))
            eq(st1[:m], np.full(m, -1, np.int32), "direct_scalarmul status of valid encodings allow=%s short=%s" % (allow, short))
            eq(o1[:m], want_enc, "direct_scalarmul == encode(scalarmul(decode)) allow=%s short=%s" % (allow, short))
    # precompute: byte-identical tables, and the comb over them
    q = p[:3]
    t1 = lib.precompute(q)
    if full:
        t2 = chk.precompute(q)
        eq(t1, t2, "precompute tables (15360 B each)")
    for k in range(len(q)):
        got = lib.precomputed_scalarmul(s, table=t1[k])
        if full:
            eq(chk.point_encode(got), chk.point_encode(chk.precomputed_scalarmul(s, table=t1[k])), "precomputed_scalarmul over a caller table")
        eq(chk.point_encode(got), chk.point_encode(chk.point_scalarmul(np.repeat(q[k:k + 1], len(s), axis=0), s)), "comb == scalarmul")
    # key conversions
    sk = stream_bytes("w/sk", n * 57).reshape(n, 57)
    pk = chk.ed448_derive_public_key(sk)
    extra = np.zeros((4, 57), np.uint8); extra[1] = le(1, 57); extra[2] = le(P - 1, 57); extra[3] = le(P + 3, 57)
    pk = np.concatenate([pk, extra, stream_bytes("w/rndpk", 16 * 57).reshape(16, 57)])
    if full:
        eq(lib.convert_public_key_to_x448(pk), chk.convert_public_key_to_x448(pk), "convert_public_key_to_x448")
        eq(lib.convert_private_key_to_x448(sk), chk.convert_private_key_to_x448(sk), "convert_private_key_to_x448")
    xs = lib.convert_private_key_to_x448(sk)
    eq(xs, np.stack([np.frombuffer(hashlib.shake_256(bytes(k)).digest(56), np.uint8) for k in sk]), "convert_private_key_to_x448 == SHAKE256(sk)[:56]")
    xpk = lib.x448_derive_public_key(xs)
    eq(xpk, chk.x448(np.tile(le(5), (n, 1)), xs)[0], "x448_derive_public_key == x448(5, k)")
    eq(xpk, lib.convert_public_key_to_x448(pk[:n]), "x448 pk of converted sk == converted ed pk")
    # debugging helpers: same group element, exact coordinates
    if full:
        eq(c(chk, lib.debugging_torque(p)), c(chk, chk.debugging_torque(p)), "debugging_torque coords")
    eq(lib.point_eq(lib.debugging_torque(p), p), np.ones(m, bool), "torque keeps the point")
    fac = np.concatenate([stream_bytes("w/fac", (m - 2) * 56).reshape(m - 2, 56), np.zeros((1, 56), np.uint8), le(P)[None]])
    if full:
        eq(c(chk, lib.debugging_pscale(p, fac)), c(chk, chk.debugging_pscale(p, fac)), "debugging_pscale coords")
    eq(lib.point_eq(lib.debugging_pscale(p, fac), p), np.ones(m, bool), "pscale keeps the point")
