"""Mechanisms that exist only on the device, each driven on purpose and compared element by element with the checker:

1. persistent scalar-multiplication kernels (k_slots_persist) past the first element of every thread, with edge scalars and
   special points spread through the batch instead of appended to it;
2. the block-shared inversion (s_block_invert4) of X448 and the comb encoders with zero cases in every subset of a quad of lanes
   {l, l+32, l+64, l+96}, in full blocks and next to the clamped lanes of a tail block;
3. point structs whose limbs use the documented range (any value below 2^60 per limb) through every entry point that loads one;
4. the `_dev` entry points, which write straight into caller memory: nothing at or past element n may change.

The limb generator of (3) is checked on Python integers in the CPU tier, and the host simulator runs the plain functors on its
output there too."""
import os
import time

import numpy as np
import pytest

import parity
import util
from util import P, Q, le, stream_bytes

FAILURE, SUCCESS = 0, -1
RADIX, CAP = 1 << 56, 1 << 60
MASK56 = RADIX - 1


# ---- (3) point structs with limbs up to 2^60 -------------------------------------------------------------------------------
def split(v):
    """radix-2^56 limbs of v, the top limb taking whatever is left (v < 2^452 keeps it below 2^60)"""
    limbs = [(v >> (56 * k)) & MASK56 for k in range(7)]
    return limbs + [v >> 392]


def value(limbs):
    return sum(int(l) << (56 * k) for k, l in enumerate(limbs))


def form_plus_kp(v, k):
    """v + k p, k <= 15"""
    return split(v + k * P)


def form_borrow(v, moves):
    """canonical limbs of v with c moved down from limb j + 1 to limb j for every (j, c) in moves: limb j gains c 2^56"""
    limbs = split(v)
    for j, c in moves:
        c = min(c, limbs[j + 1])
        limbs[j] += c << 56
        limbs[j + 1] -= c
    return limbs


def form_max(v):
    """v + 15 p with limbs 0..6 all in [15 2^56, 2^60): every limb as high as the value allows"""
    r, limbs = v + 15 * P, []
    for _ in range(7):
        l = (r & MASK56) + 15 * RADIX
        limbs.append(l)
        r = (r - l) >> 56
    return limbs + [r]


ALL_MAX = [CAP - 1] * 8
ALL_MAX_VALUE = value(ALL_MAX) % P
FORMS = ("plus_kp", "borrow_one", "borrow_all", "max", "rescaled_all_max")


def coordinate_form(v, kind, e, c):
    if kind == "plus_kp":
        return form_plus_kp(v, (e + 5 * c) % 16)
    if kind == "borrow_one":
        return form_borrow(v, [((e + c) % 7, 1 + (e + 3 * c) % 15)])
    if kind == "borrow_all":
        return form_borrow(v, [(j, 15 - (j + e + c) % 4) for j in range(7)])
    return form_max(v)


def point_form(coords, kind, e):
    """(limbs of the four coordinates, canonical values they stand for); the values are the input's except for
    rescaled_all_max, which multiplies all four by the lambda that makes X (Y for X = 0) equal to all limbs 2^60 - 1"""
    if kind == "rescaled_all_max":
        c0 = 0 if coords[0] else 1
        lam = ALL_MAX_VALUE * pow(coords[c0], -1, P) % P
        vals = [x * lam % P for x in coords]
        return [ALL_MAX if c == c0 else form_max(x) for c, x in enumerate(vals)], vals
    return [coordinate_form(x, kind, e, c) for c, x in enumerate(coords)], coords


def point_coords(pts):
    """canonical (x, y, z, t) of every point struct, as Python integers"""
    limbs = np.ascontiguousarray(pts, np.uint8).reshape(-1, 256).view("<u8").reshape(-1, 4, 8)
    return [[value(limbs[e, c]) % P for c in range(4)] for e in range(len(limbs))]


def pack_points(rows):
    """point structs from four lists of 8 limbs each"""
    return np.array(rows, dtype=np.uint64).reshape(-1, 32).view(np.uint8).reshape(-1, 256).copy()


def wide_points(pts, label):
    """(wide, canon): every point re-expressed with limbs below 2^60 in one of FORMS (chosen from the stream `label`),
    and the canonical structs of the same coordinate values -- the checker's input"""
    sel = stream_bytes(label + "/forms", len(pts))
    wide, canon = [], []
    for e, coords in enumerate(point_coords(pts)):
        limbs, vals = point_form(coords, FORMS[(int(sel[e]) + e) % len(FORMS)], e)
        wide.append(limbs)
        canon.append([split(x) for x in vals])
    return pack_points(wide), pack_points(canon)


def identity(n=1):
    pt = np.zeros((n, 4, 8), "<u8")
    pt[:, 1, 0] = 1
    pt[:, 2, 0] = 1
    return pt.view(np.uint8).reshape(n, 256).copy()


def torqued(pts):
    """p + (0, -1): (-x, -y, z, t) (goldilocks.c:675-683), canonical limbs"""
    return pack_points([[split(-x % P), split(-y % P), split(z), split(t)] for x, y, z, t in point_coords(pts)])


def test_limb_forms_keep_the_value_and_reach_2_60():
    """every form: limbs below 2^60, the same value mod p, and the shape it is named for -- on Python integers"""
    vals = [0, 1, 2, P - 1, P - 2, 2**224, 2**224 - 1, (P - 1) // 2, 2**447, RADIX - 1, RADIX]
    vals += [util.from_le(stream_bytes("limbs/v%d" % i, 56)) % P for i in range(200)]
    for i, v in enumerate(vals):
        for k in range(16):
            limbs = form_plus_kp(v, k)
            assert max(limbs) < CAP and value(limbs) == v + k * P
        for j in range(7):
            for c in (1, 7, 15):
                limbs = form_borrow(v, [(j, c)])
                assert max(limbs) < CAP and min(limbs) >= 0 and value(limbs) == v
                moved = min(c, split(v)[j + 1])
                assert limbs[j] == split(v)[j] + (moved << 56) and limbs[j + 1] == split(v)[j + 1] - moved
        limbs = form_borrow(v, [(j, 15) for j in range(7)])
        assert max(limbs) < CAP and min(limbs) >= 0 and value(limbs) == v
        if i >= 11:                                                             # random values: every limb can lend 15
            assert all(l >= 15 * RADIX for l in limbs[:7])
        limbs = form_max(v)
        assert max(limbs) < CAP and min(limbs[:7]) >= 15 * RADIX and value(limbs) % P == v
    assert value(ALL_MAX) % P == ALL_MAX_VALUE and max(ALL_MAX) == CAP - 1


def test_wide_points_are_the_same_points(chk):
    """the point-level generator: every coordinate below 2^60 per limb, each form used, the values those of `canon`, and
    `canon` the input point (the same coordinates, or all four scaled by one lambda)"""
    pts = np.concatenate([util.random_points(chk, "limbs/p", 120), identity(2), chk.point_double(util.random_points(chk, "limbs/q", 8))])
    wide, canon = wide_points(pts, "limbs/gen")
    wl = wide.view("<u8").reshape(-1, 4, 8)
    assert int(wl.max()) < CAP and int(wl.max()) == CAP - 1
    assert (wl >= RADIX).any(axis=(1, 2)).all(), "every element must use limbs above 2^56"
    for a, b, w in zip(point_coords(pts), point_coords(canon), wl):
        assert [value(w[c]) % P for c in range(4)] == b
        lam = b[1] * pow(a[1], -1, P) % P                                        # y != 0 on this curve
        assert lam and [x * lam % P for x in a] == b
    kinds = {tuple(w[0]) == tuple(ALL_MAX) or tuple(w[1]) == tuple(ALL_MAX) for w in wl}
    assert kinds == {True, False}
    assert chk.point_valid(canon).all()


def eq_enc(chk, got, want, what):
    """the same group elements: decaf and RFC 8032 encodings (the second tells torsion apart)"""
    parity.eq(chk.point_encode(got), chk.point_encode(want), what + ", decaf encoding")
    parity.eq(chk.encode_like_eddsa(got), chk.encode_like_eddsa(want), what + ", eddsa encoding")


def check_wide_points(lib, chk, n, label, heavy=True):
    """every entry point that takes a point struct, fed wide (limbs < 2^60) representatives; the expected values are the
    checker's on the canonical structs of the same coordinate values.  heavy = False stops after the plain functors; the point
    set part runs where the library has point sets"""
    c = util.coords_fast
    base = np.concatenate([util.random_points(chk, label + "/p", n - 4), identity(1)])
    base = np.concatenate([base, chk.point_add(base[:3], util.random_points(chk, label + "/r", 3))])     # Z != 1 representatives
    other = util.random_points(chk, label + "/q", n)
    other[1::3] = chk.point_double(other[1::3])
    pa, pc = wide_points(base, label + "/wp")
    qa, qc = wide_points(other, label + "/wq")
    eq = parity.eq
    eq(c(chk, lib.point_add(pa, qa)), c(chk, chk.point_add(pc, qc)), "point_add of wide limbs")
    eq(c(chk, lib.point_sub(pa, qa)), c(chk, chk.point_sub(pc, qc)), "point_sub of wide limbs")
    eq(c(chk, lib.point_double(pa)), c(chk, chk.point_double(pc)), "point_double of wide limbs")
    eq(c(chk, lib.point_negate(pa)), c(chk, chk.point_negate(pc)), "point_negate of wide limbs")
    eq(lib.point_eq(pa, qa), chk.point_eq(pc, qc), "point_eq of wide limbs")
    eq(lib.point_eq(pa, base), np.ones(n, bool), "point_eq(wide, original)")
    eq(lib.point_eq(pa[::-1].copy(), base[::-1].copy()), np.ones(n, bool), "point_eq(wide, original), reversed")
    eq(lib.point_valid(pa), np.ones(n, bool), "point_valid of wide limbs")
    eq(lib.point_encode(pa), chk.point_encode(pc), "point_encode of wide limbs")
    eq(lib.encode_like_eddsa(pa), chk.encode_like_eddsa(pc), "encode_like_eddsa of wide limbs")
    eq(lib.encode_like_x448(pa), chk.encode_like_x448(pc), "encode_like_x448 of wide limbs")
    which = (np.arange(n) % 8).astype(np.uint32)
    r1, s1 = lib.invert_elligator_nonuniform(pa, which)
    r2, s2 = chk.invert_elligator_nonuniform(pc, which)
    eq(s1, s2, "invert_elligator_nonuniform status of wide limbs")
    eq(r1, r2, "invert_elligator_nonuniform bytes of wide limbs")
    half = stream_bytes(label + "/half", n * 56).reshape(n, 56)
    u1, t1 = lib.invert_elligator_uniform(pa, half, which)
    u2, t2 = chk.invert_elligator_uniform(pc, half, which)
    eq(t1, t2, "invert_elligator_uniform status of wide limbs")
    eq(u1, u2, "invert_elligator_uniform bytes of wide limbs")
    assert (s2 == -1).sum() > n // 8
    if not heavy:
        return
    s = np.concatenate([util.random_scalars(chk, label + "/s", n - 3), np.stack([le(0), le(1), le(Q - 1)])])
    t = util.random_scalars(chk, label + "/t", n)
    want_ps, want_pt = chk.point_scalarmul(pc, s), chk.point_scalarmul(pc, t)
    eq_enc(chk, lib.point_scalarmul(pa, s), want_ps, "point_scalarmul of wide limbs")
    eq_enc(chk, lib.point_double_scalarmul(pa, s, qa, t), chk.point_double_scalarmul(pc, s, qc, t), "point_double_scalarmul of wide limbs")
    d1, d2 = lib.point_dual_scalarmul(pa, s, t)
    eq_enc(chk, d1, want_ps, "point_dual_scalarmul (first) of wide limbs")
    eq_enc(chk, d2, want_pt, "point_dual_scalarmul (second) of wide limbs")
    eq_enc(chk, lib.base_double_scalarmul_non_secret(s, pa, t), chk.base_double_scalarmul_non_secret(s, pc, t), "bdsm of wide limbs")
    # precompute: the tables hold affine niels, so a wide representative must give the canonical one's bytes
    tw, tc = lib.precompute(pa[:3]), lib.precompute(pc[:3])
    eq(tw, tc, "precompute of wide limbs")
    for k in range(3):
        got = lib.precomputed_scalarmul(s[-64:], table=tw[k])
        eq_enc(chk, got, chk.point_scalarmul(np.repeat(pc[k:k + 1], len(got), axis=0), s[-64:]), "comb over a table of a wide point")
    # torque and pscale: exact coordinates on Python integers
    cc = point_coords(pc)
    want = pack_points([[split(-x % P), split(-y % P), split(z), split(w)] for x, y, z, w in cc])
    eq(c(chk, lib.debugging_torque(pa)), c(chk, want), "debugging_torque of wide limbs")
    fac = stream_bytes(label + "/fac", n * 56).reshape(n, 56).copy()
    fac[:, 55] &= 0x7f
    fac[0] = 0
    fv = [util.from_le(f) % P or 1 for f in fac]
    want = pack_points([[split(v * f % P) for v in row] for row, f in zip(cc, fv)])
    eq(c(chk, lib.debugging_pscale(pa, fac)), c(chk, want), "debugging_pscale of wide limbs")
    if not lib.has("goldilocks_b200_pointset_create"):
        return
    # point sets: the set keeps tables of the wide points; the answers are bdsm against the canonical ones
    m = min(n, 37)
    h = lib.pointset_create(pa[:m])
    try:
        idx = (np.arange(n) * 7 % m).astype(np.uint32)
        eq_enc(chk, lib.pointset(h, idx, s, t), chk.base_double_scalarmul_non_secret(s, pc[idx], t), "point set of wide points")
    finally:
        lib.pointset_destroy(h)


def test_wide_limbs_on_the_host_simulator(sim, chk):
    """the plain functors of the CUDA sources, compiled for the host, on the wide representatives"""
    util.set_threads(sim, os.cpu_count() or 1)
    util.set_threads(chk, os.cpu_count() or 1)
    check_wide_points(sim, chk, 40, "limbs/sim")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [100, (1 << 14) + 37])
def test_wide_limbs_on_the_gpu(gpu, chk, n):
    """small n: the plain functors; n >= 2^14: the staged point rows; the scalar multiplications: the slot machine"""
    util.set_threads(chk, os.cpu_count() or 1)
    check_wide_points(gpu, chk, n, "limbs/gpu%d" % n)


# ---- (2) edge elements at every lane position of the block-shared inversion --------------------------------------------------
QUAD_LANES = (0, 1, 31)


def quad_mask():
    """48 full blocks of 128: block 16 i + s has its edge cases at lanes l + 32 w for the w in subset s of {0, 1, 2, 3},
    l = QUAD_LANES[i] -- all 16 subsets of one quad of s_block_invert4, for three lane indices"""
    mask = np.zeros(len(QUAD_LANES) * 16 * 128, bool)
    for i, l in enumerate(QUAD_LANES):
        for s in range(16):
            for w in range(4):
                if s >> w & 1:
                    mask[128 * (16 * i + s) + l + 32 * w] = True
    return mask


TAILS = (1, 31, 33, 65, 97, 127)


def tail_masks():
    """(r, mask) for batches of 128 + r: a full block, then a tail whose live lanes 0..r-1 share quads with clamped lanes
    (which repeat element n - 1); in the second mask of each r the last element is an edge case too, so the clamped lanes are"""
    for r in TAILS:
        for v in (0, 1):
            mask = np.zeros(128 + r, bool)
            mask[:128] = np.arange(128) % 5 == v
            mask[128:] = np.arange(r) % 3 == v
            if v:
                mask[-1] = True
            yield r, mask


def fill(mask, edges, rnd):
    """rnd with the edge rows put, cycling, at the positions of mask"""
    out = rnd.copy()
    pos = np.flatnonzero(mask)
    out[pos] = edges[np.arange(len(pos)) % len(edges)]
    return out


def lane_batches(label, width):
    """(name, mask, random rows) for the full-block layout and every tail layout"""
    m = quad_mask()
    yield "full blocks", m, stream_bytes(label + "/full", len(m) * width).reshape(-1, width)
    for r, mask in tail_masks():
        yield "tail %d, last %s" % (r, "edge" if mask[-1] else "random"), mask, stream_bytes("%s/%d/%d" % (label, r, mask[-1]), len(mask) * width).reshape(-1, width)


@pytest.mark.gpu
def test_x448_zero_outputs_in_every_quad_subset(gpu, chk):
    """u in {0, 1, p - 1, p, p + 1} (the checker decides which give zero) at every subset of a quad of lanes"""
    edges = np.stack([le(v) for v in (0, 1, P - 1, P, P + 1)])
    for name, mask, rnd in lane_batches("quad/x448/u", 56):
        u = fill(mask, edges, rnd)
        k = stream_bytes("quad/x448/k/" + name, len(u) * 56).reshape(-1, 56)
        o1, s1 = gpu.x448(u, k)
        o2, s2 = chk.x448(u, k)
        assert (s2[mask] == FAILURE).all() and (s2[~mask] == SUCCESS).all(), name
        parity.eq(s1, s2, "x448 status, " + name)
        parity.eq(o1, o2, "x448 output, " + name)


def twist_u(label, count):
    out, j = [], 0
    while len(out) < count:
        u = util.from_le(stream_bytes("%s/%d" % (label, j), 56)) % P
        j += 1
        if pow((u * u * u + 156326 * u * u + u) % P, (P - 1) // 2, P) == P - 1:
            out.append(u)
    return out


@pytest.mark.gpu
def test_x448_peerset_zero_outputs_in_every_quad_subset(gpu, chk):
    """missing peers and ladder peers that give zero (u = 0, 1, p - 1) at every subset of a quad, next to comb peers and a
    ladder peer on the twist"""
    honest = chk.x448_derive_public_key(stream_bytes("quad/peer/sk", 4 * 56).reshape(4, 56))
    peers = np.concatenate([honest, np.stack([le(v) for v in (0, 1, P - 1, twist_u("quad/peer/twist", 1)[0])])])
    m = len(peers)
    zero_idx = np.array([4, 5, 6, m, 2**32 - 1], np.uint32)
    h = gpu.x448_peerset_create(peers)
    try:
        for name, mask, rnd in lane_batches("quad/peer/i", 4):
            live = np.array([0, 1, 2, 3, 7], np.uint32)[rnd.view("<u4").ravel() % 5]
            idx = fill(mask, zero_idx, live)
            k = stream_bytes("quad/peer/k/" + name, len(idx) * 56).reshape(-1, 56)
            got, st = gpu.x448_peerset(h, idx, k)
            ok = idx < m
            want, wst = chk.x448(peers[np.where(ok, idx, 0)], k)
            want[~ok], wst[~ok] = 0, FAILURE
            assert (wst[mask] == FAILURE).all() and (wst[~mask] == SUCCESS).all(), name
            parity.eq(st, wst, "x448 peer set status, " + name)
            parity.eq(got, want, "x448 peer set output, " + name)
    finally:
        gpu.x448_peerset_destroy(h)


@pytest.mark.gpu
def test_comb_paths_with_edge_scalars_in_every_quad_subset(gpu, chk):
    """the comb encoder of x448_derive_public_key (its inversion is block-shared too) and precomputed_scalarmul, with edge
    scalars at every subset of a quad"""
    raw = np.stack([le(0), np.full(56, 0xff, np.uint8), le(4 * Q), le(4 * Q + 4), le(1)])
    sc = np.stack([le(v) for v in (0, 1, Q - 1, Q - 2, 2**445)])
    for name, mask, rnd in lane_batches("quad/comb", 56):
        k = fill(mask, raw, rnd)
        parity.eq(gpu.x448_derive_public_key(k), chk.x448_derive_public_key(k), "x448_derive_public_key, " + name)
        s = fill(mask, sc, chk.scalar_decode_long(rnd, 56))
        got, want = gpu.precomputed_scalarmul(s), chk.precomputed_scalarmul(s)
        parity.eq(chk.point_encode(got), chk.point_encode(want), "precomputed_scalarmul, " + name)
        parity.eq(chk.encode_like_eddsa(got), chk.encode_like_eddsa(want), "precomputed_scalarmul eddsa encoding, " + name)


# ---- (1) persistent threads past their first element -----------------------------------------------------------------------
def persistent_n():
    """3 x SMs x 2048 (the most resident threads an sm_100 SM holds) + a ragged tail: whatever occupancy the library picks,
    every thread of a persistent kernel takes at least three elements"""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return 3 * sms * 2048 + 77, sms


def edge_positions(n, sms, label):
    """chunk starts and ends (i = 0, 31 mod 32), block edges, multiples of SMs x 128 (where a second pass over the grid starts
    for every occupancy), the first and last elements and random positions"""
    pos = {0, 1, n - 1, n - 2, n - 32, n - 33}
    for b in (0, 32, 4096, n // 2 - n // 2 % 128, n - 77 - 128):
        pos.update(b + o for o in (0, 1, 31, 32, 63, 64, 95, 96, 127))
    for j in range(1, 25):
        pos.update((sms * 128 * j + o) for o in (-1, 0, 31))
    pos.update(int(x) % n for x in stream_bytes(label, 8 * 96).view("<u8"))
    return np.array(sorted(p for p in pos if 0 <= p < n))


def spread(rows, pos, edges, shift):
    out = rows.copy()
    out[pos] = edges[(np.arange(len(pos)) + shift) % len(edges)]
    return out


@pytest.fixture(scope="module")
def persistent_batch(gpu, chk):
    util.set_threads(chk, os.cpu_count() or 1)
    return make_persistent_batch(chk, *persistent_n())


def make_persistent_batch(chk, n, sms):
    """one batch of scalars, points and encodings with the edge cases spread through it"""
    pos = edge_positions(n, sms, "persist/pos")
    pool = util.random_points(chk, "persist/pool", 4096)
    pool[1::2] = chk.point_add(pool[1::2], pool[::2])                          # Z != 1 representatives
    pick = stream_bytes("persist/pick", 8 * n).view("<u8")
    p = pool[pick % 4096]
    q = pool[(pick >> 20) % 4096]
    specials = np.concatenate([identity(2), torqued(pool[:3]), wide_points(pool[3:9], "persist/wide")[0]])
    p = spread(p, pos, specials, 0)
    q = spread(q, pos, specials, 3)
    edge_s = np.stack([le(v) for v in (0, 1, Q - 1, Q - 2, 2**445)])
    s = spread(chk.scalar_decode_long(stream_bytes("persist/s", n * 56).reshape(n, 56), 56), pos, edge_s, 0)
    t = spread(chk.scalar_decode_long(stream_bytes("persist/t", n * 56).reshape(n, 56), 56), pos, edge_s, 2)
    t0 = spread(t, pos[::3], np.stack([le(0)]), 0)                             # scalar2 = 0 for bdsm
    enc_pool = chk.point_encode(pool)
    enc = enc_pool[pick % 4096]
    bad = stream_bytes("persist/bad", 4 * 56).reshape(4, 56)
    edge_e = np.concatenate([np.zeros((1, 56), np.uint8), le(P + 1)[None], le(1)[None], bad, enc_pool[:2]])
    enc = spread(enc, pos, edge_e, 0)
    return {"n": n, "p": p, "q": q, "s": s, "t": t, "t0": t0, "enc": enc}


def _report(what, secs, n):
    print("[device-paths] %s: %.2f s for %d elements" % (what, secs, n))


def run_forward_and_reversed(call, arrays, what, n):
    """call(*arrays) and call(*reversed arrays): returns the forward outputs after checking that the reversed batch gives the
    same bytes element by element"""
    t0 = time.time()
    fwd = call(*arrays)
    _report(what + " (GPU call)", time.time() - t0, n)
    rev = call(*[a[::-1].copy() for a in arrays])
    fwd_t = fwd if isinstance(fwd, tuple) else (fwd,)
    rev_t = rev if isinstance(rev, tuple) else (rev,)
    for k, (a, b) in enumerate(zip(fwd_t, rev_t)):
        parity.eq(a, b[::-1], "%s: reversed batch, output %d" % (what, k))
    return fwd


@pytest.mark.gpu
def test_persistent_scalarmul_past_the_first_element(gpu, chk, persistent_batch):
    check_persistent_scalarmul(gpu, chk, persistent_batch)


@pytest.mark.gpu
def test_persistent_bdsm_past_the_first_element(gpu, chk, persistent_batch):
    check_persistent_bdsm(gpu, chk, persistent_batch)


@pytest.mark.gpu
def test_persistent_direct_scalarmul_past_the_first_element(gpu, chk, persistent_batch):
    check_persistent_direct_scalarmul(gpu, chk, persistent_batch)


def checked(what, n, fn):
    """the checker's answer for all n elements, timed"""
    t0 = time.time()
    out = fn()
    _report(what + " (checker, all host cores)", time.time() - t0, n)
    return out


def check_persistent_scalarmul(gpu, chk, b):
    n, p, q, s, t = b["n"], b["p"], b["q"], b["s"], b["t"]
    ps = checked("point_scalarmul", n, lambda: chk.point_scalarmul(p, s))
    eq_enc(chk, run_forward_and_reversed(gpu.point_scalarmul, (p, s), "point_scalarmul", n), ps, "point_scalarmul vs checker")
    want = checked("point_double_scalarmul", n, lambda: chk.point_double_scalarmul(p, s, q, t))
    eq_enc(chk, run_forward_and_reversed(gpu.point_double_scalarmul, (p, s, q, t), "point_double_scalarmul", n), want, "point_double_scalarmul vs checker")
    g1, g2 = run_forward_and_reversed(gpu.point_dual_scalarmul, (p, s, t), "point_dual_scalarmul", n)
    eq_enc(chk, g1, ps, "point_dual_scalarmul (first) vs checker")
    eq_enc(chk, g2, chk.point_scalarmul(p, t), "point_dual_scalarmul (second) vs checker")


def check_persistent_bdsm(gpu, chk, b):
    n, s, p, t0 = b["n"], b["s"], b["p"], b["t0"]
    want = checked("base_double_scalarmul_non_secret", n, lambda: chk.base_double_scalarmul_non_secret(s, p, t0))
    got = run_forward_and_reversed(gpu.base_double_scalarmul_non_secret, (s, p, t0), "base_double_scalarmul_non_secret", n)
    eq_enc(chk, got, want, "base_double_scalarmul_non_secret vs checker")


def check_persistent_direct_scalarmul(gpu, chk, b):
    """goldilocks.c:888-903: decode (the base point when it fails), scalarmul, encode; short-circuited elements keep the
    caller's bytes"""
    n, enc, s = b["n"], b["enc"], b["s"]
    base_pt = chk.precomputed_scalarmul(le(1)[None])
    scaled = {}
    for allow in (False, True):
        d, st = chk.point_decode(enc, allow)
        ok = st == SUCCESS
        d[~ok] = base_pt
        scaled[allow] = (checked("direct_scalarmul", n, lambda: chk.point_encode(chk.point_scalarmul(d, s))), st)
        assert ok.any() and (~ok).any()
    for allow in (False, True):
        for short in (False, True):
            what = "direct_scalarmul allow_identity=%s short_circuit=%s" % (allow, short)
            o, st = run_forward_and_reversed(lambda e, k: gpu.direct_scalarmul(e, k, allow, short, prefill=0x5a), (enc, s), what, n)
            want, wst = scaled[allow]
            want = want.copy()
            if short:
                want[wst != SUCCESS] = 0x5a
            parity.eq(st, wst, what + " status vs checker")
            parity.eq(o, want, what + " bytes vs checker")


# ---- (4) `_dev` entry points leave elements >= n alone -----------------------------------------------------------------------
DEV_NS = (1, 127, 128, 129, 4095)
PAD = 64
CANARY = 0xA5


@pytest.fixture(scope="module")
def dev_env(gpu, chk):
    import torch
    from libgoldilocks_b200.engine import DeviceEngine
    util.set_threads(chk, os.cpu_count() or 1)
    nmax = max(DEV_NS)
    env = {"eng": DeviceEngine(), "torch": torch}
    sig, pk, msgs, kinds = util.verify_corpus(chk, "devpad/v", nmax)
    env.update(sig=sig, pk=pk, msgs=msgs)
    keys = np.unique(pk[: nmax // 2], axis=0)
    env["keys"] = keys
    env["kidx"] = (np.arange(nmax) * 5 % (len(keys) + 3)).astype(np.uint32)     # some beyond the set
    env["u"] = stream_bytes("devpad/u", nmax * 56).reshape(nmax, 56)
    env["k"] = stream_bytes("devpad/k", nmax * 56).reshape(nmax, 56)
    env["s"] = util.random_scalars(chk, "devpad/s", nmax)
    env["t"] = util.random_scalars(chk, "devpad/t", nmax)
    env["p"] = util.random_points(chk, "devpad/p", nmax)
    env["q"] = util.random_points(chk, "devpad/q", nmax)
    env["enc"] = np.concatenate([chk.point_encode(env["p"][: nmax - 100]), stream_bytes("devpad/bad", 100 * 56).reshape(100, 56)])
    env["peers"] = np.concatenate([chk.x448_derive_public_key(stream_bytes("devpad/peers", 6 * 56).reshape(6, 56)), le(0)[None]])
    env["pidx"] = (np.arange(nmax) * 3 % 9).astype(np.uint32)
    env["dpeers"] = np.concatenate([env["enc"][:5], env["enc"][-2:]])
    return env


def _padded(torch, n, width, dtype=None):
    """a device buffer of (n + PAD) rows of `width` bytes filled with the canary, and the n-row view handed to the call"""
    buf = torch.full(((n + PAD) * width,), CANARY, dtype=torch.uint8, device="cuda")
    return buf, buf[: n * width] if dtype is None else buf[: n * width].view(dtype)


def _dev_in(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a).reshape(-1).view(np.uint8)).cuda()


def _check_padded(buf, n, width, want, what):
    got = buf.cpu().numpy().reshape(n + PAD, width)
    tail = np.flatnonzero((got[n:] != CANARY).any(axis=1))
    assert len(tail) == 0, "%s n=%d: element %d past n was written" % (what, n, n + tail[0])
    parity.eq(got[:n], np.ascontiguousarray(want).reshape(n, width), "%s n=%d: elements below n vs the host-pointer call" % (what, n))


@pytest.mark.gpu
@pytest.mark.parametrize("n", DEV_NS)
def test_dev_entry_points_write_nothing_past_n(gpu, dev_env, n):
    from libgoldilocks_b200.capi import pack_messages
    e = dev_env
    eng, torch = e["eng"], e["torch"]
    I = lambda a: _dev_in(torch, a)
    i32 = torch.int32
    sig, pk, msgs = e["sig"][:n], e["pk"][:n], e["msgs"][:n]
    arena, off = pack_messages(msgs)
    d_sig, d_pk, d_msg, d_off = I(sig), I(pk), I(arena), I(np.asarray(off).view(np.int64))
    d_off = d_off.view(torch.int64)
    u, k, s, t, p, q, enc = (e[x][:n] for x in ("u", "k", "s", "t", "p", "q", "enc"))

    # verify
    buf, st = _padded(torch, n, 4, i32)
    scratch = torch.empty(eng.verify_scratch_bytes(n), dtype=torch.uint8, device="cuda")
    eng.ed448_verify(st, d_sig, d_pk, d_msg, d_off, scratch)
    _check_padded(buf, n, 4, gpu.ed448_verify(sig, pk, msgs).view(np.uint8), "ed448_verify_batch_dev")
    # key sets: by index and by lookup
    h = gpu.keyset_create(e["keys"])
    try:
        kidx = e["kidx"][:n]
        scratch = torch.empty(eng.keyset_scratch_bytes(n, len(arena)), dtype=torch.uint8, device="cuda")
        buf, st = _padded(torch, n, 4, i32)
        eng.ed448_verify_keyset(st, h, I(kidx).view(i32), d_sig, d_msg, d_off, scratch)
        _check_padded(buf, n, 4, gpu.ed448_verify_keyset(h, kidx, sig, msgs).view(np.uint8), "ed448_verify_keyset_batch_dev")
        buf, st = _padded(torch, n, 4, i32)
        ibuf, ki = _padded(torch, n, 4, i32)
        eng.ed448_verify_keyset_lookup(st, ki, h, d_sig, d_pk, d_msg, d_off, scratch)
        wst, widx = gpu.ed448_verify_keyset_lookup(h, sig, pk, msgs, return_index=True)
        torch.cuda.synchronize()
        _check_padded(buf, n, 4, wst.view(np.uint8), "ed448_verify_keyset_lookup_batch_dev status")
        _check_padded(ibuf, n, 4, widx.view(np.uint8), "ed448_verify_keyset_lookup_batch_dev key_index")
    finally:
        gpu.keyset_destroy(h)
    # X448 and X448 peer sets
    wo, ws = gpu.x448(u, k)
    obuf, out = _padded(torch, n, 56)
    sbuf, st = _padded(torch, n, 4, i32)
    eng.x448(out, st, I(u), I(k))
    _check_padded(obuf, n, 56, wo, "x448_batch_dev output")
    _check_padded(sbuf, n, 4, ws.view(np.uint8), "x448_batch_dev status")
    h = gpu.x448_peerset_create(e["peers"])
    try:
        pidx = e["pidx"][:n]
        wo, ws = gpu.x448_peerset(h, pidx, k)
        obuf, out = _padded(torch, n, 56)
        sbuf, st = _padded(torch, n, 4, i32)
        eng.x448_peerset(out, st, h, I(pidx).view(i32), I(k))
        _check_padded(obuf, n, 56, wo, "x448_peerset_batch_dev output")
        _check_padded(sbuf, n, 4, ws.view(np.uint8), "x448_peerset_batch_dev status")
    finally:
        gpu.x448_peerset_destroy(h)
    # decaf peer sets (scaled is read: short-circuited elements keep the canary)
    h = gpu.decaf_peerset_create(e["dpeers"])
    try:
        pidx = e["pidx"][:n]
        scratch = torch.empty(eng.decaf_peerset_scratch_bytes(n), dtype=torch.uint8, device="cuda")
        wo, ws = gpu.decaf_peerset(h, pidx, s, True, prefill=CANARY)
        obuf, out = _padded(torch, n, 56)
        sbuf, st = _padded(torch, n, 4, i32)
        eng.decaf_peerset(out, st, h, I(pidx).view(i32), I(s), scratch)
        _check_padded(obuf, n, 56, wo, "direct_scalarmul_peerset_batch_dev output")
        _check_padded(sbuf, n, 4, ws.view(np.uint8), "direct_scalarmul_peerset_batch_dev status")
    finally:
        gpu.decaf_peerset_destroy(h)
    # point sets
    h = gpu.pointset_create(e["p"][:5])
    try:
        pidx = e["pidx"][:n] % 7
        scratch = torch.empty(eng.pointset_scratch_bytes(n), dtype=torch.uint8, device="cuda")
        obuf, out = _padded(torch, n, 256)
        eng.pointset(out, h, I(pidx).view(i32), I(s), I(t), scratch)
        _check_padded(obuf, n, 256, gpu.pointset(h, pidx, s, t), "base_double_scalarmul_non_secret_pointset_batch_dev")
    finally:
        gpu.pointset_destroy(h)
    # comb, field and group
    obuf, out = _padded(torch, n, 256)
    eng.precomputed_scalarmul(out, I(s))
    _check_padded(obuf, n, 256, gpu.precomputed_scalarmul(s), "precomputed_scalarmul_batch_dev")
    obuf, out = _padded(torch, n, 56)
    eng.gf_mul(out, I(u), I(k))
    _check_padded(obuf, n, 56, gpu.gf_mul(u, k), "gf_mul_batch_dev")
    obuf, out = _padded(torch, n, 256)
    eng.point_add(out, I(p), I(q))
    _check_padded(obuf, n, 256, gpu.point_add(p, q), "point_add_batch_dev")
    obuf, out = _padded(torch, n, 256)
    eng.point_double(out, I(p))
    _check_padded(obuf, n, 256, gpu.point_double(p), "point_double_batch_dev")
    wd, wds = gpu.point_decode(enc)
    obuf, out = _padded(torch, n, 256)
    sbuf, st = _padded(torch, n, 4, i32)
    eng.point_decode(out, st, I(enc))
    _check_padded(sbuf, n, 4, wds.view(np.uint8), "point_decode_batch_dev status")
    _check_padded(obuf, n, 256, wd, "point_decode_batch_dev points")
    obuf, out = _padded(torch, n, 56)
    eng.point_encode(out, I(p))
    _check_padded(obuf, n, 56, gpu.point_encode(p), "point_encode_batch_dev")
    torch.cuda.synchronize()
