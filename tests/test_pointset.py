"""Point sets (goldilocks_b200_pointset_*, goldilocks_448_base_double_scalarmul_non_secret_pointset_batch[_dev]): every output must be
the group element goldilocks_448_base_double_scalarmul_non_secret(s1, points[point_index[i]], s2) returns -- the same encoding, and
the same point (torsion included) as the library's own window evaluation -- for random points, the base point, the identity, points
with a torsion component and points passed with non-canonical limbs; random and edge scalars in both positions (scalar2 = 0 keeps
the reference's identity quirk); out-of-range indices (the identity); both table layouts; and batches in any order."""
import os

import numpy as np
import pytest

import util
from util import stream_bytes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = 2**448 - 2**224 - 1
DEFAULT_POLICY = 32 << 30                     # goldilocks_b200_keyset_policy's default: sets up to 93 000 points are flat
P_LIMBS = np.array([(P >> (56 * k)) & ((1 << 56) - 1) for k in range(8)], np.uint64)


def identity_struct():
    e = np.zeros(256, np.uint8)
    e.view("<u8")[8] = 1    # Y limb 0
    e.view("<u8")[16] = 1   # Z limb 0
    return e


def plus_p(pt, coord):
    """the same point with coordinate `coord` (0..3 = X, Y, Z, T) passed as its value + p: every limb stays below 2^57"""
    q = np.ascontiguousarray(pt, np.uint8).copy()
    limbs = q.view("<u8").reshape(4, 8)
    limbs[coord] += P_LIMBS
    return q


def corner_points(chk, tlib, label):
    """(points (40,256), kinds): random points, the base point, the identity, points plus a torsion component (tlib's
    debugging_torque), points with non-canonical limbs (one coordinate + p, or all four)"""
    rnd = util.random_points(chk, label + "/pts", 32)
    base = chk.precomputed_scalarmul(util.le(1)[None])[0]
    rows, kinds = [r for r in rnd[:20]], ["random"] * 20
    rows.append(base); kinds.append("base")
    rows.append(identity_struct()); kinds.append("identity")
    for r in tlib.debugging_torque(rnd[20:26]):
        rows.append(r); kinds.append("torsion")
    for j, r in enumerate(rnd[26:32]):
        q = r
        for c in ((j % 4,) if j < 4 else range(4)):
            q = plus_p(q, c)
        rows.append(q); kinds.append("noncanonical")
    rows.append(plus_p(base, 1)); kinds.append("noncanonical")
    tq = tlib.debugging_torque(rnd[:1])[0]
    rows.append(plus_p(tq, 2)); kinds.append("noncanonical")
    rows.extend(rnd[:4]); kinds.extend(["random"] * 4)   # repeated points
    return np.stack(rows).astype(np.uint8), kinds


SUBSETS = {0: [], 1: [0], 7: [0, 20, 21, 22, 26, 28, 32]}   # the 7-point set mixes every kind


def corner_scalars(chk, label, n):
    """(s1, s2): random scalars with the edge scalars threaded through both positions, and s1 = 0, s2 = 0 and both = 0"""
    s1 = util.random_scalars(chk, label + "/s1", n)
    s2 = util.random_scalars(chk, label + "/s2", n)
    e = util.scalar_edge_bytes()
    for j, row in enumerate(e):
        s1[j::29] = row
        s2[(3 + 2 * j)::37] = row
    s1[5::23] = 0
    s2[11::19] = 0
    s1[13::41] = 0
    s2[13::41] = 0
    return s1, s2


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


def operands(points, idx):
    """the point each element multiplies: points[idx], the identity for idx >= m"""
    ext = np.concatenate([points.reshape(-1, 256), identity_struct()[None]])
    return ext[np.minimum(idx, len(points)).astype(np.int64)]


def affine_ints(pts):
    return [tuple(util.from_le(r[56 * c:56 * (c + 1)]) for c in range(4)) for r in util.coords(None, pts)]


def assert_same_points_exact(got, want, label):
    """same affine (x/z, y/z), in Python integers: the same point, not merely the same decaf element; and T Z == X Y"""
    for j, ((x, y, z, t), (x2, y2, z2, _)) in enumerate(zip(affine_ints(got), affine_ints(want))):
        assert z != 0 and x * z2 % P == x2 * z % P and y * z2 % P == y2 * z % P, "%s: element %d is another point" % (label, j)
        assert t * z % P == x * y % P, "%s: element %d has T Z != X Y" % (label, j)


def coord_bytes(pts):
    """(n, 4, 56) bytes of X, Y, Z, T of point structs whose limbs are all below 2^56 (canonical outputs)"""
    limbs = np.ascontiguousarray(pts, np.uint8).reshape(-1, 4, 8, 8)
    assert (limbs[..., 7] == 0).all(), "a limb is not below 2^56"
    return np.ascontiguousarray(limbs[..., :7]).reshape(-1, 4, 56)


def assert_same_points_fast(lib, got, want, label):
    """assert_same_points_exact through lib.gf_mul, for large batches"""
    a, b = coord_bytes(got), coord_bytes(want)
    for c in (0, 1):
        l, r = lib.gf_mul(a[:, c], b[:, 2]), lib.gf_mul(b[:, c], a[:, 2])
        bad = np.nonzero((l != r).any(axis=1))[0]
        assert len(bad) == 0, "%s: %d elements are other points, first %d" % (label, len(bad), bad[0])
    assert (lib.gf_mul(a[:, 3], a[:, 2]) == lib.gf_mul(a[:, 0], a[:, 1])).all(), "%s: T Z != X Y" % label


def check_set(lib, chk, exact_ref, points, idx, s1, s2, label, exact="ints"):
    """one set: encodings against the checker's base_double_scalarmul_non_secret (the original reference build where it is
    present), the exact point against exact_ref's, point_valid on every output"""
    h = lib.pointset_create(points)
    try:
        assert lib.pointset_size(h) == len(points)
        got = lib.pointset(h, idx, s1, s2)
    finally:
        lib.pointset_destroy(h)
    ops = operands(points, idx)
    want = chk.base_double_scalarmul_non_secret(s1, ops, s2)
    ge, we = chk.point_encode(got), chk.point_encode(want)
    bad = np.nonzero((ge != we).any(axis=1))[0]
    assert len(bad) == 0, "%s: %d encodings differ, first at %d (index %d)" % (label, len(bad), bad[0], idx[bad[0]])
    assert chk.point_valid(got).all(), "%s: an output fails point_valid" % label
    ref = exact_ref.base_double_scalarmul_non_secret(s1, ops, s2)
    if exact == "ints":
        assert_same_points_exact(got, ref, label)
    else:
        assert_same_points_fast(exact_ref, got, ref, label)
    return got


def run_corners(lib, chk, exact_ref, n, label, exact="ints"):
    points, kinds = corner_points(chk, exact_ref, label)
    sets = dict(SUBSETS)
    sets[len(points)] = list(range(len(points)))
    for m, rows in sets.items():
        pts = points[np.array(rows, np.int64)] if m else points[:0]
        s1, s2 = corner_scalars(chk, "%s/%d" % (label, m), n)
        idx = corner_indices("%s/%d" % (label, m), n, m)
        check_set(lib, chk, exact_ref, pts, idx, s1, s2, "%s m=%d" % (label, m), exact)


# ---- CPU tier: the device functors compiled for the host (tests/hostsim/pointset.cpp) -------------------------------------------
@pytest.fixture(scope="module")
def psim():
    """the point-set entry points on the host simulator: tests/hostsim/_hostsim_pointset.so (`make hostsim`)"""
    from libgoldilocks_b200.capi import BatchLib
    path = os.path.join(ROOT, "tests", "hostsim", "_hostsim_pointset.so")
    if not os.path.exists(path):
        pytest.skip("tests/hostsim/_hostsim_pointset.so is not built (make hostsim)")
    lib = BatchLib(path)
    util.set_threads(lib, os.cpu_count() or 4)
    return lib


@pytest.fixture(params=["flat", "compact"])
def layout(request, psim):
    psim.keyset_policy(DEFAULT_POLICY if request.param == "flat" else 0)
    yield request.param
    psim.keyset_policy(DEFAULT_POLICY)


def test_pointset_layout_follows_the_keyset_policy(psim, chk, layout):
    import ctypes as C
    h = psim.pointset_create(util.random_points(chk, "pts/layout", 3))
    try:
        psim.lib.hostsim_pointset_flat.restype = C.c_int
        assert psim.lib.hostsim_pointset_flat(h) == (1 if layout == "flat" else 0)
    finally:
        psim.pointset_destroy(h)


def test_pointset_matches_base_double_scalarmul_on_the_host_simulator(psim, sim, chk, layout):
    util.set_threads(sim, os.cpu_count() or 4)
    util.set_threads(chk, os.cpu_count() or 4)
    run_corners(psim, chk, sim, 320, "pts/sim/" + layout)


def test_pointset_edge_scalars_against_every_point_kind(psim, sim, chk, layout):
    """every pair of edge scalars (0, 1, q - 1, the recoding's carry points, ...) against every one of the 40 points"""
    points, _ = corner_points(chk, sim, "pts/edge")
    e = util.scalar_edge_bytes()
    pairs = len(e) * len(e)
    idx = np.repeat(np.arange(len(points), dtype=np.uint32), pairs)
    s1 = np.tile(np.repeat(e, len(e), axis=0), (len(points), 1))
    s2 = np.tile(np.tile(e, (len(e), 1)), (len(points), 1))
    check_set(psim, chk, sim, points, idx, s1, s2, "edge scalars " + layout)


def test_pointset_order_does_not_change_the_results(psim, sim, chk, layout):
    """the call sorts by point internally: a shuffled batch, permuted back, is byte-identical to the sorted one"""
    points, _ = corner_points(chk, sim, "pts/perm")
    n = 96
    idx = np.sort(np.frombuffer(stream_bytes("pts/perm/i", 4 * n), np.uint32) % np.uint32(len(points) + 2))
    s1, s2 = corner_scalars(chk, "pts/perm", n)
    perm = np.random.default_rng(7).permutation(n)
    h = psim.pointset_create(points)
    try:
        a = psim.pointset(h, idx, s1, s2)
        b = psim.pointset(h, idx[perm], s1[perm], s2[perm])
        assert (a[perm] == b).all()
        assert psim.pointset(h, idx[:0], s1[:0], s2[:0]).shape == (0, 256)   # n = 0
    finally:
        psim.pointset_destroy(h)


# ---- GPU tier --------------------------------------------------------------------------------------------------------------
@pytest.fixture(params=["flat", "compact"])
def gpu_layout(request, gpu):
    gpu.keyset_policy(DEFAULT_POLICY if request.param == "flat" else 0)
    yield request.param
    gpu.keyset_policy(DEFAULT_POLICY)


@pytest.mark.gpu
def test_pointset_matches_base_double_scalarmul_on_the_gpu(gpu, chk, gpu_layout):
    """the corner cases at 2^12 elements: encodings against the checker (reference build or oracle), the exact point against the
    library's own base_double_scalarmul_non_secret_batch"""
    util.set_threads(chk, os.cpu_count() or 4)
    run_corners(gpu, chk, gpu, 1 << 12, "pts/gpu/" + gpu_layout, exact="gf_mul")


@pytest.mark.gpu
def test_pointset_million_elements_against_1024_points(gpu, chk):
    """2^20 elements against 1024 points (every eighth one with a torsion component) in random order, a few out of range"""
    n, m = 1 << 20, 1024
    points = gpu.from_hash_uniform(stream_bytes("pts/big/p", m * 112).reshape(m, 112))
    points[::8] = gpu.debugging_torque(points[::8])
    s1 = gpu.scalar_decode_long(stream_bytes("pts/big/s1", n * 56).reshape(n, 56), 56)
    s2 = gpu.scalar_decode_long(stream_bytes("pts/big/s2", n * 56).reshape(n, 56), 56)
    idx = np.frombuffer(stream_bytes("pts/big/i", 4 * n), np.uint32) % np.uint32(m + 8)
    h = gpu.pointset_create(points)
    try:
        got = gpu.pointset(h, idx, s1, s2)
    finally:
        gpu.pointset_destroy(h)
    want = gpu.base_double_scalarmul_non_secret(s1, operands(points, idx), s2)
    assert (gpu.point_encode(got) == gpu.point_encode(want)).all()
    assert_same_points_fast(gpu, got, want, "2^20 x 1024")


@pytest.mark.gpu
def test_pointset_sorted_and_shuffled_batches_agree(gpu, chk, gpu_layout):
    n, m = 1 << 16, 300
    points = util.random_points(chk, "pts/shuf/p", m)
    s1, s2 = corner_scalars(gpu, "pts/shuf", n)
    idx = np.sort(np.frombuffer(stream_bytes("pts/shuf/i", 4 * n), np.uint32) % np.uint32(m + 3))
    perm = np.random.default_rng(11).permutation(n)
    h = gpu.pointset_create(points)
    try:
        a = gpu.pointset(h, idx, s1, s2)
        b = gpu.pointset(h, idx[perm], s1[perm], s2[perm])
    finally:
        gpu.pointset_destroy(h)
    assert (a[perm] == b).all()


@pytest.mark.gpu
def test_pointset_dev_equals_host_call(gpu, chk, gpu_layout):
    import torch
    from libgoldilocks_b200.engine import DeviceEngine
    eng = DeviceEngine()
    points, _ = corner_points(chk, gpu, "pts/dev")
    n = 5000
    s1, s2 = corner_scalars(chk, "pts/dev", n)
    idx = corner_indices("pts/dev", n, len(points))
    h = gpu.pointset_create(points)
    try:
        want = gpu.pointset(h, idx, s1, s2)
        scratch = torch.empty(eng.pointset_scratch_bytes(n), dtype=torch.uint8, device="cuda")
        d_idx, d_s1, d_s2 = torch.from_numpy(idx.view(np.int32)).cuda(), torch.from_numpy(s1).cuda(), torch.from_numpy(s2).cuda()
        out = torch.full((n, 256), 0xa5, dtype=torch.uint8, device="cuda")
        eng.pointset(out, h, d_idx, d_s1, d_s2, scratch)
        torch.cuda.synchronize()
        assert (out.cpu().numpy() == want).all()
        eng.pointset(out[:0], h, d_idx[:0], d_s1, d_s2, scratch)   # n = 0 succeeds
    finally:
        gpu.pointset_destroy(h)


@pytest.mark.gpu
def test_pointset_empty_set_and_empty_batch(gpu, chk, gpu_layout):
    """an empty set is valid: every index is out of range, so the result is s1 B (the identity when s2 = 0)"""
    n = 777
    s1, s2 = corner_scalars(chk, "pts/empty", n)
    idx = np.frombuffer(stream_bytes("pts/empty/i", 4 * n), np.uint32)
    h = gpu.pointset_create(np.zeros((0, 256), np.uint8))
    try:
        assert gpu.pointset_size(h) == 0
        got = gpu.pointset(h, idx, s1, s2)
        assert gpu.pointset(h, idx[:0], s1[:0], s2[:0]).shape == (0, 256)
    finally:
        gpu.pointset_destroy(h)
    want = chk.base_double_scalarmul_non_secret(s1, operands(np.zeros((0, 256), np.uint8), idx), s2)
    assert (chk.point_encode(got) == chk.point_encode(want)).all()
    zero2 = ~s2.any(axis=1)
    assert zero2.any() and (chk.point_encode(got[zero2]) == 0).all()


@pytest.mark.gpu
def test_pointset_from_another_device_fails(gpu, chk):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    points = util.random_points(chk, "pts/dev2/p", 4)
    s1, s2 = util.random_scalars(chk, "pts/dev2/s1", 8), util.random_scalars(chk, "pts/dev2/s2", 8)
    prev = torch.cuda.current_device()
    torch.cuda.set_device(1)
    try:
        h = gpu.pointset_create(points)
    finally:
        torch.cuda.set_device(prev)
    try:
        with pytest.raises(RuntimeError, match="another device"):
            gpu.pointset(h, np.zeros(8, np.uint32), s1, s2)
    finally:
        gpu.pointset_destroy(h)
