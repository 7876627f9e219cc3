"""ctypes binding of the batched C ABI declared in include/goldilocks_b200.h.

`BatchLib(path)` binds any shared library that exports the `*_batch` entry points: the CUDA product
library (libgoldilocks_b200.so), and -- in the tests only -- the reference build, the oracle and the
host simulator, which export the same names.  All arrays are numpy uint8 with one element per row
(field element/decaf point encoding: 56 bytes, point struct: 256, scalar struct: 56, EdDSA key: 57,
signature: 114), exactly the packed host layout of the C ABI.
"""
import ctypes as C
import numpy as np

SUCCESS = -1
FAILURE = 0

_P = C.c_void_p
_Z = C.c_size_t


def _ptr(a):
    return None if a is None else a.ctypes.data_as(_P)


def _u8(a, width=None):
    a = np.ascontiguousarray(a, dtype=np.uint8)
    if width is not None:
        a = a.reshape(-1, width)
    return a


ALL = (1 << 64) - 1  # goldilocks_bool_t true


def _aligned(a, align):
    """copy of the flat uint8 array `a` whose data pointer is `align`-byte aligned (the reference's AVX2
    build loads table and point structs with aligned vector moves)"""
    buf = np.empty(a.size + align, np.uint8)
    off = (-buf.ctypes.data) % align
    out = buf[off:off + a.size]
    out[:] = a
    return out


def pack_messages(msgs):
    """list of bytes -> (arena uint8[total], offsets uint64[n+1])"""
    off = np.zeros(len(msgs) + 1, dtype=np.uint64)
    if msgs:
        off[1:] = np.cumsum([len(m) for m in msgs], dtype=np.uint64)
    arena = np.frombuffer(b"".join(msgs), dtype=np.uint8).copy() if msgs and int(off[-1]) else np.zeros(1, np.uint8)
    return arena, off


class BatchLib:
    def __init__(self, path):
        self.path = str(path)
        self.lib = C.CDLL(self.path, mode=C.RTLD_LOCAL)

    def has(self, name):
        return hasattr(self.lib, name)

    def _call(self, name, *args):
        fn = getattr(self.lib, name)
        fn.restype = C.c_int32
        conv = []
        for a in args:
            if isinstance(a, np.ndarray) or a is None:
                conv.append(_ptr(a))
            else:
                conv.append(a)
        r = fn(*conv)
        if r != SUCCESS:
            err = ""
            if self.has("goldilocks_b200_last_error"):
                f = self.lib.goldilocks_b200_last_error
                f.restype = C.c_char_p
                err = (f() or b"").decode()
            raise RuntimeError("%s failed: %s" % (name, err))

    # ---- field ----
    def _gf2(self, name, a, b):
        a, b = _u8(a, 56), _u8(b, 56)
        out = np.empty_like(a)
        self._call(name, out, a, b, _Z(len(a)))
        return out

    def gf_mul(self, a, b): return self._gf2("goldilocks_448_gf_mul_batch", a, b)
    def gf_add(self, a, b): return self._gf2("goldilocks_448_gf_add_batch", a, b)
    def gf_sub(self, a, b): return self._gf2("goldilocks_448_gf_sub_batch", a, b)

    def gf_sqr(self, a):
        a = _u8(a, 56); out = np.empty_like(a)
        self._call("goldilocks_448_gf_sqr_batch", out, a, _Z(len(a)))
        return out

    def gf_mulw(self, a, w):
        a = _u8(a, 56); out = np.empty_like(a)
        self._call("goldilocks_448_gf_mulw_batch", out, a, C.c_uint32(w), _Z(len(a)))
        return out

    def gf_isr(self, a):
        a = _u8(a, 56); out = np.empty_like(a); st = np.zeros(len(a), np.int32)
        self._call("goldilocks_448_gf_isr_batch", out, st, a, _Z(len(a)))
        return out, st

    def gf_invert(self, a):
        a = _u8(a, 56); out = np.empty_like(a)
        self._call("goldilocks_448_gf_invert_batch", out, a, _Z(len(a)))
        return out

    # ---- group ----
    def _pt2(self, name, a, b):
        a, b = _u8(a, 256), _u8(b, 256); out = np.empty_like(a)
        self._call(name, out, a, b, _Z(len(a)))
        return out

    def _pt1(self, name, a):
        a = _u8(a, 256); out = np.empty_like(a)
        self._call(name, out, a, _Z(len(a)))
        return out

    def point_add(self, a, b): return self._pt2("goldilocks_448_point_add_batch", a, b)
    def point_sub(self, a, b): return self._pt2("goldilocks_448_point_sub_batch", a, b)
    def point_double(self, a): return self._pt1("goldilocks_448_point_double_batch", a)
    def point_negate(self, a): return self._pt1("goldilocks_448_point_negate_batch", a)

    def point_eq(self, a, b):
        a, b = _u8(a, 256), _u8(b, 256); out = np.zeros(len(a), np.uint64)
        self._call("goldilocks_448_point_eq_batch", out, a, b, _Z(len(a)))
        return out != 0

    def point_valid(self, a):
        a = _u8(a, 256); out = np.zeros(len(a), np.uint64)
        self._call("goldilocks_448_point_valid_batch", out, a, _Z(len(a)))
        return out != 0

    def point_encode(self, a):
        a = _u8(a, 256); out = np.empty((len(a), 56), np.uint8)
        self._call("goldilocks_448_point_encode_batch", out, a, _Z(len(a)))
        return out

    def point_decode(self, ser, allow_identity=False):
        ser = _u8(ser, 56); out = np.empty((len(ser), 256), np.uint8); st = np.zeros(len(ser), np.int32)
        self._call("goldilocks_448_point_decode_batch", out, st, ser, C.c_uint64(0xFFFFFFFFFFFFFFFF if allow_identity else 0), _Z(len(ser)))
        return out, st

    def from_hash_nonuniform(self, h):
        h = _u8(h, 56); out = np.empty((len(h), 256), np.uint8)
        self._call("goldilocks_448_point_from_hash_nonuniform_batch", out, h, _Z(len(h)))
        return out

    def from_hash_uniform(self, h):
        h = _u8(h, 112); out = np.empty((len(h), 256), np.uint8)
        self._call("goldilocks_448_point_from_hash_uniform_batch", out, h, _Z(len(h)))
        return out

    def invert_elligator_nonuniform(self, pts, which):
        """elligator.c:104-152: (recovered (n,56) u8, status int32[n]); which[i] picks the preimage branch"""
        pts = _u8(pts, 256); which = np.ascontiguousarray(which, np.uint32)
        out = np.empty((len(pts), 56), np.uint8); st = np.zeros(len(pts), np.int32)
        self._call("goldilocks_448_invert_elligator_nonuniform_batch", out, st, pts, which, _Z(len(pts)))
        return out, st

    def invert_elligator_uniform(self, pts, second_half, which):
        """elligator.c:154-164: completes (n,112) hashes whose bytes 56..111 are `second_half`"""
        pts = _u8(pts, 256); which = np.ascontiguousarray(which, np.uint32)
        buf = np.zeros((len(pts), 112), np.uint8); buf[:, 56:] = _u8(second_half, 56)
        st = np.zeros(len(pts), np.int32)
        self._call("goldilocks_448_invert_elligator_uniform_batch", buf, st, pts, which, _Z(len(pts)))
        return buf, st

    def encode_like_eddsa(self, a):
        a = _u8(a, 256); out = np.empty((len(a), 57), np.uint8)
        self._call("goldilocks_448_point_mul_by_ratio_and_encode_like_eddsa_batch", out, a, _Z(len(a)))
        return out

    def decode_like_eddsa(self, enc):
        enc = _u8(enc, 57); out = np.empty((len(enc), 256), np.uint8); st = np.zeros(len(enc), np.int32)
        self._call("goldilocks_448_point_decode_like_eddsa_and_mul_by_ratio_batch", out, st, enc, _Z(len(enc)))
        return out, st

    def encode_like_x448(self, a):
        a = _u8(a, 256); out = np.empty((len(a), 56), np.uint8)
        self._call("goldilocks_448_point_mul_by_ratio_and_encode_like_x448_batch", out, a, _Z(len(a)))
        return out

    # ---- scalar multiplication ----
    def precomputed_scalarmul(self, scalars, table=None):
        """table = None: the base-point table; else one 15360-byte table from precompute()"""
        s = _u8(scalars, 56); out = np.empty((len(s), 256), np.uint8)
        base = None
        if table is not None:
            base = _aligned(np.ascontiguousarray(table, np.uint8).reshape(-1), 32)
        elif self.has("goldilocks_448_precomputed_base"):
            base = C.c_void_p.in_dll(self.lib, "goldilocks_448_precomputed_base")
        self._call("goldilocks_448_precomputed_scalarmul_batch", out, base, s, _Z(len(s)))
        return out

    def precompute(self, pts):
        p = _u8(pts, 256); out = _aligned(np.zeros(len(p) * 15360, np.uint8), 32)
        self._call("goldilocks_448_precompute_batch", out, p, _Z(len(p)))
        return out.reshape(len(p), 15360)

    def point_dual_scalarmul(self, pts, s1, s2):
        p, s1, s2 = _u8(pts, 256), _u8(s1, 56), _u8(s2, 56); o1 = np.empty_like(p); o2 = np.empty_like(p)
        self._call("goldilocks_448_point_dual_scalarmul_batch", o1, o2, p, s1, s2, _Z(len(p)))
        return o1, o2

    def direct_scalarmul(self, base, scalars, allow_identity=False, short_circuit=True, prefill=0):
        b, s = _u8(base, 56), _u8(scalars, 56)
        out = np.full((len(b), 56), prefill, np.uint8); st = np.zeros(len(b), np.int32)
        self._call("goldilocks_448_direct_scalarmul_batch", out, st, b, s, C.c_uint64(ALL if allow_identity else 0), C.c_uint64(ALL if short_circuit else 0), _Z(len(b)))
        return out, st

    def debugging_torque(self, pts):
        p = _u8(pts, 256); out = np.empty_like(p)
        self._call("goldilocks_448_point_debugging_torque_batch", out, p, _Z(len(p)))
        return out

    def debugging_pscale(self, pts, factor):
        p, f = _u8(pts, 256), _u8(factor, 56); out = np.empty_like(p)
        self._call("goldilocks_448_point_debugging_pscale_batch", out, p, f, _Z(len(p)))
        return out

    def point_scalarmul(self, pts, scalars):
        p, s = _u8(pts, 256), _u8(scalars, 56); out = np.empty_like(p)
        self._call("goldilocks_448_point_scalarmul_batch", out, p, s, _Z(len(p)))
        return out

    def point_double_scalarmul(self, p1, s1, p2, s2):
        p1, s1, p2, s2 = _u8(p1, 256), _u8(s1, 56), _u8(p2, 256), _u8(s2, 56); out = np.empty_like(p1)
        self._call("goldilocks_448_point_double_scalarmul_batch", out, p1, s1, p2, s2, _Z(len(p1)))
        return out

    def base_double_scalarmul_non_secret(self, s1, p2, s2):
        s1, p2, s2 = _u8(s1, 56), _u8(p2, 256), _u8(s2, 56); out = np.empty_like(p2)
        self._call("goldilocks_448_base_double_scalarmul_non_secret_batch", out, s1, p2, s2, _Z(len(p2)))
        return out

    # ---- scalars ----
    def _sc2(self, name, a, b):
        a, b = _u8(a, 56), _u8(b, 56); out = np.empty_like(a)
        self._call(name, out, a, b, _Z(len(a)))
        return out

    def scalar_add(self, a, b): return self._sc2("goldilocks_448_scalar_add_batch", a, b)
    def scalar_sub(self, a, b): return self._sc2("goldilocks_448_scalar_sub_batch", a, b)
    def scalar_mul(self, a, b): return self._sc2("goldilocks_448_scalar_mul_batch", a, b)

    def scalar_invert(self, a):
        a = _u8(a, 56); out = np.empty_like(a); st = np.zeros(len(a), np.int32)
        self._call("goldilocks_448_scalar_invert_batch", out, st, a, _Z(len(a)))
        return out, st

    def scalar_halve(self, a):
        a = _u8(a, 56); out = np.empty_like(a)
        self._call("goldilocks_448_scalar_halve_batch", out, a, _Z(len(a)))
        return out

    def scalar_decode_long(self, ser, ser_len):
        ser = _u8(ser, ser_len) if ser_len else np.zeros((len(ser), 0), np.uint8)
        out = np.empty((len(ser), 56), np.uint8)
        self._call("goldilocks_448_scalar_decode_long_batch", out, ser if ser_len else np.zeros(1, np.uint8), _Z(ser_len), _Z(len(ser)))
        return out

    # ---- CFRG ----
    def x448(self, base, scalar):
        base, scalar = _u8(base, 56), _u8(scalar, 56)
        out = np.empty_like(base); st = np.zeros(len(base), np.int32)
        self._call("goldilocks_x448_batch", out, st, base, scalar, _Z(len(base)))
        return out, st

    def convert_public_key_to_x448(self, ed):
        ed = _u8(ed, 57); out = np.empty((len(ed), 56), np.uint8)
        self._call("goldilocks_ed448_convert_public_key_to_x448_batch", out, ed, _Z(len(ed)))
        return out

    def convert_private_key_to_x448(self, ed):
        ed = _u8(ed, 57); out = np.empty((len(ed), 56), np.uint8)
        self._call("goldilocks_ed448_convert_private_key_to_x448_batch", out, ed, _Z(len(ed)))
        return out

    def x448_derive_public_key(self, scalar):
        scalar = _u8(scalar, 56); out = np.empty_like(scalar)
        self._call("goldilocks_x448_derive_public_key_batch", out, scalar, _Z(len(scalar)))
        return out

    def shake256(self, msgs, outlen):
        arena, off = pack_messages(msgs)
        out = np.empty((len(msgs), outlen), np.uint8)
        self._call("goldilocks_shake256_hash_batch", out, _Z(outlen), arena, off, _Z(len(msgs)))
        return out

    def ed448_derive_public_key(self, sk):
        sk = _u8(sk, 57); out = np.empty_like(sk)
        self._call("goldilocks_ed448_derive_public_key_batch", out, sk, _Z(len(sk)))
        return out

    @staticmethod
    def _ctx(context):
        ctx = np.frombuffer(bytes(context), dtype=np.uint8).copy() if context else np.zeros(1, np.uint8)
        return ctx, len(context) if context else 0

    def ed448_sign(self, sk, pk, msgs, prehashed=False, context=b""):
        sk, pk = _u8(sk, 57), _u8(pk, 57)
        arena, off = pack_messages(msgs) if isinstance(msgs, list) else msgs
        ctx, ctx_len = self._ctx(context)
        sig = np.empty((len(sk), 114), np.uint8)
        self._call("goldilocks_ed448_sign_batch", sig, sk, pk, arena, off, C.c_uint8(1 if prehashed else 0), ctx, C.c_uint8(ctx_len), _Z(len(sk)))
        return sig

    # ---- key sets: per-key verification tables kept on the device across calls ----
    def keyset_create(self, pk):
        """handle for m public keys ((m,57) u8); free it with keyset_destroy"""
        pk = _u8(pk, 57)
        h = C.c_void_p()
        self._call("goldilocks_b200_keyset_create", C.byref(h), pk, _Z(len(pk)))
        return h

    def keyset_destroy(self, handle):
        self.lib.goldilocks_b200_keyset_destroy.restype = None
        self.lib.goldilocks_b200_keyset_destroy(handle)

    def ed448_verify_keyset(self, handle, key_index, sig, msgs, prehashed=False, context=b""):
        """status int32[n] of signature i under key key_index[i] of the set"""
        sig = _u8(sig, 114); key_index = np.ascontiguousarray(key_index, np.uint32)
        arena, off = pack_messages(msgs) if isinstance(msgs, list) else msgs
        ctx, ctx_len = self._ctx(context)
        st = np.zeros(len(sig), np.int32)
        self._call("goldilocks_ed448_verify_keyset_batch", st, handle, key_index, sig, arena, off, C.c_uint8(1 if prehashed else 0), ctx, C.c_uint8(ctx_len), _Z(len(sig)))
        return st

    def ed448_verify_keyset_lookup(self, handle, sig, pk, msgs, prehashed=False, context=b"", return_index=False):
        """status int32[n] of signature i under public key pk[i] ((n,57) u8), exactly goldilocks_ed448_verify's; keys found in the set
        use its tables, the rest the ordinary path.  With return_index: (status, key_index uint32[n]), the lowest set index whose
        57 bytes equal pk[i], or m"""
        sig, pk = _u8(sig, 114), _u8(pk, 57)
        arena, off = pack_messages(msgs) if isinstance(msgs, list) else msgs
        ctx, ctx_len = self._ctx(context)
        st = np.zeros(len(sig), np.int32)
        idx = np.zeros(len(sig), np.uint32) if return_index else None
        self._call("goldilocks_ed448_verify_keyset_lookup_batch", st, idx, handle, sig, pk, arena, off, C.c_uint8(1 if prehashed else 0), ctx, C.c_uint8(ctx_len),
                   _Z(len(sig)))
        return (st, idx) if return_index else st

    # ---- X448 peer sets: per-peer comb tables kept on the device across calls ----
    def x448_peerset_create(self, peers):
        """handle for m peer u-coordinates ((m,56) u8); free it with x448_peerset_destroy"""
        peers = _u8(peers, 56)
        h = C.c_void_p()
        self._call("goldilocks_b200_x448_peerset_create", C.byref(h), peers, _Z(len(peers)))
        return h

    def x448_peerset_destroy(self, handle):
        self.lib.goldilocks_b200_x448_peerset_destroy.restype = None
        self.lib.goldilocks_b200_x448_peerset_destroy(handle)

    def x448_peerset_size(self, handle):
        f = self.lib.goldilocks_b200_x448_peerset_size
        f.restype = _Z
        return int(f(handle))

    def x448_peerset(self, handle, peer_index, scalar):
        """(out (n,56) u8, status int32[n]): X448 of scalar i against peer peer_index[i] of the set"""
        scalar = _u8(scalar, 56); peer_index = np.ascontiguousarray(peer_index, np.uint32).reshape(-1)
        out = np.empty_like(scalar); st = np.zeros(len(scalar), np.int32)
        self._call("goldilocks_x448_peerset_batch", out, st, handle, peer_index, scalar, _Z(len(scalar)))
        return out, st

    def x448_peerset_lookup(self, handle, base, scalar, return_index=False):
        """(out (n,56) u8, status int32[n]) of X448 of scalar i against base i ((n,56) u8), exactly goldilocks_x448's; peers found in
        the set by their bytes use its tables, the rest the ladder.  With return_index: (out, status, peer_index uint32[n]), the
        lowest set index whose 56 bytes equal base[i], or m"""
        base, scalar = _u8(base, 56), _u8(scalar, 56)
        out = np.empty_like(scalar); st = np.zeros(len(scalar), np.int32)
        idx = np.zeros(len(scalar), np.uint32) if return_index else None
        self._call("goldilocks_x448_peerset_lookup_batch", out, st, idx, handle, base, scalar, _Z(len(scalar)))
        return (out, st, idx) if return_index else (out, st)

    # ---- decaf peer sets: per-peer comb tables for direct_scalarmul against recurring points ----
    def decaf_peerset_create(self, encodings, allow_identity=False):
        """handle for m peer encodings ((m,56) u8) decoded under allow_identity; free it with decaf_peerset_destroy"""
        enc = _u8(encodings, 56)
        h = C.c_void_p()
        self._call("goldilocks_b200_decaf_peerset_create", C.byref(h), enc, C.c_uint64(ALL if allow_identity else 0), _Z(len(enc)))
        return h

    def decaf_peerset_destroy(self, handle):
        self.lib.goldilocks_b200_decaf_peerset_destroy.restype = None
        self.lib.goldilocks_b200_decaf_peerset_destroy(handle)

    def decaf_peerset_size(self, handle):
        f = self.lib.goldilocks_b200_decaf_peerset_size
        f.restype = _Z
        return int(f(handle))

    def decaf_peerset(self, handle, peer_index, scalars, short_circuit=True, prefill=0):
        """(scaled (n,56) u8, status int32[n]): direct_scalarmul of scalar struct i against peer peer_index[i] of the set;
        `prefill` is what short-circuited elements keep, as in direct_scalarmul"""
        s = _u8(scalars, 56); peer_index = np.ascontiguousarray(peer_index, np.uint32).reshape(-1)
        out = np.full((len(s), 56), prefill, np.uint8); st = np.zeros(len(s), np.int32)
        self._call("goldilocks_448_direct_scalarmul_peerset_batch", out, st, handle, peer_index, s, C.c_uint64(ALL if short_circuit else 0), _Z(len(s)))
        return out, st

    # ---- point sets: key-set tables for base_double_scalarmul_non_secret against recurring points ----
    def pointset_create(self, points):
        """handle for m point structs ((m,256) u8, each goldilocks_448_point_valid); free it with pointset_destroy"""
        pts = _u8(points, 256)
        h = C.c_void_p()
        self._call("goldilocks_b200_pointset_create", C.byref(h), pts, _Z(len(pts)))
        return h

    def pointset_destroy(self, handle):
        self.lib.goldilocks_b200_pointset_destroy.restype = None
        self.lib.goldilocks_b200_pointset_destroy(handle)

    def pointset_size(self, handle):
        f = self.lib.goldilocks_b200_pointset_size
        f.restype = _Z
        return int(f(handle))

    def pointset(self, handle, point_index, s1, s2):
        """(n,256) u8: base_double_scalarmul_non_secret(s1[i], point point_index[i] of the set, s2[i]); an index >= m stands for
        the identity"""
        s1, s2 = _u8(s1, 56), _u8(s2, 56); point_index = np.ascontiguousarray(point_index, np.uint32).reshape(-1)
        out = np.empty((len(s1), 256), np.uint8)
        self._call("goldilocks_448_base_double_scalarmul_non_secret_pointset_batch", out, handle, point_index, s1, s2, _Z(len(s1)))
        return out

    def ed448_verify(self, sig, pk, msgs, prehashed=False, context=b""):
        sig, pk = _u8(sig, 114), _u8(pk, 57)
        arena, off = pack_messages(msgs) if isinstance(msgs, list) else msgs
        ctx, ctx_len = self._ctx(context)
        st = np.zeros(len(sig), np.int32)
        self._call("goldilocks_ed448_verify_batch", st, sig, pk, arena, off, C.c_uint8(1 if prehashed else 0), ctx, C.c_uint8(ctx_len), _Z(len(sig)))
        return st

    def ed448_verify_rlc(self, sig, pk, msgs, prehashed=False, context=b""):
        """(status int32[n], fast) -- goldilocks_ed448_verify_rlc_batch: random-linear-combination fast path with
        per-element fallback; fast = 1 when the batch equation decided the call"""
        sig, pk = _u8(sig, 114), _u8(pk, 57)
        arena, off = pack_messages(msgs) if isinstance(msgs, list) else msgs
        ctx, ctx_len = self._ctx(context)
        st = np.zeros(len(sig), np.int32)
        fast = C.c_int(0)
        self._call("goldilocks_ed448_verify_rlc_batch", st, sig, pk, arena, off, C.c_uint8(1 if prehashed else 0), ctx, C.c_uint8(ctx_len), _Z(len(sig)), C.byref(fast))
        return st, fast.value

    def keyset_policy(self, max_table_bytes):
        """goldilocks_b200_keyset_policy: key sets whose flat tables (369 KB per key, no doublings per signature) fit this many bytes get them"""
        self.lib.goldilocks_b200_keyset_policy.restype = None
        self.lib.goldilocks_b200_keyset_policy(C.c_ulonglong(max_table_bytes))

    def rlc_policy(self, reprobe):
        """goldilocks_b200_rlc_policy: how many calls skip the batch equation after one in which most chunks failed (0 = never skip)"""
        self.lib.goldilocks_b200_rlc_policy.restype = None
        self.lib.goldilocks_b200_rlc_policy(C.c_uint(reprobe))

    # ---- the reference's own single-element calls, and their gathering into batches (csrc/coalesce.h) ----
    def coalesce(self, window_us, max_batch=0):
        """goldilocks_b200_coalesce: concurrent single-element verify / sign / X448 calls wait up to window_us for each other and share
        one batch launch (0 = off)"""
        self.lib.goldilocks_b200_coalesce.restype = None
        self.lib.goldilocks_b200_coalesce(C.c_uint(window_us), C.c_uint(max_batch))

    def coalesce_stats(self):
        """(calls that went through a gathering, batches launched for them, largest batch)"""
        a, b, c = C.c_ulonglong(0), C.c_ulonglong(0), C.c_ulonglong(0)
        self.lib.goldilocks_b200_coalesce_stats.restype = None
        self.lib.goldilocks_b200_coalesce_stats(C.byref(a), C.byref(b), C.byref(c))
        return a.value, b.value, c.value

    def ed448_verify_one(self, sig, pk, msg, prehashed=False, context=b""):
        """goldilocks_ed448_verify (ed448.h:157-165) on one signature: -1 / 0"""
        fn = self.lib.goldilocks_ed448_verify
        fn.restype = C.c_int32
        return fn(C.c_char_p(bytes(sig)), C.c_char_p(bytes(pk)), C.c_char_p(bytes(msg)), _Z(len(msg)), C.c_uint8(1 if prehashed else 0),
                  C.c_char_p(bytes(context)) if context else None, C.c_uint8(len(context)))

    def ed448_sign_one(self, sk, pk, msg, prehashed=False, context=b""):
        """goldilocks_ed448_sign (ed448.h:108-118) on one message: the 114 signature bytes"""
        out = C.create_string_buffer(114)
        fn = self.lib.goldilocks_ed448_sign
        fn.restype = None
        fn(out, C.c_char_p(bytes(sk)), C.c_char_p(bytes(pk)), C.c_char_p(bytes(msg)), _Z(len(msg)), C.c_uint8(1 if prehashed else 0),
           C.c_char_p(bytes(context)) if context else None, C.c_uint8(len(context)))
        return out.raw

    def x448_one(self, base, scalar):
        """goldilocks_x448 on one (u, k) pair: (56 bytes, -1 / 0)"""
        out = C.create_string_buffer(56)
        fn = self.lib.goldilocks_x448
        fn.restype = C.c_int32
        st = fn(out, C.c_char_p(bytes(base)), C.c_char_p(bytes(scalar)))
        return out.raw, st

    # ---- device sets: one host-pointer batch over several GPUs (include/goldilocks_b200.h, section 4) ----
    def set_devices(self, devices):
        """spread every later `*_batch` host-pointer call over these CUDA devices ([] = the current device only)"""
        devs = (C.c_int * max(1, len(devices)))(*devices)
        self._call("goldilocks_b200_set_devices", devs, C.c_int(len(devices)))

    def get_devices(self):
        buf = (C.c_int * 64)()
        self.lib.goldilocks_b200_get_devices.restype = C.c_int
        n = self.lib.goldilocks_b200_get_devices(buf, C.c_int(64))
        return list(buf[:n])

    def shard_plan(self, n, ndev, bytes_per_elem=0, pipelined=False):
        """[(lo, hi, device_slot, lane)] -- the partition a sharded call uses (pure arithmetic, no GPU needed)"""
        cap = 1 << 16
        lo, hi = (C.c_size_t * cap)(), (C.c_size_t * cap)()
        slot, lane = (C.c_int * cap)(), (C.c_int * cap)()
        f = self.lib.goldilocks_b200_shard_plan
        f.restype = C.c_size_t
        k = f(lo, hi, slot, lane, _Z(cap), _Z(n), C.c_int(ndev), _Z(bytes_per_elem), C.c_int(1 if pipelined else 0))
        assert k <= cap
        return [(lo[i], hi[i], slot[i], lane[i]) for i in range(k)]

    def debug_niels(self, p, q, which, op):
        """goldilocks_b200_debug_niels_batch: one mixed addition / conversion of goldilocks.c:271-380 per element -> (n,256) points"""
        p, q = _u8(p, 256), _u8(q, 256); which = np.ascontiguousarray(which, np.uint32)
        out = np.empty_like(p)
        self._call("goldilocks_b200_debug_niels_batch", out, p, q, which, C.c_uint32(op), _Z(len(p)))
        return out

    # ---- tables ----
    def export_comb_table(self):
        out = np.empty(15360, np.uint8)
        name = "goldilocks_b200_export_comb_table" if self.has("goldilocks_b200_export_comb_table") else "refb_export_comb_table"
        fn = getattr(self.lib, name); fn.restype = C.c_int32
        fn(_ptr(out))
        return out

    def export_wnaf_table(self):
        out = np.empty(6144, np.uint8)
        name = "goldilocks_b200_export_wnaf_table" if self.has("goldilocks_b200_export_wnaf_table") else "refb_export_wnaf_table"
        fn = getattr(self.lib, name); fn.restype = C.c_int32
        fn(_ptr(out))
        return out
