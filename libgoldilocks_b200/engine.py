"""Device-resident calls and batch sharding.

Replaces nothing in the reference (it has no device or multi-process layer, SURVEY.md section 5);
this is the thin host plumbing the north_star asks for: a batch is split into contiguous ranges,
one per GPU / rank, with no collective on the data path (SURVEY.md section 8(e)).  torch is used
for device memory, streams and (optionally) torch.distributed rendezvous only.
"""
import ctypes as C

from . import load

_P = C.c_void_p
_Z = C.c_size_t


def shard_range(n, rank, world):
    """Contiguous range [lo, hi) of a batch of n elements owned by `rank` of `world` (8(e))."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError("bad rank/world")
    return (n * rank) // world, (n * (rank + 1)) // world


def shard_ranges(n, world):
    return [shard_range(n, r, world) for r in range(world)]


def shard_messages(off, lo, hi):
    """Message arena slice + rebased offsets for elements [lo, hi) (off has n+1 entries)."""
    base = int(off[lo])
    return base, int(off[hi]), (off[lo:hi + 1] - off[lo]).copy()


class DeviceEngine:
    """Calls the `*_dev` entry points on torch CUDA tensors (uint8 / int32), on torch's current stream."""

    def __init__(self):
        import torch
        self.torch = torch
        self.capi = load()
        self.lib = self.capi.lib
        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device: libgoldilocks_b200 has no CPU path")
        self.init()

    def init(self):
        f = self.lib.goldilocks_b200_init
        f.restype = C.c_int32
        if f() != -1:
            raise RuntimeError("goldilocks_b200_init failed: " + self.last_error())

    def last_error(self):
        f = self.lib.goldilocks_b200_last_error
        f.restype = C.c_char_p
        return (f() or b"").decode()

    def launch_count(self):
        f = self.lib.goldilocks_b200_launch_count
        f.restype = C.c_uint64
        return int(f())

    def _stream(self):
        return _P(self.torch.cuda.current_stream().cuda_stream)

    def _call(self, name, *args):
        fn = getattr(self.lib, name)
        fn.restype = C.c_int32
        if fn(*args) != -1:
            raise RuntimeError("%s failed: %s" % (name, self.last_error()))

    @staticmethod
    def _p(t):
        return _P(0 if t is None else t.data_ptr())

    def verify_scratch_bytes(self, n):
        f = self.lib.goldilocks_b200_verify_scratch_bytes
        f.restype = _Z
        f.argtypes = [_Z]
        return int(f(n))

    def ed448_verify(self, status, sig, pk, msg, msg_off, scratch, prehashed=0, ctx=None, ctx_len=0):
        n = status.numel()
        self._call("goldilocks_ed448_verify_batch_dev", self._p(status), self._p(sig), self._p(pk), self._p(msg), self._p(msg_off),
                   C.c_uint8(prehashed), self._p(ctx), C.c_uint8(ctx_len), _Z(n), self._p(scratch), self._stream())

    def ed448_verify_rlc(self, status, sig, pk, msg, msg_off, prehashed=0, ctx=None, ctx_len=0):
        """random-linear-combination fast path (goldilocks_ed448_verify_rlc_batch_dev); returns 1 when the batch equation
        decided the call, 0 when it fell back to the per-signature path.  Synchronises the current stream."""
        fast = C.c_int(0)
        self._call("goldilocks_ed448_verify_rlc_batch_dev", self._p(status), self._p(sig), self._p(pk), self._p(msg), self._p(msg_off),
                   C.c_uint8(prehashed), self._p(ctx), C.c_uint8(ctx_len), _Z(status.numel()), self._stream(), C.byref(fast))
        return fast.value

    def keyset_scratch_bytes(self, n, msg_bytes):
        f = self.lib.goldilocks_b200_keyset_scratch_bytes
        f.restype = _Z
        f.argtypes = [_Z, _Z]
        return int(f(n, msg_bytes))

    def ed448_verify_keyset_lookup(self, status, key_index, handle, sig, pk, msg, msg_off, scratch, prehashed=0, ctx=None, ctx_len=0):
        """goldilocks_ed448_verify_keyset_lookup_batch_dev against a set made by capi keyset_create; key_index (int32 tensor read as
        uint32, or None) receives the looked-up indices; `scratch` holds keyset_scratch_bytes(n, msg_off[n]).  Synchronises the current
        stream once, after the lookup."""
        self._call("goldilocks_ed448_verify_keyset_lookup_batch_dev", self._p(status), self._p(key_index), handle, self._p(sig), self._p(pk), self._p(msg),
                   self._p(msg_off), C.c_uint8(prehashed), self._p(ctx), C.c_uint8(ctx_len), _Z(status.numel()), self._p(scratch), self._stream())

    def ed448_verify_keyset(self, status, handle, key_index, sig, msg, msg_off, scratch, prehashed=0, ctx=None, ctx_len=0):
        """goldilocks_ed448_verify_keyset_batch_dev: signature i under key key_index[i] (int32 tensor read as uint32) of the set"""
        self._call("goldilocks_ed448_verify_keyset_batch_dev", self._p(status), handle, self._p(key_index), self._p(sig), self._p(msg), self._p(msg_off),
                   C.c_uint8(prehashed), self._p(ctx), C.c_uint8(ctx_len), _Z(status.numel()), self._p(scratch), self._stream())

    def x448(self, out, status, base, scalar):
        self._call("goldilocks_x448_batch_dev", self._p(out), self._p(status), self._p(base), self._p(scalar), _Z(status.numel()), self._stream())

    def x448_peerset(self, out, status, handle, peer_index, scalar):
        """X448 of scalar i against peer peer_index[i] (uint32 tensor viewed as int32) of a set made by capi x448_peerset_create"""
        self._call("goldilocks_x448_peerset_batch_dev", self._p(out), self._p(status), handle, self._p(peer_index), self._p(scalar),
                   _Z(status.numel()), self._stream())

    def x448_peerset_scratch_bytes(self, n):
        f = self.lib.goldilocks_b200_x448_peerset_scratch_bytes
        f.restype = _Z
        f.argtypes = [_Z]
        return int(f(n))

    def x448_peerset_lookup(self, out, status, peer_index, handle, base, scalar, scratch):
        """goldilocks_x448_peerset_lookup_batch_dev: X448 of scalar i against base i, peers found in a set made by capi
        x448_peerset_create by their bytes; peer_index (int32 tensor read as uint32, or None) receives the looked-up indices;
        `scratch` holds x448_peerset_scratch_bytes(n).  Asynchronous on the current stream."""
        self._call("goldilocks_x448_peerset_lookup_batch_dev", self._p(out), self._p(status), self._p(peer_index), handle, self._p(base), self._p(scalar),
                   _Z(status.numel()), self._p(scratch), self._stream())

    def decaf_peerset_scratch_bytes(self, n):
        f = self.lib.goldilocks_b200_decaf_peerset_scratch_bytes
        f.restype = _Z
        f.argtypes = [_Z]
        return int(f(n))

    def decaf_peerset(self, scaled, status, handle, peer_index, scalars, scratch, short_circuit=True):
        """direct_scalarmul of scalar struct i against peer peer_index[i] (uint32 tensor viewed as int32) of a set made by capi
        decaf_peerset_create; `scaled` is read (short-circuited elements keep it) and written in place; `scratch` holds
        decaf_peerset_scratch_bytes(n)"""
        self._call("goldilocks_448_direct_scalarmul_peerset_batch_dev", self._p(scaled), self._p(status), handle, self._p(peer_index), self._p(scalars),
                   C.c_uint64((1 << 64) - 1 if short_circuit else 0), _Z(status.numel()), self._p(scratch), self._stream())

    def pointset_scratch_bytes(self, n):
        f = self.lib.goldilocks_b200_pointset_scratch_bytes
        f.restype = _Z
        f.argtypes = [_Z]
        return int(f(n))

    def pointset(self, out, handle, point_index, s1, s2, scratch):
        """base_double_scalarmul_non_secret of scalar structs s1[i], s2[i] against point point_index[i] (uint32 tensor viewed as int32)
        of a set made by capi pointset_create, into the point structs `out`; `scratch` holds pointset_scratch_bytes(n)"""
        self._call("goldilocks_448_base_double_scalarmul_non_secret_pointset_batch_dev", self._p(out), handle, self._p(point_index), self._p(s1), self._p(s2),
                   _Z(point_index.numel()), self._p(scratch), self._stream())

    def precomputed_scalarmul(self, out_pts, scalars):
        self._call("goldilocks_448_precomputed_scalarmul_batch_dev", self._p(out_pts), self._p(scalars), _Z(scalars.numel() // 56), self._stream())

    def gf_mul(self, out, a, b):
        self._call("goldilocks_448_gf_mul_batch_dev", self._p(out), self._p(a), self._p(b), _Z(a.numel() // 56), self._stream())

    def point_add(self, out, a, b):
        self._call("goldilocks_448_point_add_batch_dev", self._p(out), self._p(a), self._p(b), _Z(a.numel() // 256), self._stream())

    def point_double(self, out, a):
        self._call("goldilocks_448_point_double_batch_dev", self._p(out), self._p(a), _Z(a.numel() // 256), self._stream())

    def point_decode(self, pts, status, ser, allow_identity=False):
        self._call("goldilocks_448_point_decode_batch_dev", self._p(pts), self._p(status), self._p(ser),
                   C.c_uint64(0xFFFFFFFFFFFFFFFF if allow_identity else 0), _Z(status.numel()), self._stream())

    def point_encode(self, ser, pts):
        self._call("goldilocks_448_point_encode_batch_dev", self._p(ser), self._p(pts), _Z(pts.numel() // 256), self._stream())
