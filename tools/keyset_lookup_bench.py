#!/usr/bin/env python3
"""Verification by public-key bytes against a key set (goldilocks_ed448_verify_keyset_lookup_batch[_dev]) against
goldilocks_ed448_verify_batch and the index form goldilocks_ed448_verify_keyset_batch on the same data, on one GPU (DESIGN.md
decision 23).

    python tools/keyset_lookup_bench.py [--n 1048576] [--reps 10] [--out FILE.json]
    python tools/keyset_lookup_bench.py --create-only [--lib OTHER/libgoldilocks_b200.so] [--out FILE.json]

The corpus is bench.py's: n signatures under n/16 keys x 16, one in eight corrupted (R, S, key bytes or message), 32-byte
messages, signed by this library (its signatures are the reference's byte for byte).  Variants of it, each against a set:
  all hits, corpus order / shuffled : the corrupted key bytes restored, the n/16 keys as the set
  bench corpus                      : as bench.py makes it (1/32 of the keys changed: misses), the n/16 intact keys as the set
  1/4 misses                        : the bench corpus against the set without every fourth key
  all misses                        : the bench corpus against n/16 other keys
For each, in both table layouts (goldilocks_b200_keyset_policy):
  host   : the lookup call, goldilocks_ed448_verify_batch and (all-hit corpora) the index form with precomputed indices, from pinned host
           buffers, wall clock over `reps` calls after a warm-up call
  device : their _dev forms, CUDA events around `reps` calls
Every timed output is compared byte for byte with goldilocks_ed448_verify_batch's on the same corpus before anything is timed and
after the timed calls.  Also: the host-side mapping of key bytes to indices a caller pays without the lookup (a Python dict and
NumPy's sorted search), and set creation.  --create-only times creation alone, with --lib naming another build of the library.
The device name and power limit are recorded beside the numbers.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
DEFAULT_POLICY = 32 << 30


def device_info(torch):
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.stdout.strip() else q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = "unavailable: %s" % e
    return info


def create_times(lib, keys, label):
    """warm creation (the arena has grown once) of a set of `keys`, flat and compact"""
    out = {}
    for layout, policy in (("flat", DEFAULT_POLICY), ("compact", 0)):
        lib.keyset_policy(policy)
        try:
            lib.keyset_destroy(lib.keyset_create(keys))
            t = []
            for _ in range(3):
                t0 = time.perf_counter()
                h = lib.keyset_create(keys)
                t.append(1e3 * (time.perf_counter() - t0))
                lib.keyset_destroy(h)
        finally:
            lib.keyset_policy(DEFAULT_POLICY)
        out[layout] = {"keys": len(keys), "ms_min": round(min(t), 2), "ms_all": [round(x, 2) for x in t]}
        print("%s: create %d keys (%s): %.2f ms" % (label, len(keys), layout, min(t)), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--create-only", action="store_true")
    ap.add_argument("--lib", default=None, help="another build of libgoldilocks_b200.so (--create-only)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("keyset_lookup_bench: no CUDA device (this measures the GPU; there is no CPU number to give)")
    import libgoldilocks_b200 as g
    from libgoldilocks_b200.capi import BatchLib
    from util import stream_bytes
    import bench
    n = args.n
    nk = n // 16
    rec = dict(device_info(torch), n=n, reps=args.reps)
    if args.create_only:
        lib = BatchLib(args.lib) if args.lib else g.load()
        lib.lib.goldilocks_b200_init.restype = C.c_int32
        assert lib.lib.goldilocks_b200_init() == -1
        sk = stream_bytes("klb/create/sk", nk * 57).reshape(nk, 57)
        rec["library"] = args.lib or "this tree"
        rec["create"] = create_times(lib, lib.ed448_derive_public_key(sk), rec["library"])
        if args.out:
            with open(args.out, "w") as f:
                json.dump(rec, f, indent=1)
        return

    from libgoldilocks_b200.engine import DeviceEngine
    lib, eng = g.load(), DeviceEngine()
    sig, pk, arena, off, expect = bench.make_corpus(lib, n, "klb/corpus")
    keys = pk[1::16].copy()                                   # entry 16 j + 1 is never corrupted: the intact key of group j
    pk_intact = np.repeat(keys, 16, axis=0)
    other = lib.ed448_derive_public_key(stream_bytes("klb/other/sk", nk * 57).reshape(nk, 57))
    perm = np.random.default_rng(9).permutation(n)
    quarter = keys[np.arange(nk) % 4 != 0]

    def pinned(a):
        t = torch.empty(a.shape, dtype=torch.from_numpy(a[:0]).dtype).pin_memory()
        t.numpy()[:] = a
        return t.numpy()

    def dev(a):
        return torch.from_numpy(np.ascontiguousarray(a)).cuda()

    def host_timed(fn):
        fn()
        t = time.perf_counter()
        for _ in range(args.reps):
            fn()
        return 1e3 * (time.perf_counter() - t) / args.reps

    def dev_timed(fn):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / args.reps

    # (name, signature order, public keys, set, index form timed)
    corpora = (("all hits, corpus order", None, pk_intact, keys, True), ("all hits, shuffled", perm, pk_intact, keys, True),
               ("bench corpus (1/32 misses)", None, pk, keys, False), ("1/4 misses", None, pk, quarter, False),
               ("all misses", None, pk, other, False))
    rec["corpora"] = {}
    h_off = pinned(off.view(np.int64))
    d_off = dev(off.view(np.int64))
    for name, order, pub, set_keys, with_index in corpora:
        s, p = (sig, pub) if order is None else (sig[order], pub[order])
        if order is None:
            msg = arena
        else:
            msg = arena[: n * bench.MSG_LEN].reshape(n, bench.MSG_LEN)[order].reshape(-1)   # fixed-length messages: same offsets
        h_sig, h_pk, h_msg = pinned(np.ascontiguousarray(s)), pinned(np.ascontiguousarray(p)), pinned(np.ascontiguousarray(msg))
        d_sig, d_pk, d_msg = dev(h_sig), dev(h_pk), dev(h_msg)
        want = lib.ed448_verify(h_sig, h_pk, (h_msg, h_off.view(np.uint64)))
        h_st = pinned(np.zeros(n, np.int32))
        h_idx = pinned(np.zeros(n, np.int32)).view(np.uint32)
        d_st = torch.empty(n, dtype=torch.int32, device="cuda")
        d_idx = torch.empty(n, dtype=torch.int32, device="cuda")
        d_scratch = torch.empty(eng.keyset_scratch_bytes(n, int(off[-1])), dtype=torch.uint8, device="cuda")
        d_vscratch = torch.empty(eng.verify_scratch_bytes(n), dtype=torch.uint8, device="cuda")
        # the mapping a caller pays without the lookup call: key bytes -> lowest set index, on the host
        t0 = time.perf_counter()
        lowest = {}
        for j in range(len(set_keys) - 1, -1, -1):
            lowest[set_keys[j].tobytes()] = j
        dict_idx = np.fromiter((lowest.get(b, len(set_keys)) for b in h_pk.view("V57").reshape(-1).tolist()), np.uint32, n)
        dict_ms = 1e3 * (time.perf_counter() - t0)
        t0 = time.perf_counter()
        sv = np.ascontiguousarray(set_keys).view("V57").reshape(-1)
        srt = np.argsort(sv, kind="stable")
        q = h_pk.view("V57").reshape(-1)
        pos = np.minimum(np.searchsorted(sv[srt], q), max(len(sv) - 1, 0))
        np_idx = np.where(sv[srt][pos] == q, srt[pos], len(set_keys)).astype(np.uint32) if len(sv) else np.full(n, 0, np.uint32)
        np_ms = 1e3 * (time.perf_counter() - t0)
        assert (dict_idx == np_idx).all()
        miss_fraction = float((np_idx == len(set_keys)).mean())
        for layout, policy in (("flat", DEFAULT_POLICY), ("compact", 0)):
            lib.keyset_policy(policy)
            try:
                t0 = time.perf_counter()
                h = lib.keyset_create(set_keys)
                create_ms = 1e3 * (time.perf_counter() - t0)
            finally:
                lib.keyset_policy(DEFAULT_POLICY)
            try:
                lookup = lambda: lib._call("goldilocks_ed448_verify_keyset_lookup_batch", h_st, h_idx, h, h_sig, h_pk, h_msg, h_off, C.c_uint8(0), None,
                                           C.c_uint8(0), C.c_size_t(n))
                base = lambda: lib._call("goldilocks_ed448_verify_batch", h_st, h_sig, h_pk, h_msg, h_off, C.c_uint8(0), None, C.c_uint8(0), C.c_size_t(n))
                index = lambda: lib._call("goldilocks_ed448_verify_keyset_batch", h_st, h, h_idx, h_sig, h_msg, h_off, C.c_uint8(0), None, C.c_uint8(0),
                                          C.c_size_t(n))
                lookup_dev = lambda: eng.ed448_verify_keyset_lookup(d_st, d_idx, h, d_sig, d_pk, d_msg, d_off, d_scratch)
                base_dev = lambda: eng.ed448_verify(d_st, d_sig, d_pk, d_msg, d_off, d_vscratch)
                index_dev = lambda: eng.ed448_verify_keyset(d_st, h, d_idx, d_sig, d_msg, d_off, d_scratch)
                r = {"layout": layout, "keys_in_set": len(set_keys), "miss_fraction": round(miss_fraction, 5), "create_ms": round(create_ms, 2),
                     "host_pinned_ms": {}, "device_ms": {}}
                calls = [("lookup", lookup, lookup_dev), ("verify_batch", base, base_dev)]
                if with_index:
                    calls.append(("index_form", index, index_dev))
                lookup()
                if not ((h_st == want).all() and (h_idx == np_idx).all()):
                    raise SystemExit("keyset_lookup_bench: the lookup call disagrees with verify_batch on %s (%s)" % (name, layout))
                d_idx.copy_(torch.from_numpy(np_idx.view(np.int32)))
                for cname, hf, df in calls:
                    h_st[:] = 7
                    r["host_pinned_ms"][cname] = round(host_timed(hf), 3)
                    if not (h_st == want).all():
                        raise SystemExit("keyset_lookup_bench: %s (host) disagrees with verify_batch on %s (%s)" % (cname, name, layout))
                    d_st.fill_(7)
                    r["device_ms"][cname] = round(dev_timed(df), 3)
                    if not (d_st.cpu().numpy() == want).all():
                        raise SystemExit("keyset_lookup_bench: %s (device) disagrees with verify_batch on %s (%s)" % (cname, name, layout))
                    if not (d_idx.cpu().numpy().view(np.uint32) == np_idx).all():
                        raise SystemExit("keyset_lookup_bench: the device key_index disagrees on %s (%s)" % (name, layout))
            finally:
                lib.keyset_destroy(h)
            for form in ("host_pinned_ms", "device_ms"):
                t = r[form]
                r[form.replace("_ms", "_Mverifies")] = {k: round(n / v / 1e3, 2) for k, v in t.items()}
                r[form.replace("_ms", "_lookup_vs")] = {k: round(v / t["lookup"], 3) for k, v in t.items() if k != "lookup"}
            r["outputs_identical_to_verify_batch"] = True
            rec["corpora"]["%s, %s" % (name, layout)] = r
            print("%-32s %-7s miss %.3f  host: lookup %.2f M/s, verify_batch x%.2f%s  device: lookup %.2f M/s, verify_batch x%.2f%s" %
                  (name, layout, miss_fraction, r["host_pinned_Mverifies"]["lookup"], r["host_pinned_lookup_vs"]["verify_batch"],
                   (", index x%.2f" % r["host_pinned_lookup_vs"]["index_form"]) if with_index else "",
                   r["device_Mverifies"]["lookup"], r["device_lookup_vs"]["verify_batch"],
                   (", index x%.2f" % r["device_lookup_vs"]["index_form"]) if with_index else ""), flush=True)
        rec["corpora"][name + ", host mapping"] = {"python_dict_ms": round(dict_ms, 1), "numpy_searchsorted_ms": round(np_ms, 1)}
        print("%-32s host mapping of key bytes to indices: dict %.1f ms, numpy %.1f ms" % (name, dict_ms, np_ms), flush=True)
        del d_sig, d_pk, d_msg, d_scratch, d_vscratch
    rec["create"] = create_times(lib, keys, "this tree")
    print(json.dumps({"device": rec["device"], "power_limit_and_max_sm_clock": rec["power_limit_and_max_sm_clock"]}))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
