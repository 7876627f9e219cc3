#!/usr/bin/env python3
"""Decaf peer sets against goldilocks_448_direct_scalarmul_batch on the same (peer, scalar) pairs, on one GPU (DESIGN.md
decision 21).

    python tools/decaf_peerset_bench.py [--n 1048576] [--reps 10] [--out FILE.json]

Corpora of n fresh scalars below q against valid peer encodings: 1 peer; 2^10 peers sorted by peer and in random order;
2^16 peers, 16 scalars each, in random order.  For each:
  host    : goldilocks_448_direct_scalarmul_batch against goldilocks_448_direct_scalarmul_peerset_batch from pinned host
            buffers (copies included), wall clock over `reps` calls after a warm-up call; outputs compared byte for byte
  device  : goldilocks_448_direct_scalarmul_peerset_batch_dev, CUDA events around `reps` calls; its outputs compared with the
            host call's.  direct_scalarmul has no device-pointer form, so its device figure is the sum of its kernel times
  kernels : per-launch CUDA-event times of one call of each (goldilocks_b200_profile), and the timeline of one _dev call
            (goldilocks_b200_profile_timeline) with the share the sort by peer takes of it
plus the creation time of sets of 2^10 and 2^16 peers.  The device name and power limit are recorded beside the numbers.
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
ALL = C.c_uint64((1 << 64) - 1)


def device_info(torch):
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.stdout.strip() else q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = "unavailable: %s" % e
    return info


def _names(buf, k):
    return buf.raw[64 * k:64 * (k + 1)].split(b"\0")[0].decode()


def kernel_times(lib, fn):
    L = lib.lib
    L.goldilocks_b200_profile.restype = None
    L.goldilocks_b200_profile_read.restype = C.c_size_t
    names = C.create_string_buffer(64 * 64)
    ms = (C.c_float * 64)()
    L.goldilocks_b200_profile(C.c_int(1))
    fn()
    L.goldilocks_b200_profile(C.c_int(0))
    cnt = L.goldilocks_b200_profile_read(names, ms, C.c_size_t(64))
    return [{"kernel": _names(names, k), "ms": round(float(ms[k]), 4)} for k in range(cnt)]


def timeline(lib, fn):
    """launches of one call as (name, start, end) relative to the first launch, and the sort's share of the whole span"""
    L = lib.lib
    L.goldilocks_b200_profile.restype = None
    L.goldilocks_b200_profile_timeline.restype = C.c_size_t
    names = C.create_string_buffer(64 * 64)
    t0, t1 = (C.c_float * 64)(), (C.c_float * 64)()
    L.goldilocks_b200_profile(C.c_int(1))
    fn()
    L.goldilocks_b200_profile(C.c_int(0))
    cnt = L.goldilocks_b200_profile_timeline(names, t0, t1, C.c_size_t(64))
    rows = [{"kernel": _names(names, k), "start_ms": round(float(t0[k]), 4), "end_ms": round(float(t1[k]), 4)} for k in range(cnt)]
    span = max(r["end_ms"] for r in rows) - min(r["start_ms"] for r in rows)
    sort = sum(r["end_ms"] - r["start_ms"] for r in rows if r["kernel"] == "pair_sort")
    return rows, sort, span


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("decaf_peerset_bench: no CUDA device (this measures the GPU; there is no CPU number to give)")
    import libgoldilocks_b200 as g
    from libgoldilocks_b200.engine import DeviceEngine
    from util import stream_bytes
    lib, eng = g.load(), DeviceEngine()
    n = args.n
    rec = dict(device_info(torch), n=n, reps=args.reps, corpora={}, create={})
    sc = lib.scalar_decode_long(stream_bytes("dpb/k", n * 56).reshape(n, 56), 56)     # fresh scalars below q
    d_sc = torch.from_numpy(sc).cuda()
    d_out = torch.empty((n, 56), dtype=torch.uint8, device="cuda")
    d_st = torch.empty(n, dtype=torch.int32, device="cuda")
    d_scratch = torch.empty(eng.decaf_peerset_scratch_bytes(n), dtype=torch.uint8, device="cuda")
    h_sc = torch.from_numpy(sc).pin_memory().numpy()
    h_out = torch.empty((n, 56), dtype=torch.uint8).pin_memory().numpy()
    h_out2 = torch.empty((n, 56), dtype=torch.uint8).pin_memory().numpy()
    h_st = torch.empty(n, dtype=torch.int32).pin_memory().numpy()
    h_st2 = torch.empty(n, dtype=torch.int32).pin_memory().numpy()
    h_idx = torch.empty(n, dtype=torch.int32).pin_memory().numpy().view(np.uint32)
    h_base = torch.empty((n, 56), dtype=torch.uint8).pin_memory().numpy()

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / args.reps

    def host_timed(fn):
        fn()
        t = time.perf_counter()
        for _ in range(args.reps):
            fn()
        return 1e3 * (time.perf_counter() - t) / args.reps

    def peers_of(label, m):
        return lib.point_encode(lib.from_hash_uniform(stream_bytes(label, m * 112).reshape(m, 112)))

    rng = np.random.default_rng(7)
    for name, m, order in (("1 peer", 1, "random"), ("1024 peers, sorted by peer", 1024, "sorted"), ("1024 peers, random order", 1024, "random"),
                           ("65536 peers, 16 per peer, random order", 65536, "random")):
        peers = peers_of("dpb/peers%d" % m, m)
        idx = (np.arange(n, dtype=np.uint64) * m // n).astype(np.uint32)        # n / m scalars per peer
        if order == "random":
            rng.shuffle(idx)
        h_idx[:] = idx
        h_base[:] = peers[idx]
        d_idx = torch.from_numpy(idx.view(np.int32)).cuda()
        t0 = time.perf_counter()
        h = lib.decaf_peerset_create(peers)
        create_ms = 1e3 * (time.perf_counter() - t0)
        try:
            direct_call = lambda: lib._call("goldilocks_448_direct_scalarmul_batch", h_out, h_st, h_base, h_sc, C.c_uint64(0), C.c_uint64(0), C.c_size_t(n))
            peer_call = lambda: lib._call("goldilocks_448_direct_scalarmul_peerset_batch", h_out2, h_st2, h, h_idx, h_sc, C.c_uint64(0), C.c_size_t(n))
            dev_call = lambda: eng.decaf_peerset(d_out, d_st, h, d_idx, d_sc, d_scratch, short_circuit=False)
            host_direct = host_timed(direct_call)
            host_peer = host_timed(peer_call)
            same_host = bool((h_out == h_out2).all() and (h_st == h_st2).all())
            ok = bool((h_st == -1).all())
            dev = timed(dev_call)
            same_dev = bool((d_out.cpu().numpy() == h_out).all() and (d_st.cpu().numpy() == h_st).all())
            kd = kernel_times(lib, direct_call)
            kp = kernel_times(lib, lambda: dev_call() or torch.cuda.synchronize())
            tl, sort_ms, span_ms = timeline(lib, lambda: dev_call() or torch.cuda.synchronize())
        finally:
            lib.decaf_peerset_destroy(h)
        direct_kernels = sum(k["ms"] for k in kd)
        r = {"peers": m, "order": order, "create_ms": round(create_ms, 2),
             "host_pinned": {"direct_ms": round(host_direct, 3), "peerset_ms": round(host_peer, 3), "direct_Mops": round(n / host_direct / 1e3, 2),
                             "peerset_Mops": round(n / host_peer / 1e3, 2), "speedup": round(host_direct / host_peer, 2)},
             "device": {"direct_kernels_ms": round(direct_kernels, 3), "peerset_dev_ms": round(dev, 3), "direct_kernels_Mops": round(n / direct_kernels / 1e3, 2),
                        "peerset_dev_Mops": round(n / dev / 1e3, 2), "speedup": round(direct_kernels / dev, 2)},
             "sort": {"sort_ms": round(sort_ms, 4), "call_span_ms": round(span_ms, 4), "share": round(sort_ms / span_ms, 4)},
             "kernels": {"direct_scalarmul": kd, "peerset_dev": kp}, "timeline_peerset_dev": tl,
             "outputs_identical_host": same_host, "outputs_identical_dev": same_dev, "all_success": ok}
        rec["corpora"][name] = r
        print("%-40s host %.2f -> %.2f M/s (x%.2f)  device %.2f -> %.2f M/s (x%.2f)  sort %.1f %% of the call  identical=%s/%s" %
              (name, r["host_pinned"]["direct_Mops"], r["host_pinned"]["peerset_Mops"], r["host_pinned"]["speedup"],
               r["device"]["direct_kernels_Mops"], r["device"]["peerset_dev_Mops"], r["device"]["speedup"], 100 * r["sort"]["share"],
               same_host, same_dev), flush=True)
        if not (same_host and same_dev):
            raise SystemExit("decaf_peerset_bench: the peer set and direct_scalarmul disagree on %s" % name)
    for m in (1 << 10, 1 << 16):
        peers = peers_of("dpb/create%d" % m, m)
        h = lib.decaf_peerset_create(peers)   # warm: the arena has grown to this size
        lib.decaf_peerset_destroy(h)
        t0 = time.perf_counter()
        h = lib.decaf_peerset_create(peers)
        rec["create"][str(m)] = {"ms": round(1e3 * (time.perf_counter() - t0), 2),
                                 "kernels": kernel_times(lib, lambda: lib.decaf_peerset_destroy(lib.decaf_peerset_create(peers)))}
        lib.decaf_peerset_destroy(h)
        print("create %6d peers: %.2f ms" % (m, rec["create"][str(m)]["ms"]), flush=True)
    print(json.dumps({"device": rec["device"], "power_limit_and_max_sm_clock": rec["power_limit_and_max_sm_clock"]}))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
