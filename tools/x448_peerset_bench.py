#!/usr/bin/env python3
"""X448 peer sets against the ladder on the same (u, k) pairs, on one GPU (DESIGN.md decision 20).

    python tools/x448_peerset_bench.py [--n 1048576] [--reps 10] [--out FILE.json]

Corpora of n fresh scalars against honest peer keys: 1 peer; 2^10 peers in random order and sorted by peer; 2^16 peers,
16 scalars each, in random order.  For each:
  device  : goldilocks_x448_batch_dev (every element runs the ladder on its own u) against goldilocks_x448_peerset_batch_dev,
            CUDA events around `reps` calls after a warm-up call; outputs and statuses compared byte for byte
  host    : goldilocks_x448_batch against goldilocks_x448_peerset_batch from pinned host buffers (copies included)
  kernels : per-launch CUDA-event times of one call of each (goldilocks_b200_profile)
plus the creation time of sets of 2^10 and 2^16 peers.  The device name and power limit are recorded beside the numbers.
The inputs total 2^20 x (56 + 56 + 4) bytes: they fit the 126 MB L2, as they would for a caller whose batch is in HBM.
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


def device_info(torch):
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.stdout.strip() else q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["power_limit_and_max_sm_clock"] = "unavailable: %s" % e
    return info


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
    out = []
    for k in range(cnt):
        raw = names.raw[64 * k:64 * (k + 1)].split(b"\0")[0].decode()
        out.append({"kernel": raw, "ms": round(float(ms[k]), 4)})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("x448_peerset_bench: no CUDA device (this measures the GPU; there is no CPU number to give)")
    import libgoldilocks_b200 as g
    from libgoldilocks_b200.engine import DeviceEngine
    from util import stream_bytes
    lib, eng = g.load(), DeviceEngine()
    n = args.n
    rec = dict(device_info(torch), n=n, reps=args.reps, corpora={}, create={})
    k = stream_bytes("psb/k", n * 56).reshape(n, 56)
    d_k = torch.from_numpy(k).cuda()
    d_out = torch.empty((n, 56), dtype=torch.uint8, device="cuda")
    d_st = torch.empty(n, dtype=torch.int32, device="cuda")
    d_out2, d_st2 = torch.empty_like(d_out), torch.empty_like(d_st)
    h_k = torch.from_numpy(k).pin_memory().numpy()
    h_out = torch.empty((n, 56), dtype=torch.uint8).pin_memory().numpy()
    h_st = torch.empty(n, dtype=torch.int32).pin_memory().numpy()
    h_idx = torch.empty(n, dtype=torch.int32).pin_memory().numpy().view(np.uint32)
    h_u = torch.empty((n, 56), dtype=torch.uint8).pin_memory().numpy()

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

    rng = np.random.default_rng(7)
    for name, m, order in (("1 peer", 1, "random"), ("1024 peers, random order", 1024, "random"), ("1024 peers, sorted by peer", 1024, "sorted"),
                           ("65536 peers, 16 per peer, random order", 65536, "random")):
        peers = lib.x448_derive_public_key(stream_bytes("psb/peers%d" % m, m * 56).reshape(m, 56))
        idx = (np.arange(n, dtype=np.uint64) * m // n).astype(np.uint32)        # n / m scalars per peer
        if order == "random":
            rng.shuffle(idx)
        h_idx[:] = idx
        h_u[:] = peers[idx]
        d_idx = torch.from_numpy(idx.view(np.int32)).cuda()
        d_u = torch.from_numpy(h_u).cuda()
        t0 = time.perf_counter()
        h = lib.x448_peerset_create(peers)
        create_ms = 1e3 * (time.perf_counter() - t0)
        try:
            ladder = timed(lambda: eng.x448(d_out, d_st, d_u, d_k))
            comb = timed(lambda: eng.x448_peerset(d_out2, d_st2, h, d_idx, d_k))
            same = bool(torch.equal(d_out, d_out2) and torch.equal(d_st, d_st2))
            ok = bool((d_st2 == -1).all())
            host_ladder = host_timed(lambda: lib._call("goldilocks_x448_batch", h_out, h_st, h_u, h_k, C.c_size_t(n)))
            want = h_out.copy()
            host_comb = host_timed(lambda: lib._call("goldilocks_x448_peerset_batch", h_out, h_st, h, h_idx, h_k, C.c_size_t(n)))
            same_host = bool((h_out == want).all())
            kl = kernel_times(lib, lambda: eng.x448(d_out, d_st, d_u, d_k) or torch.cuda.synchronize())
            kc = kernel_times(lib, lambda: eng.x448_peerset(d_out2, d_st2, h, d_idx, d_k) or torch.cuda.synchronize())
        finally:
            lib.x448_peerset_destroy(h)
        r = {"peers": m, "order": order, "create_ms": round(create_ms, 2),
             "device": {"ladder_ms": round(ladder, 3), "peerset_ms": round(comb, 3), "ladder_Mops": round(n / ladder / 1e3, 2),
                        "peerset_Mops": round(n / comb / 1e3, 2), "speedup": round(ladder / comb, 2)},
             "host_pinned": {"ladder_ms": round(host_ladder, 3), "peerset_ms": round(host_comb, 3), "ladder_Mops": round(n / host_ladder / 1e3, 2),
                             "peerset_Mops": round(n / host_comb / 1e3, 2), "speedup": round(host_ladder / host_comb, 2)},
             "kernels": {"ladder": kl, "peerset": kc},
             "outputs_identical_device": same, "outputs_identical_host": same_host, "all_success": ok}
        rec["corpora"][name] = r
        print("%-40s device %.3f -> %.3f ms (%.2f -> %.2f M/s, x%.2f)  host %.2f -> %.2f M/s  identical=%s/%s" %
              (name, ladder, comb, r["device"]["ladder_Mops"], r["device"]["peerset_Mops"], r["device"]["speedup"],
               r["host_pinned"]["ladder_Mops"], r["host_pinned"]["peerset_Mops"], same, same_host), flush=True)
        if not (same and same_host):
            raise SystemExit("x448_peerset_bench: the peer set and the ladder disagree on %s" % name)
    for m in (1 << 10, 1 << 16):
        peers = lib.x448_derive_public_key(stream_bytes("psb/create%d" % m, m * 56).reshape(m, 56))
        h = lib.x448_peerset_create(peers)   # warm: the arena has grown to this size
        lib.x448_peerset_destroy(h)
        t0 = time.perf_counter()
        h = lib.x448_peerset_create(peers)
        rec["create"][str(m)] = {"ms": round(1e3 * (time.perf_counter() - t0), 2),
                                 "kernels": kernel_times(lib, lambda: lib.x448_peerset_destroy(lib.x448_peerset_create(peers)))}
        lib.x448_peerset_destroy(h)
        print("create %6d peers: %.2f ms" % (m, rec["create"][str(m)]["ms"]), flush=True)
    print(json.dumps({"device": rec["device"], "power_limit_and_max_sm_clock": rec["power_limit_and_max_sm_clock"]}))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
