#!/usr/bin/env python3
"""X448 against a peer set by the peer's bytes (goldilocks_x448_peerset_lookup_batch[_dev]) against the ladder on the same (u, k)
pairs, on one GPU (DESIGN.md decision 24).

    python tools/x448_peerset_lookup_bench.py [--n 1048576] [--reps 10] [--parent-lib PATH] [--out FILE.json]

Corpora of n fresh scalars, each against the u bytes of a peer: 1 peer; 2^10 peers sorted by peer and in random order; 2^16
peers, 16 scalars each, in random order; 2^10 peers in random order with every 32nd u a key outside the set; and all u outside
a set of 2^10 peers.  For each:
  device  : goldilocks_x448_batch_dev against goldilocks_x448_peerset_lookup_batch_dev, the two alternated call by call, CUDA
            events around each call after a warm-up; outputs and statuses compared byte for byte
  host    : goldilocks_x448_batch against goldilocks_x448_peerset_lookup_batch from pinned host buffers (copies included),
            alternated the same way
  kernels : per-launch CUDA-event times of one call of each (goldilocks_b200_profile): the lookup's and the sort's share
plus the creation time of sets of 2^10 and 2^16 peers (median of 5), alternated with the library at --parent-lib when given.
The device name and power limit are recorded beside the numbers.  The inputs total 2^20 x (56 + 56) bytes: they fit the
126 MB L2, as they would for a caller whose batch is in HBM.
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from x448_peerset_bench import device_info, kernel_times  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--parent-lib", default=None, help="another build of libgoldilocks_b200.so whose set creation is timed alongside")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("x448_peerset_lookup_bench: no CUDA device (this measures the GPU; there is no CPU number to give)")
    import libgoldilocks_b200 as g
    from libgoldilocks_b200.capi import BatchLib
    from libgoldilocks_b200.engine import DeviceEngine
    from util import stream_bytes
    lib, eng = g.load(), DeviceEngine()
    n = args.n
    rec = dict(device_info(torch), n=n, reps=args.reps, corpora={}, create={})
    k = stream_bytes("pslb/k", n * 56).reshape(n, 56)
    d_k = torch.from_numpy(k).cuda()
    d_out = torch.empty((n, 56), dtype=torch.uint8, device="cuda")
    d_st = torch.empty(n, dtype=torch.int32, device="cuda")
    d_out2, d_st2 = torch.empty_like(d_out), torch.empty_like(d_st)
    d_scratch = torch.empty(eng.x448_peerset_scratch_bytes(n), dtype=torch.uint8, device="cuda")
    pinned = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory().numpy()
    h_k = torch.from_numpy(k).pin_memory().numpy()
    h_u = pinned((n, 56), torch.uint8)
    h_out, h_out2 = pinned((n, 56), torch.uint8), pinned((n, 56), torch.uint8)
    h_st, h_st2 = pinned(n, torch.int32), pinned(n, torch.int32)

    def alternate_device(fa, fb):
        fa(); fb()
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(2 * args.reps)]
        for r in range(args.reps):
            for j, fn in enumerate((fa, fb)):
                a, b = ev[2 * r + j]
                a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ta = sum(ev[2 * r][0].elapsed_time(ev[2 * r][1]) for r in range(args.reps)) / args.reps
        tb = sum(ev[2 * r + 1][0].elapsed_time(ev[2 * r + 1][1]) for r in range(args.reps)) / args.reps
        return ta, tb

    def alternate_host(fa, fb):
        fa(); fb()
        ta = tb = 0.0
        for _ in range(args.reps):
            t = time.perf_counter(); fa(); ta += time.perf_counter() - t
            t = time.perf_counter(); fb(); tb += time.perf_counter() - t
        return 1e3 * ta / args.reps, 1e3 * tb / args.reps

    rng = np.random.default_rng(11)
    corpora = (("1 peer", 1, "random", 0), ("1024 peers, sorted by peer", 1024, "sorted", 0), ("1024 peers, random order", 1024, "random", 0),
               ("65536 peers, 16 per peer, random order", 65536, "random", 0), ("1024 peers, random order, 1/32 misses", 1024, "random", 32),
               ("all misses (1024-peer set)", 1024, "random", 1))
    for name, m, order, miss_every in corpora:
        peers = lib.x448_derive_public_key(stream_bytes("pslb/peers%d" % m, m * 56).reshape(m, 56))
        idx = (np.arange(n, dtype=np.uint64) * m // n).astype(np.uint32)        # n / m scalars per peer
        if order == "random":
            rng.shuffle(idx)
        u = peers[idx]
        if miss_every:
            q = len(u[::miss_every])
            u[::miss_every] = lib.x448_derive_public_key(stream_bytes("pslb/miss%d" % miss_every, q * 56).reshape(q, 56))
        h_u[:] = u
        d_u = torch.from_numpy(h_u).cuda()
        h = lib.x448_peerset_create(peers)
        try:
            ladder, lookup = alternate_device(lambda: eng.x448(d_out, d_st, d_u, d_k),
                                              lambda: eng.x448_peerset_lookup(d_out2, d_st2, None, h, d_u, d_k, d_scratch))
            same = bool(torch.equal(d_out, d_out2) and torch.equal(d_st, d_st2))
            ok = bool((d_st2 == -1).all())
            host_ladder, host_lookup = alternate_host(lambda: lib._call("goldilocks_x448_batch", h_out, h_st, h_u, h_k, C.c_size_t(n)),
                                                      lambda: lib._call("goldilocks_x448_peerset_lookup_batch", h_out2, h_st2, None, h, h_u, h_k, C.c_size_t(n)))
            same_host = bool((h_out == h_out2).all() and (h_st == h_st2).all() and (h_out == d_out.cpu().numpy()).all())
            _, _, looked = lib.x448_peerset_lookup(h, u[:4096], k[:4096], return_index=True)
            kl = kernel_times(lib, lambda: eng.x448(d_out, d_st, d_u, d_k) or torch.cuda.synchronize())
            kc = kernel_times(lib, lambda: eng.x448_peerset_lookup(d_out2, d_st2, None, h, d_u, d_k, d_scratch) or torch.cuda.synchronize())
        finally:
            lib.x448_peerset_destroy(h)
        total = sum(x["ms"] for x in kc)
        slot = sum(x["ms"] for x in kc if "SlotX448PeerLookup" in x["kernel"])
        r = {"peers": m, "order": order, "misses": ("1/%d" % miss_every) if miss_every > 1 else ("all" if miss_every else "none"),
             "hits_in_first_4096": int((looked < m).sum()),
             "device": {"ladder_ms": round(ladder, 3), "lookup_ms": round(lookup, 3), "ladder_Mops": round(n / ladder / 1e3, 2),
                        "lookup_Mops": round(n / lookup / 1e3, 2), "speedup": round(ladder / lookup, 3)},
             "host_pinned": {"ladder_ms": round(host_ladder, 3), "lookup_ms": round(host_lookup, 3), "ladder_Mops": round(n / host_ladder / 1e3, 2),
                             "lookup_Mops": round(n / host_lookup / 1e3, 2), "speedup": round(host_ladder / host_lookup, 3)},
             "kernels": {"ladder": kl, "lookup": kc, "lookup_and_sort_share": round((total - slot) / total, 4) if total else None},
             "outputs_identical_device": same, "outputs_identical_host": same_host, "all_success": ok}
        rec["corpora"][name] = r
        print("%-42s device %.3f -> %.3f ms (%.2f -> %.2f M/s, x%.3f)  host %.2f -> %.2f M/s (x%.3f)  lookup+sort %.2f %%  identical=%s/%s" %
              (name, ladder, lookup, r["device"]["ladder_Mops"], r["device"]["lookup_Mops"], r["device"]["speedup"], r["host_pinned"]["ladder_Mops"],
               r["host_pinned"]["lookup_Mops"], r["host_pinned"]["speedup"], 100 * r["kernels"]["lookup_and_sort_share"], same, same_host), flush=True)
        if not (same and same_host):
            raise SystemExit("x448_peerset_lookup_bench: the lookup call and goldilocks_x448_batch disagree on %s" % name)
    libs = [("this", lib)] + ([("parent", BatchLib(args.parent_lib))] if args.parent_lib else [])
    for m in (1 << 10, 1 << 16):
        peers = lib.x448_derive_public_key(stream_bytes("pslb/create%d" % m, m * 56).reshape(m, 56))
        times = {name: [] for name, _ in libs}
        for name, L in libs:
            L.x448_peerset_destroy(L.x448_peerset_create(peers))   # warm: the arena has grown to this size
        for _ in range(5):
            for name, L in libs:
                t0 = time.perf_counter()
                h = L.x448_peerset_create(peers)
                times[name].append(1e3 * (time.perf_counter() - t0))
                L.x448_peerset_destroy(h)
        rec["create"][str(m)] = {"ms": round(float(np.median(times["this"])), 2), "runs_ms": [round(t, 2) for t in times["this"]],
                                 "kernels": kernel_times(lib, lambda: lib.x448_peerset_destroy(lib.x448_peerset_create(peers)))}
        if args.parent_lib:
            rec["create"][str(m)]["parent_ms"] = round(float(np.median(times["parent"])), 2)
            rec["create"][str(m)]["parent_runs_ms"] = [round(t, 2) for t in times["parent"]]
        print("create %6d peers: %.2f ms%s" % (m, rec["create"][str(m)]["ms"],
                                               "  (parent %.2f ms)" % rec["create"][str(m)]["parent_ms"] if args.parent_lib else ""), flush=True)
    print(json.dumps({"device": rec["device"], "power_limit_and_max_sm_clock": rec["power_limit_and_max_sm_clock"]}))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
