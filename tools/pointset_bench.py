#!/usr/bin/env python3
"""Point sets against goldilocks_448_base_double_scalarmul_non_secret_batch on the same (s1, P, s2) triples, on one GPU (DESIGN.md
decision 22).

    python tools/pointset_bench.py [--n 1048576] [--reps 10] [--out FILE.json]

Corpora of n elements with fresh scalars below q against random points: 1 point; 2^10 points sorted by point and in random order;
2^16 points, 16 elements each, in random order -- all with the flat table layout -- and 2^10 points in random order with the
compact layout (goldilocks_b200_keyset_policy(0)).  For each:
  check   : one call of each; the point set's outputs must encode byte for byte like the baseline's before anything is timed
  host    : goldilocks_448_base_double_scalarmul_non_secret_batch against goldilocks_448_base_double_scalarmul_non_secret_pointset_batch
            from pinned host buffers (copies included), wall clock over `reps` calls after a warm-up call
  device  : goldilocks_448_base_double_scalarmul_non_secret_pointset_batch_dev, CUDA events around `reps` calls, outputs compared
            with the host call's.  The baseline has no device-pointer form, so its device figure is its kernel time in
            goldilocks_b200_profile_timeline
  sort    : the share the sort by point takes of one _dev call (goldilocks_b200_profile_timeline)
plus the creation time of each set and of warm sets of 2^10 and 2^16 points.  The device name, power limit and maximum SM clock
are recorded beside the numbers.
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


def _names(buf, k):
    return buf.raw[64 * k:64 * (k + 1)].split(b"\0")[0].decode()


def timeline(lib, fn):
    """launches of one call as (name, start, end) relative to the first launch"""
    L = lib.lib
    L.goldilocks_b200_profile.restype = None
    L.goldilocks_b200_profile_timeline.restype = C.c_size_t
    names = C.create_string_buffer(64 * 64)
    t0, t1 = (C.c_float * 64)(), (C.c_float * 64)()
    L.goldilocks_b200_profile(C.c_int(1))
    fn()
    L.goldilocks_b200_profile(C.c_int(0))
    cnt = L.goldilocks_b200_profile_timeline(names, t0, t1, C.c_size_t(64))
    return [{"kernel": _names(names, k), "start_ms": round(float(t0[k]), 4), "end_ms": round(float(t1[k]), 4)} for k in range(cnt)]


def span(rows):
    return max(r["end_ms"] for r in rows) - min(r["start_ms"] for r in rows)


def busy(rows, name):
    return sum(r["end_ms"] - r["start_ms"] for r in rows if name in r["kernel"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("pointset_bench: no CUDA device (this measures the GPU; there is no CPU number to give)")
    import libgoldilocks_b200 as g
    from libgoldilocks_b200.engine import DeviceEngine
    from util import stream_bytes
    lib, eng = g.load(), DeviceEngine()
    n = args.n
    rec = dict(device_info(torch), n=n, reps=args.reps, corpora={}, create={})

    def pinned(shape, dtype=torch.uint8):
        return torch.empty(shape, dtype=dtype).pin_memory().numpy()

    h_s1, h_s2 = pinned((n, 56)), pinned((n, 56))
    h_s1[:] = lib.scalar_decode_long(stream_bytes("ptb/s1", n * 56).reshape(n, 56), 56)   # fresh scalars below q
    h_s2[:] = lib.scalar_decode_long(stream_bytes("ptb/s2", n * 56).reshape(n, 56), 56)
    h_base, h_out, h_out2 = pinned((n, 256)), pinned((n, 256)), pinned((n, 256))
    h_idx = pinned(n, torch.int32).view(np.uint32)
    d_s1, d_s2 = torch.from_numpy(h_s1).cuda(), torch.from_numpy(h_s2).cuda()
    d_out = torch.empty((n, 256), dtype=torch.uint8, device="cuda")
    d_scratch = torch.empty(eng.pointset_scratch_bytes(n), dtype=torch.uint8, device="cuda")

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

    def points_of(label, m):
        return lib.from_hash_uniform(stream_bytes(label, m * 112).reshape(m, 112))

    rng = np.random.default_rng(7)
    for name, m, order, layout in (("1 point", 1, "random", "flat"), ("1024 points, sorted by point", 1024, "sorted", "flat"),
                                   ("1024 points, random order", 1024, "random", "flat"),
                                   ("65536 points, 16 per point, random order", 65536, "random", "flat"),
                                   ("1024 points, random order, compact layout", 1024, "random", "compact")):
        points = points_of("ptb/points%d" % m, m)
        idx = (np.arange(n, dtype=np.uint64) * m // n).astype(np.uint32)        # n / m elements per point
        if order == "random":
            rng.shuffle(idx)
        h_idx[:] = idx
        h_base[:] = points[idx]
        d_idx = torch.from_numpy(idx.view(np.int32)).cuda()
        lib.keyset_policy(DEFAULT_POLICY if layout == "flat" else 0)
        try:
            t0 = time.perf_counter()
            h = lib.pointset_create(points)
            create_ms = 1e3 * (time.perf_counter() - t0)
        finally:
            lib.keyset_policy(DEFAULT_POLICY)
        try:
            base_call = lambda: lib._call("goldilocks_448_base_double_scalarmul_non_secret_batch", h_out, h_s1, h_base, h_s2, C.c_size_t(n))
            set_call = lambda: lib._call("goldilocks_448_base_double_scalarmul_non_secret_pointset_batch", h_out2, h, h_idx, h_s1, h_s2, C.c_size_t(n))
            dev_call = lambda: eng.pointset(d_out, h, d_idx, d_s1, d_s2, d_scratch)
            base_call()
            set_call()
            same_enc = bool((lib.point_encode(h_out) == lib.point_encode(h_out2)).all())
            if not same_enc:
                raise SystemExit("pointset_bench: the point set and base_double_scalarmul_non_secret_batch disagree on %s" % name)
            host_base = host_timed(base_call)
            host_set = host_timed(set_call)
            dev = timed(dev_call)
            same_dev = bool((d_out.cpu().numpy() == h_out2).all())
            tl_base = timeline(lib, base_call)
            tl_set = timeline(lib, lambda: dev_call() or torch.cuda.synchronize())
        finally:
            lib.pointset_destroy(h)
        base_kernel = busy(tl_base, "SlotBaseDoubleScalarmul")
        sort_ms, set_span = busy(tl_set, "pair_sort"), span(tl_set)
        r = {"points": m, "order": order, "layout": layout, "create_ms": round(create_ms, 2),
             "host_pinned": {"baseline_ms": round(host_base, 3), "pointset_ms": round(host_set, 3), "baseline_Mops": round(n / host_base / 1e3, 2),
                             "pointset_Mops": round(n / host_set / 1e3, 2), "speedup": round(host_base / host_set, 2)},
             "device": {"baseline_kernel_ms": round(base_kernel, 3), "pointset_dev_ms": round(dev, 3), "baseline_kernel_Mops": round(n / base_kernel / 1e3, 2),
                        "pointset_dev_Mops": round(n / dev / 1e3, 2), "speedup": round(base_kernel / dev, 2)},
             "sort": {"sort_ms": round(sort_ms, 4), "call_span_ms": round(set_span, 4), "share": round(sort_ms / set_span, 4)},
             "timeline_baseline": tl_base, "timeline_pointset_dev": tl_set,
             "encodings_identical_to_baseline": same_enc, "dev_identical_to_host": same_dev}
        rec["corpora"][name] = r
        print("%-44s host %.2f -> %.2f M/s (x%.2f)  device %.2f -> %.2f M/s (x%.2f)  sort %.2f %% of the call  identical=%s/%s" %
              (name, r["host_pinned"]["baseline_Mops"], r["host_pinned"]["pointset_Mops"], r["host_pinned"]["speedup"],
               r["device"]["baseline_kernel_Mops"], r["device"]["pointset_dev_Mops"], r["device"]["speedup"], 100 * r["sort"]["share"],
               same_enc, same_dev), flush=True)
        if not same_dev:
            raise SystemExit("pointset_bench: the _dev call and the host call disagree on %s" % name)
    for m in (1 << 10, 1 << 16):
        points = points_of("ptb/create%d" % m, m)
        lib.pointset_destroy(lib.pointset_create(points))   # warm: the arena has grown to this size
        t0 = time.perf_counter()
        h = lib.pointset_create(points)
        ms = 1e3 * (time.perf_counter() - t0)
        lib.pointset_destroy(h)
        rec["create"][str(m)] = {"ms": round(ms, 2), "timeline": timeline(lib, lambda: lib.pointset_destroy(lib.pointset_create(points)))}
        print("create %6d points (flat): %.2f ms" % (m, ms), flush=True)
    print(json.dumps({"device": rec["device"], "power_limit_and_max_sm_clock": rec["power_limit_and_max_sm_clock"]}))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
