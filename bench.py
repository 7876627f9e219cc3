#!/usr/bin/env python3
"""bench.py -- BASELINE.json's metric on its own config: Ed448 verifies/s at batch 2^20 (configs[3]); the other
configs ride along in `extra`: field / point ops (config 1), fixed-base comb (2), X448 (3), decaf + Elligator (5),
sign, variable-base multiplications, and ONE batch sharded over all N GPUs by the library (`extra.strong`).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   our arm  (under torchrun for N > 1)
  python bench.py --impl reference [...]                        the reference's CPU path on all host cores

A step = one pass of the hot path over one batch of 2^20 synthetic signatures per GPU.  Two multi-GPU readings:
  * `value` (weak scaling, one process per GPU as the contract launches it): every rank verifies its own 2^20 batch,
    no collective on the data path -- torch.distributed (gloo: there is nothing to exchange, so no NCCL) only carries
    the barrier and the max-over-ranks time;
  * `extra.strong`: rank 0 alone drives ONE batch through the library's own device set
    (goldilocks_b200_set_devices: contiguous ranges, a worker thread per device, no collective) while the other ranks
    wait -- Ed448 verify and X448 at 2^20, decaf encode + decode + Elligator at 2^24 (BASELINE configs[4]).

`value`   : device-resident -- inputs already in HBM, CUDA events on the launching stream.
`e2e`     : the same batch through the host-pointer C-ABI call with pinned host buffers; H2D + kernels + D2H timed.
`roofline`: the dominant kernel, timed per launch with CUDA events inside the timed region.  `achieved` = IMAD.WIDE the
            kernel EXECUTES per second (counted per functor on the host simulator of the CUDA sources,
            profiles/executed_ops.json), `peak` = the IMAD.WIDE.U32 rate tools/imad_peak measures ON THIS BOX just
            before the timed region, `frac` = achieved / peak.  The reference's algorithmic work (SURVEY 8(d)) over
            the same time is reported beside it as `algorithmic_speedup` -- it exceeds the executed figure wherever the
            engine does less work for the same result (dedicated squaring, per-key tables, no R decode).
`cpu_baseline`: the unmodified reference (oracle/_ref, arch_x86_64) on all host cores over a bounded sample.
The corpus is signed by the REFERENCE (SURVEY 8(d)) and the reference re-verifies all 2^20 signatures once, outside
the timed region.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

N_PER_GPU = 1 << 20
MSG_LEN = 32
# SURVEY.md 8(d): the REFERENCE's algorithmic MAC32 per unit (M = S = 192, w = 16)
MAC32 = {"verify": 981120, "verify_finish": 800300, "x448": 870208, "comb": 142656, "encode": 89696, "decode": 90064, "gf_mul": 192, "point_add": 1552,
         "point_double": 1536, "sign": 233000, "point_scalarmul": 760592, "bdsm": 800300, "elligator": 90672, "elligator_uniform": 182896}
METRIC = "Ed448 verifies/s at batch 2^20 per GPU (X448 and comb ops/s in extra)"
UNIT = "verifies/s"
DTYPE = "u32 limbs (448-bit integers)"
# per user: on a shared machine another user's cache directory is not writable
CACHE = os.environ.get("GOLDILOCKS_B200_BENCH_CACHE", os.path.join(tempfile.gettempdir(), "goldilocks_b200_bench_cache_%d" % os.getuid()))
DUMP_BYTES = 64 << 20


# ------------------------------------------------------------------------------------------------
# peaks
# ------------------------------------------------------------------------------------------------
def imad_peak(device_index, measure=True):
    """IMAD.WIDE.U32 lanes/s of THIS GPU, measured now by tools/imad_peak (built by __graft_entry__.build(), ~2 s, the GPU
    is otherwise idle); the committed figure of round 1 only if the binary is missing or fails."""
    exe = os.path.join(ROOT, "tools", "imad_peak")
    if measure and os.path.exists(exe):
        try:
            env = dict(os.environ, CUDA_VISIBLE_DEVICES=str(device_index))
            out = subprocess.run([exe, "--quick"], capture_output=True, text=True, timeout=120, env=env)
            j = json.loads(out.stdout)
            return float(j["imad_wide_u32_gmac_s"]), {"source": "measured on this box by tools/imad_peak inside this run", "per_clk_per_sm": j["imad_wide_u32_per_clk_per_sm"],
                                                      "sm_mhz_during": j["sm_mhz_during"], "sms": j["sms"], "gpu": j["gpu_name"]}
        except Exception as e:  # noqa: BLE001
            why = "tools/imad_peak failed (%s)" % type(e).__name__
    else:
        why = "tools/imad_peak not built" if measure else "measurement skipped (--no-peak, or not rank 0)"
    try:
        with open(os.path.join(ROOT, "profiles", "r01_imad_peak.json")) as f:
            j = json.load(f)
        return float(j["imad_wide_u32_gmac_s"]), {"source": "committed profiles/r01_imad_peak.json (%s)" % why}
    except Exception:  # noqa: BLE001
        return 148 * 32 * 1.965, {"source": "nominal 148 SMs x 32 IMAD.WIDE/clk x 1.965 GHz (%s)" % why}


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback"


def executed_ops():
    """IMAD.WIDE each kernel executes per element, counted on the host simulator (tools/count_ops.py)"""
    with open(os.path.join(ROOT, "profiles", "executed_ops.json")) as f:
        j = json.load(f)
    inv = j["_device_only"]["gf_invert_imad_wide"]
    shared_inv = -0.75 * inv + 9 / 4 * 193          # device: one inversion per four lanes (slot_algos.cuh s_block_invert4)
    ops = {"gf_mul": j["gf_mul"]["_total_imad_wide"], "point_add": j["point_add"]["_total_imad_wide"], "point_double": j["point_double"]["_total_imad_wide"],
           "comb": j["precomputed_scalarmul"]["_total_imad_wide"], "x448": j["x448"]["_total_imad_wide"] + shared_inv,
           "encode": j["point_encode"]["_total_imad_wide"], "decode": j["point_decode"]["_total_imad_wide"],
           "elligator": j["from_hash_nonuniform"]["_total_imad_wide"], "elligator_uniform": j["from_hash_uniform"]["_total_imad_wide"],
           "sign": j["ed448_sign"]["_total_imad_wide"] + shared_inv, "derive_public_key": j["ed448_derive_public_key"]["_total_imad_wide"] + shared_inv,
           "point_scalarmul": j["point_scalarmul"]["_total_imad_wide"], "bdsm": j["base_double_scalarmul_non_secret"]["_total_imad_wide"],
           "verify_16_per_key": j["ed448_verify_16_per_key"]["_total_imad_wide"], "verify_distinct": j["ed448_verify_distinct_keys"]["_total_imad_wide"],
           "verify_64_per_key": j["ed448_verify_64_per_key"]["_total_imad_wide"], "verify_one_signer": j["ed448_verify_one_signer"]["SlotEdVerifyFinishShared"]["imad_wide"] + j["ed448_verify_one_signer"]["LaneVerifySign"]["imad_wide"],   # one table per 2^20 signatures: its build does not count
           
           "verify_keyset": j["ed448_verify_keyset"]["_total_imad_wide"], "verify_keyset_compact": j["ed448_verify_keyset_compact"]["_total_imad_wide"],
           "finish_shared": j["ed448_verify_16_per_key"]["SlotEdVerifyFinishShared"]["imad_wide"],
           "finish_alone": j["ed448_verify_distinct_keys"]["SlotEdVerifyFinishShared"]["imad_wide"],
           "key_table": (j["ed448_verify_16_per_key"]["SlotKeyChain"]["imad_wide"] + j["ed448_verify_16_per_key"]["SlotKeyColumns"]["imad_wide"])
                        / j["ed448_verify_16_per_key"]["SlotKeyChain"]["lanes_per_unit"]}   # per key: the chain has one lane per key
    return ops


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel per launch, from the newest committed
    `ncu --set full` summary of this workload (profiles/r02*_finish_ncu.txt, else round 1's); (bytes, file) or (None, None)."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r02*_finish_ncu.txt"))) or [os.path.join(ROOT, "profiles", "r01f_finish_ncu.txt")]
    try:
        tot, mult = 0.0, {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        with open(files[-1]) as f:
            for line in f:
                t = line.split()
                if len(t) >= 3 and t[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    tot += float(t[2]) * mult[t[1]]
        return (tot or None), os.path.relpath(files[-1], ROOT)
    except Exception:  # noqa: BLE001
        return None, None


# ------------------------------------------------------------------------------------------------
# workload (synthetic, seeded): 2^16 keys x 16 messages of 32 bytes, 1/8 corrupted, SIGNED BY THE REFERENCE
# ------------------------------------------------------------------------------------------------
def make_corpus(signer, n, label, per=16, varlen=False, corrupt=True):
    """varlen: message lengths uniform in [0, 256) (SURVEY 8(d) C4, second run) instead of MSG_LEN bytes each"""
    from util import stream_bytes
    nk = max(1, n // per)
    sk = stream_bytes(label + "/sk", nk * 57).reshape(nk, 57)
    pk = signer.ed448_derive_public_key(sk)
    sk_all = np.repeat(sk, per, axis=0)[:n]
    pk_all = np.repeat(pk, per, axis=0)[:n].copy()
    if varlen:
        lens = stream_bytes(label + "/len", n).astype(np.uint64)
        off = np.concatenate([np.zeros(1, np.uint64), np.cumsum(lens, dtype=np.uint64)])
        arena = stream_bytes(label + "/msg", int(off[-1]) + 1)
    else:
        arena = stream_bytes(label + "/msg", n * MSG_LEN)
        off = np.arange(n + 1, dtype=np.uint64) * MSG_LEN
    sig = signer.ed448_sign(sk_all, pk_all, (arena, off))
    kinds = np.zeros(n, np.int32)
    if corrupt:
        kinds[::8] = 1 + (np.arange((n + 7) // 8) % 4)
    sel = stream_bytes(label + "/sel", n)
    i = np.flatnonzero(kinds == 1); sig[i, sel[i] % 57] ^= 1
    i = np.flatnonzero(kinds == 2); sig[i, 57 + sel[i] % 56] ^= 2
    i = np.flatnonzero(kinds == 3); pk_all[i, sel[i] % 57] ^= 4
    i = np.flatnonzero(kinds == 4)
    if varlen:
        i = i[off[i + 1] > off[i]]                       # an empty message has no byte to flip: left valid
        kinds[np.setdiff1d(np.flatnonzero(kinds == 4), i)] = 0
        arena[(off[i] + sel[i] % (off[i + 1] - off[i])).astype(np.int64)] ^= 8
    else:
        arena[i * MSG_LEN + sel[i] % MSG_LEN] ^= 8
    expect = np.where(kinds == 0, -1, 0).astype(np.int32)
    return sig, pk_all, arena, off, expect


def reference_signer():
    """the compiled reference (oracle/_ref) on all host cores: the corpus' signatures are its goldilocks_ed448_sign output"""
    import util
    ref = util.ref_lib()
    kind = "reference"
    if ref is None:
        ref, kind = util.oracle_lib(), "port"
    util.set_threads(ref, host_cores())
    return ref, kind


def cached_corpus(n, label, rank, world, barrier, **kw):
    """One signing per box: rank 0 makes the corpus with the reference and parks it under CACHE (the driver runs N = 1, 2,
    4, 8 back to back on one box), the other ranks load it and rotate it by their share so no two ranks see the same order."""
    tag = "%s_n%d_%s.npz" % (label.replace("/", "_"), n, "_".join("%s%s" % (k, v) for k, v in sorted(kw.items())))
    path = os.path.join(CACHE, tag)
    if rank == 0 and not os.path.exists(path):
        os.makedirs(CACHE, exist_ok=True)
        signer, _ = reference_signer()
        sig, pk, arena, off, expect = make_corpus(signer, n, label, **kw)
        tmp = path + ".tmp%d.npz" % os.getpid()
        np.savez(tmp, sig=sig, pk=pk, arena=arena, off=off, expect=expect)
        os.replace(tmp, path)
    barrier()
    z = np.load(path)
    sig, pk, arena, off, expect = z["sig"], z["pk"], z["arena"], z["off"], z["expect"]
    shift = (n // world) * rank // 16 * 16
    if shift and not kw.get("varlen"):
        sig, pk, expect = np.roll(sig, shift, axis=0), np.roll(pk, shift, axis=0), np.roll(expect, shift)
        arena = np.roll(arena[: n * MSG_LEN].reshape(n, MSG_LEN), shift, axis=0).reshape(-1)
    return np.ascontiguousarray(sig), np.ascontiguousarray(pk), np.ascontiguousarray(arena), np.ascontiguousarray(off), expect


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc, self.window = index, [], None, None

    def start(self):
        """started before the warm-up steps (nvidia-smi needs ~0.1 s to deliver its first sample); mark() brackets the timed region"""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def mark(self, t0, t1):
        self.window = (t0, t1)

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:  # noqa: BLE001
                self.proc.kill()
        rows, where = [r for _, r in self.rows], "warm-up + timed region (same load)"
        if self.window:
            inside = [r for t, r in self.rows if self.window[0] <= t <= self.window[1] + 0.02]
            if inside:
                rows, where = inside, "timed region"
        sm = [float(r[1]) for r in rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": where}


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        return os.cpu_count() or 1


def cpu_reference_rate(n_sample, steps, warmup, corpus=None):
    """The reference's own goldilocks_ed448_verify over `n_sample` signatures of the bench corpus, all host cores."""
    ref, kind = reference_signer()
    cores = host_cores()
    if corpus is None:
        corpus = make_corpus(ref, n_sample, "bench/cpu")
    sig, pk, arena, off, expect = corpus
    sig, pk, arena, off, expect = sig[:n_sample], pk[:n_sample], arena[: n_sample * MSG_LEN], off[: n_sample + 1], expect[:n_sample]
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        st = ref.ed448_verify(sig, pk, (arena, off))
        dt = time.perf_counter() - t0
        assert (st == expect).all(), "reference disagrees with the corpus' expected accept bits"
        if it >= warmup:
            times.append(dt)
    t = sum(times) / len(times)
    return {"value": n_sample / t, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": "%d signatures of the bench corpus (32-byte messages, 1/8 corrupted) per pass, %d timed passes, %s threads via pthreads" % (n_sample, len(times), cores),
            "lib": os.path.basename(ref.path)}, t


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    n_sample = min(N_PER_GPU, 2048 * cores)
    base, t = cpu_reference_rate(n_sample, args.steps, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE,
            "data": "synthetic", "config": config_dict(args.gpus),
            "cpu_baseline": base, "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def config_dict(gpus, per_key=16, n=N_PER_GPU):
    return {"workload": "BASELINE configs[3]: Ed448 batch verify (SHAKE256 + double scalarmul), 2^16 keys x 16 messages of 32 B, 1/8 corrupted, signed by the reference"
                        + ("" if per_key == 16 else " -- NON-DEFAULT corpus: %d signatures per key" % per_key) + ("" if n == N_PER_GPU else " -- NON-DEFAULT batch %d" % n),
            "keys": "SURVEY 8(d) C4: 2^16 distinct keys x 16 signatures each; byte-identical keys of a batch share one per-key table "
                    "(extra.verify_distinct_keys = the same batch size with 2^20 distinct keys, no sharing possible)",
            "signatures_per_gpu_per_step": N_PER_GPU, "parallelism": "independent shards x%d, no collective" % gpus,
            "l2": "inputs+scratch per step (>700 MB) exceed the 126 MB L2; no flush needed"}


class Profile:
    """the library's per-launch CUDA-event log (goldilocks_b200_profile*)"""

    def __init__(self, lib):
        self.lib = lib.lib
        self.lib.goldilocks_b200_profile_read.restype = C.c_size_t
        self.names = C.create_string_buffer(64 * 8192)
        self.ms = (C.c_float * 8192)()

    def start(self):
        self.lib.goldilocks_b200_profile(C.c_int(1))

    def stop(self, per=1):
        """{functor: ms per `per` calls}"""
        self.lib.goldilocks_b200_profile(C.c_int(0))
        cnt = self.lib.goldilocks_b200_profile_read(self.names, self.ms, C.c_size_t(8192))
        out = {}
        for k in range(cnt):
            nm = self.names.raw[64 * k:64 * k + 64].split(b"\0")[0].decode()
            out[nm] = out.get(nm, 0.0) + self.ms[k] / per
        return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    from libgoldilocks_b200.engine import DeviceEngine
    from util import stream_bytes

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import datetime
        os.environ.setdefault("GLOO_SOCKET_IFNAME", "lo")   # one node: never depend on the container's hostname resolving
        dist.init_process_group("gloo", timeout=datetime.timedelta(minutes=30))   # rendezvous, barrier and max-over-ranks only: the data path has no exchange step
    dev = torch.device("cuda", local)
    n = args.n
    K, W = args.steps, args.warmup

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # the integer-multiply peak of this very GPU, before anything of ours runs on it (rank 0; the line is rank 0's)
    peak, peak_how = imad_peak(local, measure=(rank == 0 and not args.no_peak))
    barrier()
    eng = DeviceEngine()
    lib = eng.capi
    prof = Profile(lib)
    ops = executed_ops()
    hbm, _ = hbm_peak()

    # ---- inputs (host, pinned) -----------------------------------------------------------------------
    t_c = time.time()
    sig, pk, arena, off, expect = cached_corpus(n, "bench/c4", rank, world, barrier, per=args.per_key)
    t_corpus = time.time() - t_c

    def pinned(a):
        return torch.from_numpy(np.ascontiguousarray(a)).pin_memory()

    h_sig, h_pk, h_msg = pinned(sig.reshape(-1)), pinned(pk.reshape(-1)), pinned(arena)
    h_off = pinned(off.view(np.int64))
    h_st = torch.empty(n, dtype=torch.int32).pin_memory()
    d_sig, d_pk, d_msg, d_off = (t.to(dev) for t in (h_sig, h_pk, h_msg, h_off))
    d_st = torch.empty(n, dtype=torch.int32, device=dev)
    d_scratch = torch.empty(eng.verify_scratch_bytes(n), dtype=torch.uint8, device=dev)

    def step():
        eng.ed448_verify(d_st, d_sig, d_pk, d_msg, d_off, d_scratch)

    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(W):
        step()
    torch.cuda.synchronize()
    dev_status = d_st.cpu().numpy()
    assert (dev_status == expect).all(), "device verify disagrees with the corpus' expected accept bits"

    # ---- device-resident timed region -------------------------------------------------------------------
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.time()
    l0 = eng.launch_count()
    prof.start()
    e0.record()
    for _ in range(K):
        step()
    e1.record()
    barrier()
    sampler.mark(t_wall0, time.time())
    kavg = prof.stop(per=K)                     # ms per step and kernel (a kernel may launch more than once per step)
    launches = eng.launch_count() - l0
    clocks = sampler.stop()
    t_step = max_over_ranks(e0.elapsed_time(e1) / 1e3 / K)
    if args.dump_outputs and rank == 0:
        dump_output(args.dump_outputs, "verify_status", d_st.cpu().numpy())    # the legs below reuse d_st
    dominant = "SlotEdVerifyFinishShared" if "SlotEdVerifyFinishShared" in kavg else "SlotEdVerifyFinish"
    t_finish = kavg.get(dominant, 0.0) / 1e3
    # signatures whose key occurs at least twice in the batch go through the per-key tables (what the device-side grouping finds)
    _, inv, cnt = np.unique(np.ascontiguousarray(pk).view(np.dtype((np.void, 57))).ravel(), return_inverse=True, return_counts=True)
    n_shared = int((cnt[inv.reshape(-1)] >= 2).sum())
    n_tables = int((cnt >= 2).sum())
    executed = n_shared * ops["finish_shared"] + (n - n_shared) * ops["finish_alone"]
    executed_step = executed + n_tables * ops["key_table"] + n * (ops["verify_16_per_key"] - ops["finish_shared"] - ops["key_table"] / 16)
    traffic, traffic_file = ncu_traffic()
    achieved = executed / t_finish / 1e9 if t_finish > 0 else 0.0
    roofline = {"bound": "imad", "kernel": "k_slots_persist<%s>" % dominant, "achieved": achieved, "peak": peak, "unit": "GMAC32/s (IMAD.WIDE lanes/s)",
                "frac": achieved / peak, "traffic": traffic, "traffic_unit": "bytes/launch (ncu --set full, %s)" % traffic_file,
                "algorithmic_bytes_per_launch": n * (512 + 112 + 8 + 4), "peak_source": peak_how,
                "executed_mac32_per_launch": executed, "executed_mac32_source": "profiles/executed_ops.json (tools/count_ops.py: multiplier calls counted per functor on the host simulator x 193/110/16)",
                "signatures_under_a_shared_key_table": n_shared, "kernel_ms_per_launch": t_finish * 1e3,
                "algorithmic_mac32_per_signature": MAC32["verify_finish"],
                "algorithmic_speedup": n * MAC32["verify_finish"] / t_finish / 1e9 / peak if t_finish > 0 else None,
                "kernel_ms": kavg,
                "hbm": None if not traffic or t_finish <= 0 else {"achieved": traffic / t_finish / 1e9, "peak": hbm, "unit": "GB/s", "frac": traffic / t_finish / 1e9 / hbm,
                                                                  "note": "informational: DRAM traffic of the ncu capture / this run's launch time; the kernel is multiplier-bound"},
                "kernel_share_of_step": t_finish / (e0.elapsed_time(e1) / 1e3 / K) if t_finish > 0 else None,
                "step_frac_executed": executed_step / t_step / 1e9 / peak,
                "step_algorithmic_speedup": n * MAC32["verify"] / t_step / 1e9 / peak,
                "note": "integer-multiply-pipe roofline (north_star). achieved/frac = IMAD.WIDE this kernel really issues per second / the rate tools/imad_peak measured on "
                        "this GPU minutes earlier. algorithmic_speedup divides the REFERENCE's work (SURVEY 8(d): 800 300 MAC32 per double-scalar multiplication) by the same "
                        "time and peak: it is > frac because a squaring costs 110 not 192 and 16 signatures share one per-key table."}

    # ---- end to end through the host-pointer C ABI ---------------------------------------------------------
    fn = lib.lib.goldilocks_ed448_verify_batch
    fn.restype = C.c_int32
    argv = [C.c_void_p(h_st.data_ptr()), C.c_void_p(h_sig.data_ptr()), C.c_void_p(h_pk.data_ptr()), C.c_void_p(h_msg.data_ptr()),
            C.c_void_p(h_off.data_ptr()), C.c_uint8(0), None, C.c_uint8(0), C.c_size_t(n)]
    for _ in range(max(1, W - 1)):
        assert fn(*argv) == -1
    assert (h_st.numpy() == expect).all()
    ke = max(2, min(K, 5))
    barrier()
    t0 = time.perf_counter()
    for _ in range(ke):
        assert fn(*argv) == -1
    torch.cuda.synchronize()
    t_e2e = max_over_ranks((time.perf_counter() - t0) / ke)
    barrier()
    h2d = sig.nbytes + pk.nbytes + arena.nbytes + off.nbytes
    # what the PCIe path of this rank delivers on its own: the same pinned buffers copied to the device with nothing else running on it
    # (all ranks at once, slowest rank reported: at 8 GPUs they share the host's memory system)
    ca, cb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ca.record()
    for _ in range(3):
        for hsrc, ddst in ((h_sig, d_sig), (h_pk, d_pk), (h_msg, d_msg), (h_off, d_off)):
            ddst.copy_(hsrc, non_blocking=True)
    cb.record()
    barrier()
    t_copy = max_over_ranks(ca.elapsed_time(cb) / 1e3 / 3)
    e2e = {"value": world * n / t_e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(4 * n), "ms_per_step": t_e2e * 1e3,
           "api": "goldilocks_ed448_verify_batch (host pointers, pinned)",
           "h2d_gbs_per_rank_copy_alone": h2d / t_copy / 1e9, "h2d_ms_copy_alone": t_copy * 1e3}

    extra = {"corpus_seconds": round(t_corpus, 1)}

    def timed_dev(fnc, reps):
        """device-resident: CUDA events on the launching stream around `reps` calls, max over ranks; seconds per call"""
        for _ in range(2):
            fnc()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a.record()
        for _ in range(reps):
            fnc()
        b.record()
        barrier()
        return max_over_ranks(a.elapsed_time(b) / 1e3 / reps)

    def timed_host(fnc, reps):
        """host-pointer call: (wall seconds per call, kernel seconds per call from the library's per-launch events), max over ranks"""
        fnc()
        barrier()
        prof.start()
        t0 = time.perf_counter()
        for _ in range(reps):
            fnc()
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) / reps
        k = prof.stop(per=reps)
        barrier()
        return max_over_ranks(wall), max_over_ranks(sum(k.values()) / 1e3), k

    def entry(nn, t, key, unit="ops/s", **more):
        """one extra line: whole-job ops/s, the executed-IMAD fraction of the pipe peak and the algorithmic ratio beside it"""
        d = {"value": world * nn / t, "unit": unit, "ms_per_step": t * 1e3, "batch_per_gpu": nn,
             "imad_frac_executed": nn * ops[key] / t / 1e9 / peak, "executed_mac32_per_op": ops[key]}
        if key in MAC32:
            d["algorithmic_mac32_per_op"] = MAC32[key]
            d["algorithmic_speedup"] = nn * MAC32[key] / t / 1e9 / peak
        d.update(more)
        return d

    kx = max(2, min(K, 3))
    if not args.no_extra:
        # ---- config 3 and 2: X448, comb (device-resident) --------------------------------------------------------------
        u = torch.from_numpy(stream_bytes("bench/x448/u%d" % rank, n * 56)).to(dev)
        kk = torch.from_numpy(stream_bytes("bench/x448/k%d" % rank, n * 56)).to(dev)
        xo = torch.empty(n * 56, dtype=torch.uint8, device=dev)
        xs = torch.empty(n, dtype=torch.int32, device=dev)
        h_sc = lib.scalar_decode_long(stream_bytes("bench/comb/s%d" % rank, n * 56).reshape(n, 56), 56)
        sc = torch.from_numpy(h_sc.reshape(-1)).to(dev)
        co = torch.empty(n * 256, dtype=torch.uint8, device=dev)
        extra["x448"] = entry(n, timed_dev(lambda: eng.x448(xo, xs, u, kk), kx), "x448")
        extra["comb"] = entry(n, timed_dev(lambda: eng.precomputed_scalarmul(co, sc), kx), "comb")
        # ---- config 1: field multiplication and the group law on 2^20 elements (device-resident; these sit at the HBM ridge) ----
        co2 = torch.empty_like(co)
        eng.point_double(co2, co)
        po = torch.empty_like(co)
        for name, fnc, key, nbytes in (("gf_mul", lambda: eng.gf_mul(xo, u, kk), "gf_mul", 168), ("point_add", lambda: eng.point_add(po, co, co2), "point_add", 768),
                                       ("point_double", lambda: eng.point_double(po, co), "point_double", 512)):
            t = timed_dev(fnc, 10)
            extra[name] = entry(n, t, key, hbm_gbs=n * nbytes / t / 1e9, hbm_frac=n * nbytes / t / 1e9 / hbm)
        del co2, po
        # ---- config 5 (per GPU): decaf encode / decode on the comb outputs (valid points), device-resident ----------------------
        enc = torch.empty(n * 56, dtype=torch.uint8, device=dev)
        dpts = torch.empty(n * 256, dtype=torch.uint8, device=dev)
        dstat = torch.empty(n, dtype=torch.int32, device=dev)
        for name, fnc, key, nbytes in (("decaf_encode", lambda: eng.point_encode(enc, co), "encode", 256 + 56),
                                       ("decaf_decode", lambda: eng.point_decode(dpts, dstat, enc, True), "decode", 56 + 256 + 4)):
            t = timed_dev(fnc, kx)
            extra[name] = entry(n, t, key, hbm_gbs=n * nbytes / t / 1e9, hbm_frac=n * nbytes / t / 1e9 / hbm)
        assert int((dstat == -1).sum().item()) == n, "decode(encode(P)) must succeed for every comb output"
        del enc, dpts, dstat, xo, xs, u, kk
        # ---- host-pointer entry points without a device-pointer twin: kernel time from the library's per-launch events, wall time beside it ----
        hh = stream_bytes("bench/h2c/%d" % rank, n * 112).reshape(n, 112)
        h56 = np.ascontiguousarray(hh[:, :56])
        hpts = lib.precomputed_scalarmul(h_sc)
        skk = stream_bytes("bench/sign/sk%d" % rank, n * 57).reshape(n, 57)
        pkk = lib.ed448_derive_public_key(skk)
        sarena = stream_bytes("bench/sign/msg%d" % rank, n * MSG_LEN)
        soff = np.arange(n + 1, dtype=np.uint64) * MSG_LEN
        for name, fnc, key in (("elligator_nonuniform", lambda: lib.from_hash_nonuniform(h56), "elligator"),
                               ("elligator_uniform", lambda: lib.from_hash_uniform(hh), "elligator_uniform"),
                               ("ed448_sign", lambda: lib.ed448_sign(skk, pkk, (sarena, soff)), "sign"),
                               ("ed448_derive_public_key", lambda: lib.ed448_derive_public_key(skk), "derive_public_key"),
                               ("point_scalarmul", lambda: lib.point_scalarmul(hpts, h_sc), "point_scalarmul"),
                               ("base_double_scalarmul_non_secret", lambda: lib.base_double_scalarmul_non_secret(h_sc, hpts, h_sc[::-1].copy()), "bdsm")):
            wall, kern, ks = timed_host(fnc, 2)
            extra[name] = entry(n, kern, key, e2e_value=world * n / wall, e2e_ms=wall * 1e3, kernel_ms=ks,
                                timing="value = batch / sum of this call's kernel times (CUDA events per launch); e2e_value = batch / wall time of the host-pointer call "
                                       "(pageable numpy buffers)")
        del hpts, hh, h56

    # ---- extra: the same batch size (a) with 2^20 DISTINCT keys (no table can be shared), (b) with message lengths
    #      uniform in [0, 256) under the 2^16 x 16 keys (SURVEY 8(d) C4, second run) --------------------------------------
    if not args.no_extra:
        for name, kw, key in (("verify_distinct_keys", {"per": 1}, "verify_distinct"), ("verify_varlen_msgs", {"varlen": True}, "verify_16_per_key"),
                              ("verify_64_per_key", {"per": 64}, "verify_64_per_key"), ("verify_one_signer", {"per": n}, "verify_one_signer")):
            sig1, pk1, arena1, off1, expect1 = cached_corpus(n, "bench/" + name, rank, world, barrier, **kw)
            t_sig, t_pk, t_msg, t_off = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (sig1.reshape(-1), pk1.reshape(-1), arena1, off1.view(np.int64)))
            eng.ed448_verify(d_st, t_sig, t_pk, t_msg, t_off, d_scratch)
            torch.cuda.synchronize()
            assert (d_st.cpu().numpy() == expect1).all(), "device verify (%s) disagrees with the expected accept bits" % name
            t = timed_dev(lambda: eng.ed448_verify(d_st, t_sig, t_pk, t_msg, t_off, d_scratch), kx)
            extra[name] = entry(n, t, key, unit=UNIT, algorithmic_mac32_per_op=MAC32["verify"], algorithmic_speedup=n * MAC32["verify"] / t / 1e9 / peak)
            del t_sig, t_pk, t_msg, t_off

    # ---- extra: the same corpus against a KEY SET (tables of the 2^16 keys built once, outside the timed region), host pointers ----
    if not args.no_extra and args.per_key == 16:
        nk = n // 16
        pk2d = np.ascontiguousarray(pk.reshape(n, 57))
        idx8 = np.flatnonzero(expect == 0)
        keys = pk2d[1::16].copy()                                  # entry 16j + 1 is never corrupted: the intact key of group j
        changed = idx8[(pk2d[idx8] != keys[idx8 // 16]).any(axis=1)]   # make_corpus kind 3: the key bytes of these entries were changed
        expect_ks = expect.copy(); expect_ks[changed] = -1         # under the key SET they verify against the intact key
        h_idx = pinned((np.arange(n, dtype=np.uint32) // 16).astype(np.uint32))
        fk = lib.lib.goldilocks_ed448_verify_keyset_batch
        fk.restype = C.c_int32
        # both table layouts (goldilocks_b200_keyset_policy): flat = a table per digit position, 369 KB per key, no doublings per signature
        # (the default for a set of 2^16 keys: 24 GB); compact = ten columns, 41 KB per key, forty doublings per signature
        for name, opkey, policy, what in (("verify_keyset_e2e", "verify_keyset", 32 << 30, "flat tables: 369 KB per key, additions only"),
                                          ("verify_keyset_compact_e2e", "verify_keyset_compact", 0, "compact tables: 41 KB per key")):
            lib.keyset_policy(policy)
            t_create = time.perf_counter()
            handle = lib.keyset_create(keys)
            t_create = time.perf_counter() - t_create
            lib.keyset_policy(32 << 30)
            argk = [C.c_void_p(h_st.data_ptr()), handle, C.c_void_p(h_idx.data_ptr()), C.c_void_p(h_sig.data_ptr()), C.c_void_p(h_msg.data_ptr()),
                    C.c_void_p(h_off.data_ptr()), C.c_uint8(0), None, C.c_uint8(0), C.c_size_t(n)]
            for _ in range(2):
                assert fk(*argk) == -1
            assert (h_st.numpy() == expect_ks).all(), "key-set verify (%s) disagrees with the expected accept bits" % name
            barrier()
            t0 = time.perf_counter()
            for _ in range(kx):
                assert fk(*argk) == -1
            torch.cuda.synchronize()
            t = max_over_ranks((time.perf_counter() - t0) / kx)
            barrier()
            lib.keyset_destroy(handle)
            extra[name] = entry(n, t, opkey, unit=UNIT, keys_in_set=int(nk), layout=what, keyset_create_ms=t_create * 1e3,
                                api="goldilocks_ed448_verify_keyset_batch (host pointers, pinned; tables of the key set built once, not timed)")

    # ---- extra: random-linear-combination batch verification (SURVEY 8(f)3), host pointers: all-valid corpus of the bench shape, and a
    #      sweep of corruption rates -- a bad signature sends only its chunk to the per-signature path -----------------------------------
    if not args.no_extra and lib.has("goldilocks_ed448_verify_rlc_batch"):
        sig2, pk2, arena2, off2, _ = cached_corpus(n, "bench/rlc", rank, world, barrier, per=args.per_key, corrupt=False)
        r_sig, r_pk, r_msg, r_off = pinned(sig2.reshape(-1)), pinned(pk2.reshape(-1)), pinned(arena2), pinned(off2.view(np.int64))
        fr = lib.lib.goldilocks_ed448_verify_rlc_batch
        fr.restype = C.c_int32
        fast = C.c_int(0)
        argr = [C.c_void_p(h_st.data_ptr()), C.c_void_p(r_sig.data_ptr()), C.c_void_p(r_pk.data_ptr()), C.c_void_p(r_msg.data_ptr()),
                C.c_void_p(r_off.data_ptr()), C.c_uint8(0), None, C.c_uint8(0), C.c_size_t(n), C.byref(fast)]
        lib.rlc_policy(16)
        for _ in range(2):
            assert fr(*argr) == -1
        assert (h_st.numpy() == -1).all() and fast.value == 1, "the batch equation must decide an all-valid batch"
        barrier()
        prof.start()
        t0 = time.perf_counter()
        for _ in range(kx):
            assert fr(*argr) == -1
        torch.cuda.synchronize()
        t = max_over_ranks((time.perf_counter() - t0) / kx)
        krlc = prof.stop(per=kx)
        barrier()
        extra["verify_rlc_all_valid_e2e"] = {"value": world * n / t, "unit": UNIT, "ms_per_step": t * 1e3, "batch_per_gpu": n, "fast_path": 1, "kernel_ms": krlc,
                                             "api": "goldilocks_ed448_verify_rlc_batch (host pointers, pinned): one multi-scalar multiplication per chunk with secret "
                                                    "weights decides it; per-signature fallback for the chunks whose equation fails; corpus = the bench shape with NO corrupted entries"}
        # corruption sweep: flip one S bit in every `1/rate`-th signature (spread evenly), time the call, check the statuses
        sweep = {"note": "per rate: one untimed call, then two timed ones (steady state: after a call in which most chunks failed the library "
                         "skips the equation for the next calls, goldilocks_b200_rlc_policy); fast_path 1 = whole-batch equation, 2 = per-chunk "
                         "equations + the failing chunks re-verified, 0 = per-signature path over everything"}
        clean = sig2.copy()
        for label, every in (("0", 0), ("1_bad", n), ("2^-14", 1 << 14), ("2^-10", 1 << 10), ("2^-6", 1 << 6), ("1/8", 8)):
            cur = clean.copy()
            bad = np.arange(every // 2, n, every) if every else np.zeros(0, np.int64)
            cur[bad, 70] ^= 1
            r_sig.copy_(torch.from_numpy(cur.reshape(-1)))
            want = np.full(n, -1, np.int32); want[bad] = 0
            assert fr(*argr) == -1
            assert (h_st.numpy() == want).all(), "rlc sweep %s: statuses" % label
            t0 = time.perf_counter()
            for _ in range(2):
                assert fr(*argr) == -1
            tt = max_over_ranks((time.perf_counter() - t0) / 2)
            sweep[label] = {"bad_signatures": int(len(bad)), "ms": tt * 1e3, "value": world * n / tt, "fast_path": int(fast.value)}
            barrier()
        r_sig.copy_(torch.from_numpy(cur.reshape(-1)))                    # ordinary path on the 1/8-corrupted copy, same buffers
        argo = [C.c_void_p(h_st.data_ptr()), C.c_void_p(r_sig.data_ptr()), C.c_void_p(r_pk.data_ptr()), C.c_void_p(r_msg.data_ptr()),
                C.c_void_p(r_off.data_ptr()), C.c_uint8(0), None, C.c_uint8(0), C.c_size_t(n)]
        assert fn(*argo) == -1
        t0 = time.perf_counter()
        for _ in range(2):
            assert fn(*argo) == -1
        tt = max_over_ranks((time.perf_counter() - t0) / 2)
        sweep["ordinary_path_same_buffers"] = {"ms": tt * 1e3, "value": world * n / tt}
        extra["rlc_sweep"] = sweep
        del r_sig, r_pk, r_msg, r_off
        # the same entry point on 2^20 DISTINCT keys (no key repeats: the key class is as big as the R class): all valid, one bad, 1/8 bad
        sig3, pk3, arena3, off3, _ = cached_corpus(n, "bench/rlc_distinct", rank, world, barrier, per=1, corrupt=False)
        q_sig, q_pk, q_msg, q_off = pinned(sig3.reshape(-1)), pinned(pk3.reshape(-1)), pinned(arena3), pinned(off3.view(np.int64))
        argq = [C.c_void_p(h_st.data_ptr()), C.c_void_p(q_sig.data_ptr()), C.c_void_p(q_pk.data_ptr()), C.c_void_p(q_msg.data_ptr()),
                C.c_void_p(q_off.data_ptr()), C.c_uint8(0), None, C.c_uint8(0), C.c_size_t(n), C.byref(fast)]
        lib.rlc_policy(16)
        sweep_d = {}
        for label, every in (("0", 0), ("1_bad", n), ("1/8", 8)):
            cur = sig3.copy()
            bad = np.arange(every // 2, n, every) if every else np.zeros(0, np.int64)
            cur[bad, 70] ^= 1
            q_sig.copy_(torch.from_numpy(cur.reshape(-1)))
            want = np.full(n, -1, np.int32); want[bad] = 0
            assert fr(*argq) == -1
            assert (h_st.numpy() == want).all(), "rlc sweep (distinct keys) %s: statuses" % label
            t0 = time.perf_counter()
            for _ in range(2):
                assert fr(*argq) == -1
            tt = max_over_ranks((time.perf_counter() - t0) / 2)
            sweep_d[label] = {"bad_signatures": int(len(bad)), "ms": tt * 1e3, "value": world * n / tt, "fast_path": int(fast.value)}
            barrier()
        argo = [C.c_void_p(h_st.data_ptr()), C.c_void_p(q_sig.data_ptr()), C.c_void_p(q_pk.data_ptr()), C.c_void_p(q_msg.data_ptr()),
                C.c_void_p(q_off.data_ptr()), C.c_uint8(0), None, C.c_uint8(0), C.c_size_t(n)]
        assert fn(*argo) == -1
        t0 = time.perf_counter()
        assert fn(*argo) == -1
        tt = max_over_ranks(time.perf_counter() - t0)
        sweep_d["ordinary_path_same_buffers"] = {"ms": tt * 1e3, "value": world * n / tt}
        extra["rlc_sweep_distinct_keys"] = sweep_d
        lib.rlc_policy(16)
        del q_sig, q_pk, q_msg, q_off

    # ---- extra.two_batches_in_flight: the same step with TWO batches in flight -- the device-pointer entry point on two streams with two scratch
    # areas, and the host-pointer entry point from two host threads (the library deals them two of its three contexts per device) ----------
    if not args.no_extra:
        s_a, s_b = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        d_st2, d_scratch2 = torch.empty_like(d_st), torch.empty_like(d_scratch)
        lanes2 = ((d_st, d_scratch, s_a), (d_st2, d_scratch2, s_b))

        def step2(i):
            st, scr, strm = lanes2[i & 1]
            with torch.cuda.stream(strm):
                eng.ed448_verify(st, d_sig, d_pk, d_msg, d_off, scr)

        d_st.zero_(); d_st2.zero_()
        torch.cuda.synchronize()
        for i in range(4):
            step2(i)
        torch.cuda.synchronize()
        assert (d_st.cpu().numpy() == expect).all() and (d_st2.cpu().numpy() == expect).all(), "two batches in flight: statuses"
        k2 = 2 * max(2, K // 2)
        a2, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        cur = torch.cuda.current_stream()
        a2.record()
        s_a.wait_stream(cur); s_b.wait_stream(cur)
        for i in range(k2):
            step2(i)
        cur.wait_stream(s_a); cur.wait_stream(s_b)
        b2.record()
        barrier()
        t2 = max_over_ranks(a2.elapsed_time(b2) / 1e3 / k2)
        h_st2 = torch.empty(n, dtype=torch.int32).pin_memory()
        argv2 = list(argv); argv2[0] = C.c_void_p(h_st2.data_ptr())
        ke2 = max(2, min(K, 5))
        h_st.zero_(); h_st2.zero_()

        gate = threading.Barrier(3)
        thread_errors = []
        dev_index = torch.cuda.current_device()

        def caller(av):
            try:
                torch.cuda.set_device(dev_index)    # a new host thread starts on device 0: bind it to this rank's GPU before its first call
                assert fn(*av) == -1                # first call of this thread: its context of the device allocates its arena
                assert fn(*av) == -1
                gate.wait(timeout=300)
                gate.wait(timeout=300)              # the main thread has taken the start time
                for _ in range(ke2):
                    assert fn(*av) == -1
            except BaseException as e:  # noqa: BLE001 -- never leave the main thread waiting at the gate
                thread_errors.append(repr(e))
                gate.abort()

        th2 = [threading.Thread(target=caller, args=(av,)) for av in (argv, argv2)]
        barrier()
        t2e = float("inf")
        if world == 1:      # the host-thread half is measured on one GPU only (each thread holds an 11 GB arena of its own: kept out of the scaling runs)
            for x in th2:
                x.start()
            t0 = time.perf_counter()
            try:
                gate.wait(timeout=300)
                t0 = time.perf_counter()
                gate.wait(timeout=300)
            except threading.BrokenBarrierError:
                thread_errors.append("a caller thread failed before the timed region")
            for x in th2:
                x.join()
            torch.cuda.synchronize()
            t_end = time.perf_counter()
            ok2 = not thread_errors and bool((h_st.numpy() == expect).all()) and bool((h_st2.numpy() == expect).all())
            if ok2:
                t2e = (t_end - t0) / (2 * ke2)
            else:
                sys.stderr.write("[bench] two host threads: %s\n" % (thread_errors[:1] or ["statuses differ"]))
        barrier()
        extra["two_batches_in_flight"] = {
            "value": world * n / t2, "unit": UNIT, "ms_per_step": t2 * 1e3, "steps": k2, "step_frac_executed": executed_step / t2 / 1e9 / peak,
            "api": "goldilocks_ed448_verify_batch_dev on two streams, each with its own scratch and status array (same inputs)",
            "e2e": ({"skipped": "measured at N = 1 only" if world > 1 else "failed, see stderr"} if t2e == float("inf") else
                    {"value": world * n / t2e, "unit": UNIT, "ms_per_step": t2e * 1e3, "calls": 2 * ke2,
                     "api": "goldilocks_ed448_verify_batch (host pointers, pinned) from two host threads, each on its own status array"}),
            "note": "the headline `value` and `e2e` run one batch at a time; with a second batch in flight the latency-bound phases of one (key grouping, decodes, "
                    "the doubling chain of the key tables, copies) run beside the finish kernel of the other"}
        del d_st2, d_scratch2

    # ---- extra.single_calls_from_threads: the reference's own one-signature call from a pool of host threads, gathered or not -------
    if not args.no_extra:
        barrier()
        if rank == 0:
            extra["single_calls_from_threads"] = single_call_leg(lib, sig, pk, arena, off, expect)
        barrier()

    # ---- extra.strong: ONE batch sharded over all N GPUs by the library itself (rank 0 drives, the other ranks wait) ------------------
    if not args.no_extra and not args.no_strong:
        barrier()
        if rank == 0:
            extra["strong"] = strong_leg(lib, torch, world, n, (h_st, h_sig, h_pk, h_msg, h_off, expect), peak, ops, kx)
        barrier()

    # ---- the reference re-verifies the WHOLE corpus once (rank 0, outside every timed region) and must agree bit for bit ----------------
    ref_check = None
    if rank == 0 and not args.no_cpu:
        ref, kind = reference_signer()
        t0 = time.time()
        st_ref = ref.ed448_verify(sig, pk, (arena, off))
        assert (st_ref == expect).all(), "the reference disagrees with the corpus' expected accept bits"
        assert (st_ref == dev_status).all(), "the reference disagrees with the statuses of the timed device-resident path"
        ref_check = {"signatures": int(n), "seconds": round(time.time() - t0, 1), "kind": kind, "agrees_with_device_statuses": True}
    # ---- CPU baseline (rank 0, N = 1 only) ---------------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cores = host_cores()
        n_cpu = min(n, 4096 * cores)       # ~0.6 s per pass on all cores, 1 warm-up + 2 timed = ~25 core-seconds
        cpu, _ = cpu_reference_rate(n_cpu, 2, 1, corpus=(sig, pk, arena, off, expect))
    if rank == 0:
        extra["reference_check_of_the_full_corpus"] = ref_check
        line = {"metric": METRIC, "value": world * n / t_step, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": t_step * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
                "config": config_dict(world, args.per_key, n), "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
                "cpu_baseline": cpu, "extra": extra}
        emit(line)
    barrier()
    if world > 1:
        dist.destroy_process_group()


def single_call_leg(lib, sig, pk, arena, off, expect):
    """goldilocks_ed448_verify (the reference's one-signature entry point, ed448.h:157-165) called from host threads on signatures of
    the bench corpus: every thread makes its calls one after the other.  Without gathering each call is a batch of one on the GPU;
    with goldilocks_b200_coalesce(window) concurrent calls share a launch (csrc/coalesce.h).  Python threads: ctypes drops the GIL
    for the duration of a call."""
    import threading
    try:
        import torch
        dev_index = torch.cuda.current_device()
    except Exception:  # noqa: BLE001
        torch, dev_index = None, None
    fn = lib.lib.goldilocks_ed448_verify
    fn.restype = C.c_int32
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint8, C.c_void_p, C.c_uint8]
    sp, pp, ap = sig.ctypes.data, pk.ctypes.data, arena.ctypes.data
    o = off.astype(np.int64)

    def run(T, K, window_us):
        lib.coalesce(window_us)
        wrong = []
        c0, b0, _ = lib.coalesce_stats()

        def worker(t):
            if dev_index is not None:
                torch.cuda.set_device(dev_index)    # new host threads start on device 0
            for j in range(K):
                i = t * K + j
                st = fn(sp + 114 * i, pp + 57 * i, ap + int(o[i]), int(o[i + 1] - o[i]), 0, None, 0)
                if st != expect[i]:
                    wrong.append(i)

        th = [threading.Thread(target=worker, args=(t,)) for t in range(T)]
        t0 = time.perf_counter()
        for x in th:
            x.start()
        for x in th:
            x.join()
        dt = time.perf_counter() - t0
        lib.coalesce(0)
        assert not wrong, "single calls: %d statuses differ from the corpus' expected accept bits" % len(wrong)
        c1, b1, big = lib.coalesce_stats()
        return {"threads": T, "calls": T * K, "window_us": window_us, "value": T * K / dt, "unit": UNIT, "seconds": dt,
                "batches": int(b1 - b0), "largest_batch": int(big) if window_us else 1}

    run(8, 2, 0)                                    # warm-up of the one-element shapes
    out = {"alone": run(8, 16, 0), "gathered": run(256, 24, 250), "gathered_64_threads": run(64, 48, 250)}
    out["speedup_gathered_over_alone"] = out["gathered"]["value"] / out["alone"]["value"]
    exe = os.path.join(ROOT, "tools", "single_calls")          # the same experiment from native threads (no interpreter in the loop)
    if os.path.exists(exe):
        try:
            p = subprocess.run([exe, "1024", "16", "250"], capture_output=True, text=True, timeout=300)
            out["native_threads"] = json.loads(p.stdout) if p.returncode == 0 else {"failed": p.stderr[-300:]}
        except Exception as e:  # noqa: BLE001
            out["native_threads"] = {"failed": type(e).__name__}
    return out


def strong_leg(lib, torch, world, n, corpus, peak, ops, reps):
    """rank 0: goldilocks_b200_set_devices(all N GPUs of the box), then ONE host-pointer call per workload.  The same code path
    at N = 1 (a set of one device) is the baseline of the strong-scaling curve."""
    from util import stream_bytes
    h_st, h_sig, h_pk, h_msg, h_off, expect = corpus
    out = {"devices": list(range(world)), "api": "goldilocks_b200_set_devices + the ordinary *_batch host-pointer calls (pinned buffers); no collective, no peer traffic"}
    lib.set_devices(list(range(world)))
    try:
        L = lib.lib

        def call(name, *args):
            f = getattr(L, name)
            f.restype = C.c_int32
            assert f(*args) == -1, name

        def timed(fnc, k):
            fnc()
            t0 = time.perf_counter()
            for _ in range(k):
                fnc()
            return (time.perf_counter() - t0) / k

        P = lambda t: C.c_void_p(t.data_ptr())   # noqa: E731
        # -- configs[3]: one 2^20 verify batch
        argv = [P(h_st), P(h_sig), P(h_pk), P(h_msg), P(h_off), C.c_uint8(0), None, C.c_uint8(0), C.c_size_t(n)]
        t = timed(lambda: call("goldilocks_ed448_verify_batch", *argv), reps)
        assert (h_st.numpy() == expect).all(), "sharded verify disagrees with the expected accept bits"
        out["verify_2^20"] = {"value": n / t, "unit": UNIT, "ms": t * 1e3, "batch": n, "imad_frac_executed_per_gpu": n * ops["verify_16_per_key"] / t / 1e9 / peak / world}
        # -- configs[2]: one 2^20 X448 batch
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()   # noqa: E731
        u, k = pin(stream_bytes("bench/strong/u", n * 56)), pin(stream_bytes("bench/strong/k", n * 56))
        xo, xs = torch.empty(n * 56, dtype=torch.uint8).pin_memory(), torch.empty(n, dtype=torch.int32).pin_memory()
        t = timed(lambda: call("goldilocks_x448_batch", P(xo), P(xs), P(u), P(k), C.c_size_t(n)), reps)
        assert int((xs == -1).sum()) == n
        out["x448_2^20"] = {"value": n / t, "unit": "ops/s", "ms": t * 1e3, "batch": n, "imad_frac_executed_per_gpu": n * ops["x448"] / t / 1e9 / peak / world}
        del u, k, xo, xs
        # -- configs[4]: 2^24 elements: Elligator hash-to-curve -> decaf encode -> decaf decode (pipelined in chunks over three contexts per device)
        m = 1 << 24
        hs = pin(stream_bytes("bench/strong/h", m * 56))
        pts = torch.empty(m * 256, dtype=torch.uint8).pin_memory()
        ser = torch.empty(m * 56, dtype=torch.uint8).pin_memory()
        dst = torch.empty(m, dtype=torch.int32).pin_memory()
        legs = (("elligator_2^24", lambda: call("goldilocks_448_point_from_hash_nonuniform_batch", P(pts), P(hs), C.c_size_t(m)), "elligator", 56, 256),
                ("decaf_encode_2^24", lambda: call("goldilocks_448_point_encode_batch", P(ser), P(pts), C.c_size_t(m)), "encode", 256, 56),
                ("decaf_decode_2^24", lambda: call("goldilocks_448_point_decode_batch", P(pts), P(dst), P(ser), C.c_uint64(0), C.c_size_t(m)), "decode", 56, 260))
        total = 0.0
        for name, fnc, key, bin_, bout in legs:
            t = timed(fnc, 2)
            total += t
            out[name] = {"value": m / t, "unit": "ops/s", "ms": t * 1e3, "batch": m, "imad_frac_executed_per_gpu": m * ops[key] / t / 1e9 / peak / world,
                         "h2d_gbs": m * bin_ / t / 1e9, "d2h_gbs": m * bout / t / 1e9}
        assert int((dst == -1).sum()) == m, "decode(encode(elligator(h))) must succeed for every element"
        out["config4_2^24_total"] = {"value": m / total, "unit": "elements/s through hash-to-curve + encode + decode", "ms": total * 1e3, "batch": m}
    finally:
        lib.set_devices([])
    return out


def dump_output(out_dir, name, a):
    """<out_dir>/<name>.npy in float32 (statuses -1 / 0 are exact), at most DUMP_BYTES: a larger array keeps a sample
    at sorted indices drawn with a fixed seed, the same for every build"""
    os.makedirs(out_dir, exist_ok=True)
    a = np.asarray(a).reshape(-1)
    keep = DUMP_BYTES // 4 - 64
    if a.size > keep:
        a = a[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
    np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def emit(line):
    """the ONE JSON line on the real stdout (library banners are kept off it)"""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)          # anything a library prints to fd 1 from here on goes to stderr
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=N_PER_GPU, help="signatures per GPU per step (default 2^20, the BASELINE size)")
    ap.add_argument("--per-key", type=int, default=16, help="signatures per public key in the corpus (SURVEY 8(d) C4: 16); other values are for the "
                    "sensitivity table in DESIGN.md, not the headline")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-peak", action="store_true", help="skip the on-box IMAD.WIDE peak measurement (use the committed figure)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps write the statuses of the last one (rank 0's batch) "
                    "as DIR/verify_status.npy, float32, for comparing two builds on the same inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
