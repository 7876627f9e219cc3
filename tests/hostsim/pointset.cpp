// tests/hostsim/pointset.cpp -- TEST INFRASTRUCTURE ONLY (never shipped, never loaded by the product).
//
// The point-set entry points of include/goldilocks_b200.h (goldilocks_b200_pointset_*,
// goldilocks_448_base_double_scalarmul_non_secret_pointset_batch) on the host, in the manner of hostsim.cpp and decaf_peerset.cpp:
// the device functors SlotKeysetChain, SlotKeysetColumns, SlotKeysetTables, LaneKeysetNormalize, LaneDecafPeerKeys and
// SlotPointset compiled with the host compiler and run in plain loops over host memory, so the CPU tier checks the CUDA source of
// point sets.  goldilocks_b200_keyset_policy picks the layout here as in the library.  Built as its own library
// (tests/hostsim/_hostsim_pointset.so).
#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

#include "../../libgoldilocks_b200/csrc/slot_lanes.cuh"

#define EXPORT extern "C" __attribute__((visibility("default")))

static int g_threads = 1;
EXPORT void hostsim_set_threads(int t) { g_threads = t < 1 ? 1 : t; }

template <class Work>
static void split(size_t n, const Work &work) { /* [0, n) in g_threads contiguous ranges; work(lo, hi, worker) */
    int nt = g_threads;
    if ((size_t)nt > n) nt = n ? (int)n : 1;
    if (nt <= 1) { work(0, n, 0); return; }
    std::vector<std::thread> th;
    for (int t = 0; t < nt; t++) th.emplace_back([&work, n, nt, t]() { work(n * t / nt, n * (t + 1) / nt, (size_t)t); });
    for (auto &x : th) x.join();
}
template <class F>
static void run(const F &f, size_t n) {
    split(n, [&f](size_t lo, size_t hi, size_t) { for (size_t i = lo; i < hi; i++) f(i); });
}
template <class F>
static void run_smp(const F &f, size_t n) { /* persistent slot machine: F::NSLOTS field elements of scratch per worker */
    split(n, [&f](size_t lo, size_t hi, size_t slot) {
        std::vector<gf> slots(F::NSLOTS);
        sref base = {slots.data()};
        for (size_t i = lo; i < hi; i++) f(i, base, slot);
    });
}

static std::vector<uint4> g_slots;
static uint4 *slots(size_t tables_per_thread) { /* window tables (wtab): workers rounded up to whole warps of 32 */
    g_slots.resize((size_t)((g_threads + 31) / 32 * 32) * tables_per_thread * WTAB_QUADS_PER_LANE);
    return g_slots.data();
}
static fixed_tables *tables() {
    static fixed_tables *ft = nullptr;
    if (!ft) {
        ft = (fixed_tables *)aligned_alloc(64, sizeof(fixed_tables));
        for (int lane = 0; lane < TABLE_LANES; lane++) build_tables_lane(ft, lane);
    }
    return ft;
}
static niels *wide_table() {
    static niels *w = nullptr;
    if (!w) {
        w = (niels *)aligned_alloc(64, sizeof(niels) * WIDE_ENTRIES * WIDE_TABLES);
        std::vector<pniels> tmp(WIDE_ENTRIES * WIDE_TABLES);
        std::vector<gf> pre(WIDE_ENTRIES * WIDE_TABLES);
        LaneBuildWide fw = {w, tmp.data(), pre.data(), tables()};   /* 3.3 M entries: every core, whatever hostsim_set_threads says */
        const int keep = g_threads;
        g_threads = (int)std::max(1u, std::thread::hardware_concurrency());
        run(fw, (size_t)WIDE_LANES * WIDE_TABLES);
        g_threads = keep;
    }
    return w;
}

static unsigned long long g_keyset_flat_bytes = 32ull << 30;
EXPORT void goldilocks_b200_keyset_policy(unsigned long long max_table_bytes) { g_keyset_flat_bytes = max_table_bytes; }
struct hostsim_pointset { size_t m; std::vector<uint4> ktabs; bool flat; };
EXPORT int32_t goldilocks_b200_pointset_create(hostsim_pointset **out, const abi_pt *points, size_t m) {
    const size_t mm = m + 1;   /* table m: the identity's, for every index >= m */
    const bool flat = (unsigned long long)mm * KSET_QUADS * sizeof(uint4) <= g_keyset_flat_bytes;
    hostsim_pointset *ps = new hostsim_pointset{m, std::vector<uint4>(mm * (size_t)(flat ? KSET_QUADS : KTAB_QUADS)), flat};
    std::vector<abi_pt> pts(mm);
    if (m) memcpy(pts.data(), points, sizeof(abi_pt) * m);
    memset(&pts[m], 0, sizeof(abi_pt));
    pts[m].y.limb[0] = pts[m].z.limb[0] = 1;
    if (flat) {
        SlotKeysetChain fc = {pts.data(), ps->ktabs.data()};
        run_smp(fc, mm);
        SlotKeysetColumns fcol = {ps->ktabs.data(), slots(1)};
        run_smp(fcol, mm * KSET_COLS);
    } else {
        SlotKeysetTables ft = {pts.data(), ps->ktabs.data()};
        run_smp(ft, mm);
    }
    LaneKeysetNormalize fn = {ps->ktabs.data(), flat ? (uint32_t)KSET_COLS : (uint32_t)VSH_CHUNKS, flat ? (uint32_t)KSET_QUADS : (uint32_t)KTAB_QUADS};
    run(fn, mm * (flat ? KSET_COLS : VSH_CHUNKS));
    *out = ps;
    return -1;
}
EXPORT void goldilocks_b200_pointset_destroy(hostsim_pointset *ps) { delete ps; }
EXPORT size_t goldilocks_b200_pointset_size(const hostsim_pointset *ps) { return ps ? ps->m : 0; }
// The device sorts (min(point_index[j], m), j) with a stable radix sort; std::stable_sort gives the same order,
// so SlotPointset runs here over the same permuted indices as on the GPU.
EXPORT int32_t goldilocks_448_base_double_scalarmul_non_secret_pointset_batch(abi_pt *out, const hostsim_pointset *ps, const uint32_t *point_index,
                                                                              const abi_sc *s1, const abi_sc *s2, size_t n) {
    std::vector<uint32_t> keys(n), vals(n);
    LaneDecafPeerKeys fk = {keys.data(), vals.data(), point_index, (uint32_t)ps->m};
    run(fk, n);
    std::stable_sort(vals.begin(), vals.end(), [&keys](uint32_t a, uint32_t b) { return keys[a] < keys[b]; });
    if (ps->flat) {
        SlotPointset<true> f = {out, s1, s2, wide_table(), ps->ktabs.data(), point_index, vals.data(), (uint32_t)ps->m};
        run_smp(f, n);
    } else {
        SlotPointset<false> f = {out, s1, s2, wide_table(), ps->ktabs.data(), point_index, vals.data(), (uint32_t)ps->m};
        run_smp(f, n);
    }
    return -1;
}
// test hook: 1 when the set has the flat layout
EXPORT int hostsim_pointset_flat(const hostsim_pointset *ps) { return ps->flat ? 1 : 0; }
