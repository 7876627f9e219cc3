// tests/hostsim/decaf_peerset.cpp -- TEST INFRASTRUCTURE ONLY (never shipped, never loaded by the product).
//
// The decaf peer-set entry points of include/goldilocks_b200.h (goldilocks_b200_decaf_peerset_*,
// goldilocks_448_direct_scalarmul_peerset_batch) on the host, in the manner of hostsim.cpp and peerset.cpp: the device functors
// LaneDecafPeerDecode, LanePrecompute, LaneNielsFromAbi, LaneDecafPeerKeys and SlotDecafPeer compiled with the host compiler and
// run in plain loops over host memory, so the CPU tier checks the CUDA source of decaf peer sets against the checker.  Built as
// its own library (tests/hostsim/_hostsim_decaf_peerset.so).
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <thread>
#include <vector>

#include "../../libgoldilocks_b200/csrc/slot_lanes.cuh"

#define EXPORT extern "C" __attribute__((visibility("default")))

static int g_threads = 1;
EXPORT void hostsim_set_threads(int t) { g_threads = t < 1 ? 1 : t; }

template <class Work>
static void split(size_t n, const Work &work) { /* [0, n) in g_threads contiguous ranges */
    int nt = g_threads;
    if ((size_t)nt > n) nt = n ? (int)n : 1;
    if (nt <= 1) { work(0, n); return; }
    std::vector<std::thread> th;
    for (int t = 0; t < nt; t++) th.emplace_back([&work, n, nt, t]() { work(n * t / nt, n * (t + 1) / nt); });
    for (auto &x : th) x.join();
}
template <class F>
static void run(const F &f, size_t n) {
    split(n, [&f](size_t lo, size_t hi) { for (size_t i = lo; i < hi; i++) f(i); });
}
template <class F>
static void run_sm(const F &f, size_t n) { /* slot machine: F::NSLOTS field elements of scratch per worker */
    split(n, [&f](size_t lo, size_t hi) {
        std::vector<gf> slots(F::NSLOTS);
        sref base = {slots.data()};
        for (size_t i = lo; i < hi; i++) f(i, base, true);
    });
}

static fixed_tables *tables() {
    static fixed_tables *ft = nullptr;
    if (!ft) {
        ft = new fixed_tables;
        for (int lane = 0; lane < TABLE_LANES; lane++) build_tables_lane(ft, lane);
    }
    return ft;
}
struct hostsim_decaf_peerset { size_t m; std::vector<int32_t> peer_ok; std::vector<niels> tables; };
EXPORT int32_t goldilocks_b200_decaf_peerset_create(hostsim_decaf_peerset **out, const uint8_t *peers, uint64_t allow_identity, size_t m) {
    const size_t mm = m + 1;
    hostsim_decaf_peerset *ps = new hostsim_decaf_peerset{m, std::vector<int32_t>(mm), std::vector<niels>(mm * COMB_ENTRIES)};
    std::vector<abi_pt> pts(mm);
    LaneDecafPeerDecode fd = {pts.data(), ps->peer_ok.data(), peers, tables(), (uint32_t)m, allow_identity ? 1u : 0u};
    run(fd, mm);
    std::vector<abi_niels> up(mm * COMB_ENTRIES);
    std::vector<niels> scratch(16 * COMB_N * mm);
    LanePrecompute fp = {up.data(), pts.data(), scratch.data()};
    run(fp, COMB_N * mm);
    LaneNielsFromAbi fc = {ps->tables.data(), up.data()};
    run(fc, COMB_ENTRIES * mm);
    *out = ps;
    return -1;
}
EXPORT void goldilocks_b200_decaf_peerset_destroy(hostsim_decaf_peerset *ps) { delete ps; }
EXPORT size_t goldilocks_b200_decaf_peerset_size(const hostsim_decaf_peerset *ps) { return ps ? ps->m : 0; }
// The device sorts (min(peer_index[j], m), j) with a stable radix sort; std::stable_sort gives the same order,
// so SlotDecafPeer runs here over the same permuted indices as on the GPU.
EXPORT int32_t goldilocks_448_direct_scalarmul_peerset_batch(uint8_t *scaled, int32_t *st, const hostsim_decaf_peerset *ps, const uint32_t *peer_index,
                                                            const abi_sc *sc, uint64_t short_circuit, size_t n) {
    std::vector<uint32_t> keys(n), vals(n);
    LaneDecafPeerKeys fk = {keys.data(), vals.data(), peer_index, (uint32_t)ps->m};
    run(fk, n);
    std::stable_sort(vals.begin(), vals.end(), [&keys](uint32_t a, uint32_t b) { return keys[a] < keys[b]; });
    SlotDecafPeer f = {scaled, st, ps->tables.data(), ps->peer_ok.data(), peer_index, vals.data(), sc, (uint32_t)ps->m, short_circuit ? ~0u : 0u};
    run_sm(f, n);
    return -1;
}
// test hook: the per-peer decode statuses of a set, m + 1 of them (the last one stands for indices >= m)
EXPORT void hostsim_decaf_peerset_flags(int32_t *out, const hostsim_decaf_peerset *ps) { memcpy(out, ps->peer_ok.data(), sizeof(int32_t) * (ps->m + 1)); }
