// tests/hostsim/peerset.cpp -- TEST INFRASTRUCTURE ONLY (never shipped, never loaded by the product).
//
// The X448 peer-set entry points of include/goldilocks_b200.h (goldilocks_b200_x448_peerset_*, goldilocks_x448_peerset_batch)
// on the host, in the manner of hostsim.cpp: the device functors LaneX448PeerLift, LanePrecompute, LaneNielsFromAbi and
// SlotX448Peer compiled with the host compiler and run in plain loops over host memory, so the CPU tier checks the CUDA
// source of peer sets against the checker.  Built as its own library (tests/hostsim/_hostsim_peerset.so).
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

struct hostsim_peerset { size_t m; std::vector<uint8_t> peers; std::vector<int32_t> table_ok; std::vector<niels> tables; };
EXPORT int32_t goldilocks_b200_x448_peerset_create(hostsim_peerset **out, const uint8_t *peers, size_t m) {
    hostsim_peerset *ps = new hostsim_peerset{m, std::vector<uint8_t>(peers, peers + 56 * m), std::vector<int32_t>(m + 1), std::vector<niels>((m + 1) * COMB_ENTRIES)};
    std::vector<abi_pt> pts(m + 1);
    LaneX448PeerLift fl = {pts.data(), ps->table_ok.data(), ps->peers.data()};
    run(fl, m);
    std::vector<abi_niels> up((m + 1) * COMB_ENTRIES);
    std::vector<niels> scratch(16 * COMB_N * m + 1);
    LanePrecompute fp = {up.data(), pts.data(), scratch.data()};
    run(fp, COMB_N * m);
    LaneNielsFromAbi fc = {ps->tables.data(), up.data()};
    run(fc, COMB_ENTRIES * m);
    *out = ps;
    return -1;
}
EXPORT void goldilocks_b200_x448_peerset_destroy(hostsim_peerset *ps) { delete ps; }
EXPORT size_t goldilocks_b200_x448_peerset_size(const hostsim_peerset *ps) { return ps ? ps->m : 0; }
EXPORT int32_t goldilocks_x448_peerset_batch(uint8_t *o, int32_t *st, const hostsim_peerset *ps, const uint32_t *peer_index, const uint8_t *sc, size_t n) {
    SlotX448Peer f = {o, st, ps->tables.data(), ps->table_ok.data(), ps->peers.data(), peer_index, sc, (uint32_t)ps->m};
    run_sm(f, n);
    return -1;
}
// test hook: the per-peer path flags of a set (-1 = comb table, 0 = ladder)
EXPORT void hostsim_x448_peerset_flags(int32_t *out, const hostsim_peerset *ps) { memcpy(out, ps->table_ok.data(), sizeof(int32_t) * ps->m); }
