// tests/hostsim/peerset_lookup.cpp -- TEST INFRASTRUCTURE ONLY (never shipped, never loaded by the product).
//
// goldilocks_x448_peerset_lookup_batch (include/goldilocks_b200.h) on the host, in the manner of hostsim.cpp: the device functors
// LaneX448PeerLookup, LaneDecafPeerKeys and SlotX448PeerLookup compiled with the host compiler and run in plain loops over host
// memory, so the CPU tier checks the CUDA source of the lookup call.  It builds on peerset.cpp (its peer sets, loops and index
// form) and exports everything that library exports plus the lookup call.  Built as its own library
// (tests/hostsim/_hostsim_peerset_lookup.so).
#include <algorithm>

#include "peerset.cpp"

// The set's indices in peer-byte order, ties by index: what goldilocks_b200_x448_peerset_create keeps on the device (abi.cu sorts
// them with the same std::stable_sort); peerset.cpp's sets do not keep it, so it is made here, per call.
static std::vector<uint32_t> peerset_sorted(const hostsim_peerset *ps) {
    std::vector<uint32_t> sorted(ps->m);
    for (size_t i = 0; i < ps->m; i++) sorted[i] = (uint32_t)i;
    const uint8_t *u = ps->peers.data();
    std::stable_sort(sorted.begin(), sorted.end(), [u](uint32_t a, uint32_t b) { return memcmp(u + 56 * (size_t)a, u + 56 * (size_t)b, 56) < 0; });
    return sorted;
}
// The lookup call as abi.cu runs it: LaneX448PeerLookup, the order (std::stable_sort gives the device's stable radix sort's order,
// as in decaf_peerset.cpp), SlotX448PeerLookup over the elements in that order.
EXPORT int32_t goldilocks_x448_peerset_lookup_batch(uint8_t *o, int32_t *st, uint32_t *peer_index, const hostsim_peerset *ps, const uint8_t *base,
                                                   const uint8_t *sc, size_t n) {
    if (n == 0) return -1;
    const uint32_t m = (uint32_t)ps->m;
    const std::vector<uint32_t> sorted = peerset_sorted(ps);
    std::vector<uint32_t> idx(n), keys(n), order(n);
    LaneX448PeerLookup fl = {idx.data(), base, ps->peers.data(), sorted.data(), m};
    run(fl, n);
    LaneDecafPeerKeys fk = {keys.data(), order.data(), idx.data(), m};
    run(fk, n);
    std::stable_sort(order.begin(), order.end(), [&keys](uint32_t a, uint32_t b) { return keys[a] < keys[b]; });
    SlotX448PeerLookup f = {o, st, ps->tables.data(), ps->table_ok.data(), idx.data(), order.data(), base, sc, m};
    run_sm(f, n);
    if (peer_index) memcpy(peer_index, idx.data(), sizeof(uint32_t) * n);
    return -1;
}
