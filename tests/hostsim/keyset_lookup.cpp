// tests/hostsim/keyset_lookup.cpp -- TEST INFRASTRUCTURE ONLY (never shipped, never loaded by the product).
//
// goldilocks_ed448_verify_keyset_lookup_batch (include/goldilocks_b200.h) on the host, in the manner of hostsim.cpp: the device
// functors LaneKeysetLookup, LaneDecafPeerKeys, LaneKeysetHits, LaneEdVerifyScalars, SlotEdVerifyFinishKeysetOrdered,
// LaneVerifySign, LaneKeysetMissLengths, LaneKeysetMissGather and LaneKeysetScatter compiled with the host compiler and run in
// plain loops over host memory, so the CPU tier checks the CUDA source of the lookup call.  It builds on hostsim.cpp (its key sets,
// loops and goldilocks_ed448_verify_batch for the misses) and exports everything that library exports plus the lookup call.
// Built as its own library (tests/hostsim/_hostsim_keyset_lookup.so).
#include "hostsim.cpp"

// The set's indices in key-byte order, ties by index: what goldilocks_b200_keyset_create keeps on the device (abi.cu sorts them
// with the same std::stable_sort); hostsim.cpp's key sets do not keep it, so it is made here, per call.
static std::vector<uint32_t> keyset_sorted(const hostsim_keyset *ks) {
    std::vector<uint32_t> sorted(ks->m);
    for (size_t i = 0; i < ks->m; i++) sorted[i] = (uint32_t)i;
    const uint8_t *pk = ks->pk.data();
    std::stable_sort(sorted.begin(), sorted.end(), [pk](uint32_t a, uint32_t b) { return memcmp(pk + 57 * (size_t)a, pk + 57 * (size_t)b, 57) < 0; });
    return sorted;
}
// The lookup call as abi.cu runs it: LaneKeysetLookup, the order (std::stable_sort gives the device's stable radix sort's order, as
// in pointset.cpp), the hits through SlotEdVerifyFinishKeysetOrdered, the misses packed by the device's gather functors and
// through hostsim.cpp's goldilocks_ed448_verify_batch, the statuses scattered back.
EXPORT int32_t goldilocks_ed448_verify_keyset_lookup_batch(int32_t *st, uint32_t *key_index, const hostsim_keyset *ks, const uint8_t *sig, const uint8_t *pk,
                                                           const uint8_t *msg, const size_t *off, uint8_t prehashed, const uint8_t *ctx, uint8_t ctx_len, size_t n) {
    if (n == 0) return -1;
    const uint32_t m = (uint32_t)ks->m;
    const std::vector<uint32_t> sorted = keyset_sorted(ks);
    std::vector<uint32_t> idx(n), keys(n), order(n);
    LaneKeysetLookup fl = {idx.data(), pk, ks->pk.data(), sorted.data(), m};
    run(fl, n);
    LaneDecafPeerKeys fk = {keys.data(), order.data(), idx.data(), m};
    run(fk, n);
    std::stable_sort(order.begin(), order.end(), [&keys](uint32_t a, uint32_t b) { return keys[a] < keys[b]; });
    std::vector<uint32_t> keys_s(n);
    for (size_t j = 0; j < n; j++) keys_s[j] = keys[order[j]];
    uint32_t hits = 0;
    LaneKeysetHits fh = {&hits, keys_s.data(), m, n};
    run(fh, n);
    std::vector<int32_t> st_sorted(n);
    if (hits) {
        std::vector<abi_sc> chal(n), resp(n);
        LaneEdVerifyScalars f2 = {chal.data(), resp.data(), sig, pk, msg, off, prehashed, ctx, ctx_len, 0};
        run(f2, n);
        std::vector<verify_aux> aux(hits);
        if (ks->flat) {
            SlotEdVerifyFinishKeysetOrdered<true> f3 = {aux.data(), ks->key_ok.data(), chal.data(), resp.data(), wide_table(), ks->ktabs.data(), idx.data(), order.data(), sig};
            run_smp(f3, hits);
        } else {
            SlotEdVerifyFinishKeysetOrdered<false> f3 = {aux.data(), ks->key_ok.data(), chal.data(), resp.data(), wide_table(), ks->ktabs.data(), idx.data(), order.data(), sig};
            run_smp(f3, hits);
        }
        LaneVerifySign fv = {st_sorted.data(), aux.data(), 1, hits};
        run(fv, (hits + VSIGN_BATCH - 1) / VSIGN_BATCH);
    }
    const size_t misses = n - hits;
    if (misses) {
        std::vector<size_t> len(misses + 1), off2(misses + 1);
        LaneKeysetMissLengths fln = {len.data(), off, order.data(), hits, misses};
        run(fln, misses + 1);
        for (size_t q = 0, acc = 0; q <= misses; q++) { off2[q] = acc; acc += len[q]; }   /* the device's exclusive scan */
        std::vector<uint8_t> sig2(114 * misses), pk2(57 * misses), msg2(off2[misses] + 1);
        LaneKeysetMissGather fg = {sig2.data(), pk2.data(), msg2.data(), off2.data(), sig, pk, msg, off, order.data(), hits};
        run(fg, misses);
        goldilocks_ed448_verify_batch(st_sorted.data() + hits, sig2.data(), pk2.data(), msg2.data(), off2.data(), prehashed, ctx, ctx_len, misses);
    }
    LaneKeysetScatter fs = {st, st_sorted.data(), order.data()};
    run(fs, n);
    if (key_index) memcpy(key_index, idx.data(), sizeof(uint32_t) * n);
    return -1;
}
