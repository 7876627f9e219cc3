// k_keyset.cu -- explicit kernel instantiations (see launch.cuh): key-set lookup calls, and the scan of their miss path
#include <cub/device/device_scan.cuh>
#include "launch.cuh"
INSTANTIATE_PLAIN(LaneKeysetLookup)
INSTANTIATE_PLAIN(LaneKeysetHits)
INSTANTIATE_PLAIN(LaneKeysetMissLengths)
INSTANTIATE_PLAIN(LaneKeysetMissGather)
INSTANTIATE_PLAIN(LaneKeysetScatter)
INSTANTIATE_SMP(SlotEdVerifyFinishKeysetOrdered<true>)
INSTANTIATE_SMP(SlotEdVerifyFinishKeysetOrdered<false>)

// Exclusive prefix sum of `count` message lengths (the offsets of the packed misses); a CUB primitive, plumbing.
size_t length_scan_scratch_bytes(size_t count) {
    size_t b = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, b, (const size_t *)nullptr, (size_t *)nullptr, (int)count);
    return b + 256;
}
cudaError_t length_scan(void *tmp, size_t tmp_bytes, const size_t *len, size_t *off, size_t count, cudaStream_t s) {
    return cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, len, off, (int)count, s);
}
