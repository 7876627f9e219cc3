// launch.cuh -- kernel shapes around the lane functors of lanes.cuh and their host-side launchers.
//
// Each heavy functor is compiled in its own translation unit (k_*.cu explicitly instantiates the
// launchers for its functors); abi.cu only sees `extern template` declarations, so the library
// builds in parallel and a change to one kernel recompiles one file.
#pragma once
#include <cuda_runtime.h>
#include "slot_lanes.cuh"
#include "rlc.cuh"

#define BLOCK 128

// Resident blocks per SM the register allocator is asked to allow (default: whatever fits).
template <class F> struct lane_min_blocks { static constexpr int value = 1; };
/* The one-inverse-square-root kernels run the by-value multiplier and want ~186 registers, i.e. two blocks = two warps per scheduler.
 * Capping the registers for three / four resident blocks costs 64-600 bytes of spills outside the squaring loop and wins 2-3.5 %
 * (B200, 2^20: RLC call 17.96 -> 17.43 ms with 3, 17.56 with 4; decaf decode 8.24 -> 8.07 / 7.95 ms, encode 8.12 -> 7.87 / 7.89,
 * Elligator 8.29 -> 8.13 / 8.05; tools/gpu_variants_decode.sh). */
#ifndef DECODE_MIN_BLOCKS
#define DECODE_MIN_BLOCKS 3
#endif
#ifndef CODEC_MIN_BLOCKS
#define CODEC_MIN_BLOCKS 4
#endif
template <> struct lane_min_blocks<LaneRlcDecode> { static constexpr int value = DECODE_MIN_BLOCKS; };
template <> struct lane_min_blocks<LaneEdVerifyDecode> { static constexpr int value = DECODE_MIN_BLOCKS; };
template <> struct lane_min_blocks<LanePtDecode> { static constexpr int value = CODEC_MIN_BLOCKS; };
template <> struct lane_min_blocks<LanePtEncode> { static constexpr int value = CODEC_MIN_BLOCKS; };
template <> struct lane_min_blocks<LaneFromHash<false>> { static constexpr int value = CODEC_MIN_BLOCKS; };

template <class F>
__global__ void __launch_bounds__(BLOCK, lane_min_blocks<F>::value) k_lanes(F f, size_t n) {
    const size_t i = (size_t)blockIdx.x * BLOCK + threadIdx.x;
    if (i < n) f(i);
}
template <class F>
cudaError_t launch_lanes(const F &f, size_t n, cudaStream_t s) {
    k_lanes<F><<<(unsigned)((n + BLOCK - 1) / BLOCK), BLOCK, 0, s>>>(f, n);
    return cudaGetLastError();
}
// Slot-machine kernels (slots.cuh): F::NSLOTS x 64 B of dynamic shared memory per lane.
// Resident blocks per SM: measured choice per functor (registers <= 65536 / (128 * blocks)).
#ifndef SLOT7_MIN_BLOCKS
#define SLOT7_MIN_BLOCKS 4 /* 7 slots = 56 KB per block: four blocks (16 warps) per SM, 128 registers */
#endif
template <> struct slot_min_blocks<SlotX448> { static constexpr int value = 4; };
template <> struct slot_min_blocks<SlotX448Peer> { static constexpr int value = 4; };
template <> struct slot_min_blocks<SlotX448PeerLookup> { static constexpr int value = 4; };
template <> struct slot_min_blocks<SlotNielsDebug> { static constexpr int value = 4; };
template <> struct slot_min_blocks<SlotComb> { static constexpr int value = SLOT7_MIN_BLOCKS; };
template <> struct slot_min_blocks<SlotX448DerivePk> { static constexpr int value = SLOT7_MIN_BLOCKS; };
template <> struct slot_min_blocks<SlotEdDerivePk> { static constexpr int value = SLOT7_MIN_BLOCKS; };
template <> struct slot_min_blocks<SlotEdSignR> { static constexpr int value = SLOT7_MIN_BLOCKS; };
template <> struct slot_min_blocks<SlotCombTable> { static constexpr int value = SLOT7_MIN_BLOCKS; };
template <> struct slot_min_blocks<SlotDecafPeer> { static constexpr int value = SLOT7_MIN_BLOCKS; };
template <> struct slot_min_blocks<SlotDualScalarmul> { static constexpr int value = SLOT7_MIN_BLOCKS; };
template <> struct slot_min_blocks<SlotDirectScalarmul> { static constexpr int value = SLOT7_MIN_BLOCKS; };
template <> struct slot_min_blocks<SlotScalarmul> { static constexpr int value = SLOT7_MIN_BLOCKS; };
template <> struct slot_min_blocks<SlotDoubleScalarmul> { static constexpr int value = SLOT7_MIN_BLOCKS; };
template <> struct slot_min_blocks<SlotEdVerifyFinish> { static constexpr int value = 4; }; /* 3 blocks (no spills): 111.7 vs 110.9 ms */
template <> struct slot_min_blocks<SlotBaseDoubleScalarmul> { static constexpr int value = 4; };
template <> struct slot_min_blocks<SlotEdVerifyFinishShared> { static constexpr int value = 4; };
template <> struct slot_min_blocks<SlotKeyChain> { static constexpr int value = 4; };
template <> struct slot_min_blocks<SlotKeyColumns> { static constexpr int value = 4; };
template <> struct slot_min_blocks<SlotRlcBucket> { static constexpr int value = 4; };
template <> struct slot_min_blocks<SlotKeysetTables> { static constexpr int value = 4; };
template <> struct slot_min_blocks<SlotEdVerifyFinishKeyset> { static constexpr int value = 4; };
template <> struct slot_min_blocks<SlotEdVerifyFinishKeysetFlat> { static constexpr int value = 4; };
template <> struct slot_min_blocks<SlotKeysetChain> { static constexpr int value = 4; };
template <> struct slot_min_blocks<SlotKeysetColumns> { static constexpr int value = 4; };
template <bool FLAT> struct slot_min_blocks<SlotPointset<FLAT>> { static constexpr int value = 4; };
template <bool FLAT> struct slot_min_blocks<SlotEdVerifyFinishKeysetOrdered<FLAT>> { static constexpr int value = 4; };
template <class F>
cudaError_t launch_sm(const F &f, size_t n, cudaStream_t s) {
    const int smem = F::NSLOTS * 64 * SLOT_BLOCK;
    static bool configured_dev[64]; /* per functor and device; racing first calls set the same values */
    int dev = 0;
    cudaError_t e0 = cudaGetDevice(&dev);
    if (e0 != cudaSuccess) return e0;
    bool &configured = configured_dev[dev & 63];
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(k_slots<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(k_slots<F>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
        configured = true;
    }
    k_slots<F><<<(unsigned)((n + SLOT_BLOCK - 1) / SLOT_BLOCK), SLOT_BLOCK, smem, s>>>(f, n);
    return cudaGetLastError();
}

// Persistent variant: grid = SMs x resident blocks (sm_persist_grid), one HBM scratch area per thread.
template <class F>
cudaError_t sm_configure(int *blocks_per_sm) {
    const int smem = F::NSLOTS * 64 * SLOT_BLOCK;
    cudaError_t e = cudaFuncSetAttribute(k_slots_persist<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_slots_persist<F>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, k_slots_persist<F>, SLOT_BLOCK, smem);
}
template <class F>
cudaError_t launch_sm_persist(const F &f, size_t n, int grid, cudaStream_t s, unsigned *work_counter) {
    k_slots_persist<F><<<grid, SLOT_BLOCK, F::NSLOTS * 64 * SLOT_BLOCK, s>>>(f, n, work_counter); /* *work_counter == 0 on entry */
    return cudaGetLastError();
}

#define LANES_PLAIN(X)                                                                              \
    X(LanePt<PTOP_NEG>) X(LanePt<PTOP_TORQUE>) X(LanePtPscale)                 \
    X(LanePtEq) X(LanePtValid) X(LanePtEncode) X(LanePtDecode)                                      \
    X(LaneFromHash<false>) X(LaneFromHash<true>) X(LaneInvertElligator<false>) X(LaneInvertElligator<true>)                                                    \
    X(LaneEncodeEddsa) X(LaneDecodeEddsa) X(LaneEncodeX448)                                         \
    X(LaneSc<SCOP_ADD>) X(LaneSc<SCOP_SUB>) X(LaneSc<SCOP_MUL>) X(LaneSc<SCOP_HALVE>)               \
    X(LaneScDecodeLong) X(LaneScInvert) X(LaneShake256) X(LaneSpongeUpdate) X(LaneSpongeOutput) X(LaneEdPkToX448) X(LaneEdSkToX448) X(LanePrecompute) X(LaneNielsFromAbi) X(LaneX448PeerLift) X(LaneDecafPeerDecode) X(LaneDecafPeerKeys)                                                             \
    X(LaneEdSecretScalar) X(LaneEdSignExpand) X(LaneEdSignNonce) X(LaneEdSignFinish)   \
    X(LaneEdVerifyDecode) X(LaneEdVerifyScalars) X(LaneVerifySign) X(LaneVerifyHalf) X(LaneKeysetNormalize) X(LaneBuildTables) X(LaneBuildWide) \
    X(LaneRlcDecode) X(LaneRlcZ) X(LaneRlcWeights) X(LaneRlcLate) X(LaneRlcKeyScalars) X(LaneRlcDigits) X(LaneRlcBucketRuns) X(LaneRlcSegments) X(LaneRlcNodes) X(LaneRlcWindows) X(LaneRlcTotal) X(LaneRlcVerdict) X(LaneRlcPackPlan) X(LaneRlcPack) X(LaneRlcUnpack) X(LanePtNiels) \
    X(LaneKeysetLookup) X(LaneX448PeerLookup) X(LaneKeysetHits) X(LaneKeysetMissLengths) X(LaneKeysetMissGather) X(LaneKeysetScatter)

#define LANES_SM(X) X(SlotNielsDebug) X(SlotX448) X(SlotX448Peer) X(SlotX448PeerLookup) X(SlotComb) X(SlotCombTable) X(SlotDecafPeer) X(SlotX448DerivePk) X(SlotEdDerivePk) X(SlotEdSignR) X(SlotRlcBucket)
#define INSTANTIATE_SM(F) template cudaError_t launch_sm<F>(const F &, size_t, cudaStream_t);
#define DECLARE_SM(F) extern INSTANTIATE_SM(F)
#define LANES_SMP(X) X(SlotEdVerifyFinish) X(SlotEdVerifyFinishShared) X(SlotKeyChain) X(SlotKeyColumns) X(SlotKeysetTables) X(SlotKeysetChain) X(SlotKeysetColumns) X(SlotEdVerifyFinishKeyset) X(SlotEdVerifyFinishKeysetFlat) X(SlotPointset<true>) X(SlotPointset<false>) X(SlotEdVerifyFinishKeysetOrdered<true>) X(SlotEdVerifyFinishKeysetOrdered<false>) X(SlotBaseDoubleScalarmul) X(SlotScalarmul) X(SlotDoubleScalarmul) X(SlotDualScalarmul) X(SlotDirectScalarmul)
#define INSTANTIATE_SMP(F)                                                                          \
    template cudaError_t sm_configure<F>(int *);                                                    \
    template cudaError_t launch_sm_persist<F>(const F &, size_t, int, cudaStream_t, unsigned *);
#define DECLARE_SMP(F)                                                                              \
    extern template cudaError_t sm_configure<F>(int *);                                             \
    extern template cudaError_t launch_sm_persist<F>(const F &, size_t, int, cudaStream_t, unsigned *);
#define INSTANTIATE_PLAIN(F) template cudaError_t launch_lanes<F>(const F &, size_t, cudaStream_t);
#define DECLARE_PLAIN(F) extern INSTANTIATE_PLAIN(F)
