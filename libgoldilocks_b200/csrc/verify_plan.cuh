// verify_plan.cuh -- work lists of a verification batch, made on the device by the key-grouping pass (k_group.cu).
#pragma once
#include <stddef.h>
#include <stdint.h>
// Signatures whose 57 public-key bytes occur at least twice in the batch are verified against one per-key table
// (SlotKeyChain + SlotKeyColumns / SlotEdVerifyFinishShared); everything else goes through SlotEdVerifyFinish on its own.
//   shared_sig[j], shared_tab[j] : signature index and key-table index of the j-th table-path signature, ordered so
//                                  that signatures under one key are adjacent lanes (their table rows stay in L1/L2)
//   unique_sig[j]                : signature index of the j-th stand-alone signature
//   tab_rep[t]                   : a signature whose public key is key t (its decoded point seeds the table)
//   counts[0..2]                 : number of table-path signatures, stand-alone signatures, key tables;
//                                  counts[3..5] = 0: work counters of the finish / key-chain / key-column kernels' dynamic hand-out
// A null unique_sig means "no plan: every signature, in order, stand-alone".
struct verify_plan {
    const uint32_t *shared_sig, *shared_tab, *unique_sig, *tab_rep, *counts;
};
#if defined(__CUDACC__)
#include <cuda_runtime.h>
// Bytes of device scratch group_keys() needs for n signatures and at most `cap` key tables.
size_t group_scratch_bytes(size_t n, size_t cap);
// Enqueues the grouping pass on `s`; `plan` receives pointers into `scratch`.  No host synchronisation.
// Every distinct key of a batch (k_group.cu group_keys_all): the view the random-linear-combination path works from.
struct key_groups { const uint32_t *order, *gid, *gstart, *ngroups; };
size_t group_all_scratch_bytes(size_t n);
cudaError_t group_keys_all(const uint8_t *pk, size_t n, void *scratch, key_groups *out, cudaStream_t s, uint64_t *launches, uint32_t csize = 0);
cudaError_t key_chunks(uint32_t *kchunk, const key_groups *g, uint32_t m, uint32_t nch, uint32_t csize, cudaStream_t s);
size_t pair_sort_scratch_bytes(size_t npairs);
cudaError_t pair_sort(void *tmp, size_t tmp_bytes, const uint32_t *keys_in, uint32_t *keys_out, const uint32_t *vals_in, uint32_t *vals_out, size_t npairs,
                      int key_bits, cudaStream_t s);
size_t length_scan_scratch_bytes(size_t count);
cudaError_t length_scan(void *tmp, size_t tmp_bytes, const size_t *len, size_t *off, size_t count, cudaStream_t s);
cudaError_t group_keys(const uint8_t *pk, size_t n, uint32_t cap, void *scratch, verify_plan *plan, cudaStream_t s, uint64_t *launches);
#endif
