// tools/ct_layout.cpp -- kernel-parameter layout of the secret-handling kernels, for tools/ct_audit.py.
//
// Every kernel takes its lane functor by value as the first parameter, so field `f` of the functor sits at
// constant-bank offset PARAM_BASE + offsetof(F, f).  This program prints, as JSON, each audited kernel with the byte
// offset of every field and how the audit has to treat data loaded through it:
//   secret : private keys, scalars, nonces, seeds -- everything loaded through it is TAINTED
//   public : public inputs (peer points, messages, offsets, contexts, fixed tables) -- loads are clean
//   out    : results / scratch written by this or an earlier kernel -- loads are treated as tainted (conservative)
//   value  : a scalar parameter (flags, lengths) -- public
// Built and run by ct_audit.py with the host compiler (the CUDA headers are host-clean, like tests/hostsim).
#include <cstddef>
#include <cstdio>

#include "../libgoldilocks_b200/csrc/slot_lanes.cuh"

static bool first_kernel = true, first_field = true;
static void kernel(const char *functor, size_t size) {
    printf("%s\n \"%s\": {\"size\": %zu, \"fields\": [", first_kernel ? "" : "]},", functor, size);
    first_kernel = false;
    first_field = true;
}
static void field(const char *name, size_t off, size_t size, const char *cls) {
    printf("%s{\"name\": \"%s\", \"offset\": %zu, \"size\": %zu, \"class\": \"%s\"}", first_field ? "" : ", ", name, off, size, cls);
    first_field = false;
}
#define K(F) kernel(#F, sizeof(F))
#define FLD(F, f, cls) field(#f, offsetof(F, f), sizeof(((F *)0)->f), cls)

int main() {
    printf("{");
    K(SlotX448); FLD(SlotX448, out, "out"); FLD(SlotX448, status, "out"); FLD(SlotX448, base, "public"); FLD(SlotX448, scalar, "secret");
    K(SlotX448Peer); FLD(SlotX448Peer, out, "out"); FLD(SlotX448Peer, status, "out"); FLD(SlotX448Peer, tables, "public"); FLD(SlotX448Peer, table_ok, "public");
    FLD(SlotX448Peer, peers, "public"); FLD(SlotX448Peer, peer_index, "public"); FLD(SlotX448Peer, scalar, "secret"); FLD(SlotX448Peer, n_peers, "value");
    K(SlotX448PeerLookup); FLD(SlotX448PeerLookup, out, "out"); FLD(SlotX448PeerLookup, status, "out"); FLD(SlotX448PeerLookup, tables, "public");
    FLD(SlotX448PeerLookup, table_ok, "public"); FLD(SlotX448PeerLookup, peer_index, "public"); FLD(SlotX448PeerLookup, order, "public");
    FLD(SlotX448PeerLookup, base, "public"); FLD(SlotX448PeerLookup, scalar, "secret"); FLD(SlotX448PeerLookup, n_peers, "value");
    K(SlotDecafPeer); FLD(SlotDecafPeer, scaled, "out"); FLD(SlotDecafPeer, status, "out"); FLD(SlotDecafPeer, tables, "public"); FLD(SlotDecafPeer, peer_ok, "public");
    FLD(SlotDecafPeer, peer_index, "public"); FLD(SlotDecafPeer, order, "public"); FLD(SlotDecafPeer, scalar, "secret"); FLD(SlotDecafPeer, n_peers, "value");
    FLD(SlotDecafPeer, short_circuit, "value");
    K(SlotComb); FLD(SlotComb, out, "out"); FLD(SlotComb, scalar, "secret"); FLD(SlotComb, ft, "public");
    K(SlotCombTable); FLD(SlotCombTable, out, "out"); FLD(SlotCombTable, scalar, "secret"); FLD(SlotCombTable, table, "public");
    K(SlotX448DerivePk); FLD(SlotX448DerivePk, out, "out"); FLD(SlotX448DerivePk, scalar, "secret"); FLD(SlotX448DerivePk, ft, "public");
    K(SlotEdDerivePk); FLD(SlotEdDerivePk, pk, "out"); FLD(SlotEdDerivePk, sk, "secret"); FLD(SlotEdDerivePk, ft, "public");
    K(SlotEdSignR); FLD(SlotEdSignR, sig, "out"); FLD(SlotEdSignR, nonce4, "secret"); FLD(SlotEdSignR, ft, "public");
    K(SlotScalarmul); FLD(SlotScalarmul, out, "out"); FLD(SlotScalarmul, base, "public"); FLD(SlotScalarmul, scalar, "secret"); FLD(SlotScalarmul, scratch, "out");
    K(SlotDoubleScalarmul); FLD(SlotDoubleScalarmul, out, "out"); FLD(SlotDoubleScalarmul, base1, "public"); FLD(SlotDoubleScalarmul, scalar1, "secret");
    FLD(SlotDoubleScalarmul, base2, "public"); FLD(SlotDoubleScalarmul, scalar2, "secret"); FLD(SlotDoubleScalarmul, scratch, "out"); FLD(SlotDoubleScalarmul, nthreads, "value");
    K(SlotDualScalarmul); FLD(SlotDualScalarmul, out1, "out"); FLD(SlotDualScalarmul, out2, "out"); FLD(SlotDualScalarmul, base, "public");
    FLD(SlotDualScalarmul, scalar1, "secret"); FLD(SlotDualScalarmul, scalar2, "secret"); FLD(SlotDualScalarmul, scratch, "out");
    K(SlotDirectScalarmul); FLD(SlotDirectScalarmul, scaled, "out"); FLD(SlotDirectScalarmul, status, "out"); FLD(SlotDirectScalarmul, base, "public");
    FLD(SlotDirectScalarmul, scalar, "secret"); FLD(SlotDirectScalarmul, allow_identity, "value"); FLD(SlotDirectScalarmul, short_circuit, "value");
    FLD(SlotDirectScalarmul, ft, "public"); FLD(SlotDirectScalarmul, scratch, "out");
    K(LaneEdSignExpand); FLD(LaneEdSignExpand, secret, "out"); FLD(LaneEdSignExpand, seed, "out"); FLD(LaneEdSignExpand, sk, "secret");
    K(LaneEdSignNonce); FLD(LaneEdSignNonce, nonce, "out"); FLD(LaneEdSignNonce, nonce4, "out"); FLD(LaneEdSignNonce, seed, "secret"); FLD(LaneEdSignNonce, msg, "public");
    FLD(LaneEdSignNonce, off, "public"); FLD(LaneEdSignNonce, prehashed, "value"); FLD(LaneEdSignNonce, ctx, "public"); FLD(LaneEdSignNonce, ctx_len, "value");
    K(LaneEdSignFinish); FLD(LaneEdSignFinish, sig, "public"); /* reads the R half it is about to complete: public */
    FLD(LaneEdSignFinish, secret, "secret"); FLD(LaneEdSignFinish, nonce, "secret"); FLD(LaneEdSignFinish, pk, "public"); FLD(LaneEdSignFinish, msg, "public");
    FLD(LaneEdSignFinish, off, "public"); FLD(LaneEdSignFinish, prehashed, "value"); FLD(LaneEdSignFinish, ctx, "public"); FLD(LaneEdSignFinish, ctx_len, "value");
    K(LaneEdSecretScalar); FLD(LaneEdSecretScalar, out, "out"); FLD(LaneEdSecretScalar, sk, "secret");
    K(LaneEdSkToX448); FLD(LaneEdSkToX448, x, "out"); FLD(LaneEdSkToX448, ed, "secret");
    /* negative control: the verification multiply indexes its tables with digits of its (public) scalars; labelled secret here, the audit must FAIL it */
    K(SlotBaseDoubleScalarmul); FLD(SlotBaseDoubleScalarmul, out, "out"); FLD(SlotBaseDoubleScalarmul, scalar1, "secret"); FLD(SlotBaseDoubleScalarmul, base2, "public");
    FLD(SlotBaseDoubleScalarmul, scalar2, "secret"); FLD(SlotBaseDoubleScalarmul, wide, "public"); FLD(SlotBaseDoubleScalarmul, scratch, "out");
    printf("]}\n}\n");
    return 0;
}
