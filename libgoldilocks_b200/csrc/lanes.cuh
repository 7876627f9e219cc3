// lanes.cuh -- one functor per batched entry point: `operator()(i)` processes element i of the
// packed host-layout arrays (include/goldilocks_b200.h).  The CUDA kernels in kernels.cu are thin
// launch wrappers around these functors; the test-only host simulator runs the same functors in a
// plain loop.  Nothing here allocates or synchronises.
#pragma once
#include <stddef.h>
#include "algos.cuh"
#include "verify_plan.cuh"

// ---- host-ABI layouts (reference x86_64 ABI: f_field.h:23-27, point_448.h:66-86) -------------
struct abi_gf { uint64_t limb[8]; };
struct abi_pt { abi_gf x, y, z, t; };
struct abi_sc { uint64_t limb[7]; };

// radix-2^56 limbs (any value < 2^60 per limb) -> TIGHT radix-2^28
GD void gf_from_abi(gf &o, const abi_gf *a) {
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const uint64_t l = a->limb[k];
        o.v[2 * k] = (uint32_t)l & GF_MASK;
        o.v[2 * k + 1] = (uint32_t)(l >> 28);
    }
    gf_weak_reduce(o);
}
// canonical radix-2^56 limbs
GD void gf_to_abi(abi_gf *o, const gf &a_in) {
    gf a;
    gf_copy(a, a_in);
    gf_strong_reduce(a);
#pragma unroll
    for (int k = 0; k < 8; k++) o->limb[k] = (uint64_t)a.v[2 * k] | ((uint64_t)a.v[2 * k + 1] << 28);
}
GD void pt_from_abi(pt &o, const abi_pt *a) { gf_from_abi(o.x, &a->x); gf_from_abi(o.y, &a->y); gf_from_abi(o.z, &a->z); gf_from_abi(o.t, &a->t); }
GD void pt_to_abi(abi_pt *o, const pt &a) { gf_to_abi(&o->x, a.x); gf_to_abi(&o->y, a.y); gf_to_abi(&o->z, a.z); gf_to_abi(&o->t, a.t); }
GD void sc_from_abi(sc &o, const abi_sc *a) {
#pragma unroll
    for (int k = 0; k < 7; k++) { o.w[2 * k] = (uint32_t)a->limb[k]; o.w[2 * k + 1] = (uint32_t)(a->limb[k] >> 32); }
}
GD void sc_to_abi(abi_sc *o, const sc &a) {
#pragma unroll
    for (int k = 0; k < 7; k++) o->limb[k] = (uint64_t)a.w[2 * k] | ((uint64_t)a.w[2 * k + 1] << 32);
}
// 56-byte records are 8-byte aligned in every batch array (element stride 56, 256-byte aligned base)
GD void words_load56(uint32_t w[14], const uint8_t *p) {
    const uint64_t *q = (const uint64_t *)p;
#pragma unroll
    for (int k = 0; k < 7; k++) { const uint64_t x = q[k]; w[2 * k] = (uint32_t)x; w[2 * k + 1] = (uint32_t)(x >> 32); }
}
GD void words_store56(uint8_t *p, const uint32_t w[14]) {
    uint64_t *q = (uint64_t *)p;
#pragma unroll
    for (int k = 0; k < 7; k++) q[k] = (uint64_t)w[2 * k] | ((uint64_t)w[2 * k + 1] << 32);
}
// unaligned byte records (57-byte EdDSA strings)
GD void words_load_bytes(uint32_t *w, int nwords, const uint8_t *p, int nbytes) {
    for (int k = 0; k < nwords; k++) {
        uint32_t x = 0;
        for (int b = 0; b < 4; b++) { const int idx = 4 * k + b; if (idx < nbytes) x |= (uint32_t)p[idx] << (8 * b); }
        w[k] = x;
    }
}
GD void words_store_bytes(uint8_t *p, int nbytes, const uint32_t *w) {
    for (int idx = 0; idx < nbytes; idx++) p[idx] = (uint8_t)(w[idx >> 2] >> (8 * (idx & 3)));
}
#define ST_OK(m) ((int32_t)(m)) /* mask -> goldilocks_error_t (-1 success / 0 failure) */

// ---- field level (BASELINE config 1) --------------------------------------------------------
enum { GFOP_MUL, GFOP_SQR, GFOP_ADD, GFOP_SUB, GFOP_MULW, GFOP_ISR, GFOP_INVERT };
template <int OP>
struct LaneGf {
    uint8_t *out; int32_t *status; const uint8_t *a, *b; uint32_t w;
    GDM void operator()(size_t i) const {
        uint32_t wa[14], wb[14], wo[14];
        gf x, y, z;
        words_load56(wa, a + 56 * i);
        (void)gf_from_words(x, wa);
        if (OP == GFOP_MUL || OP == GFOP_ADD || OP == GFOP_SUB) { words_load56(wb, b + 56 * i); (void)gf_from_words(y, wb); }
        if (OP == GFOP_MUL) gf_mul(z, x, y);
        if (OP == GFOP_SQR) gf_sqr(z, x);
        if (OP == GFOP_ADD) gf_add(z, x, y);
        if (OP == GFOP_SUB) gf_sub(z, x, y);
        if (OP == GFOP_MULW) gf_mulw(z, x, w);
        if (OP == GFOP_ISR) status[i] = ST_OK(gf_isr(z, x));
        if (OP == GFOP_INVERT) gf_invert(z, x);
        gf_to_words(wo, z);
        words_store56(out + 56 * i, wo);
    }
};

// ---- group level -----------------------------------------------------------------------------
enum { PTOP_ADD, PTOP_SUB, PTOP_DBL, PTOP_NEG, PTOP_TORQUE };
template <int OP>
struct LanePt {
    abi_pt *out; const abi_pt *a, *b;
    GDM void operator()(size_t i) const {
        pt p, q, r;
        pt_from_abi(q, a + i);
        if (OP == PTOP_ADD || OP == PTOP_SUB) pt_from_abi(r, b + i);
        if (OP == PTOP_ADD) pt_add(p, q, r);
        if (OP == PTOP_SUB) pt_sub(p, q, r);
        if (OP == PTOP_DBL) pt_double(p, q, false);
        if (OP == PTOP_NEG) pt_negate(p, q);
        if (OP == PTOP_TORQUE) { gf_neg(p.x, q.x); gf_neg(p.y, q.y); gf_copy(p.z, q.z); gf_copy(p.t, q.t); } /* goldilocks.c:675-683: add the 2-torsion point */
        pt_to_abi(out + i, p);
    }
};
struct LanePtPscale { /* goldilocks_448_point_debugging_pscale (goldilocks.c:685-702): another representative of the same point */
    abi_pt *out; const abi_pt *a; const uint8_t *factor;
    GDM void operator()(size_t i) const {
        pt q, p; gf f, one; uint32_t w[14];
        pt_from_abi(q, a + i);
        words_load56(w, factor + 56 * i);
        (void)gf_from_words(f, w);
        gf_set_ui(one, 1);
        gf_cond_sel(f, f, one, gf_is_zero(f));
        gf_mul(p.x, q.x, f); gf_mul(p.y, q.y, f); gf_mul(p.z, q.z, f); gf_mul(p.t, q.t, f);
        pt_to_abi(out + i, p);
    }
};
struct LanePtEq {
    uint64_t *out; const abi_pt *a, *b;
    GDM void operator()(size_t i) const {
        pt q, r;
        pt_from_abi(q, a + i);
        pt_from_abi(r, b + i);
        out[i] = pt_eq(q, r) ? ~0ull : 0ull;
    }
};
struct LanePtValid {
    uint64_t *out; const abi_pt *a;
    GDM void operator()(size_t i) const {
        pt q;
        pt_from_abi(q, a + i);
        out[i] = pt_valid(q) ? ~0ull : 0ull;
    }
};
struct LanePtEncode {
    uint8_t *out; const abi_pt *a;
    GDM void operator()(size_t i) const {
        pt q; gf s; uint32_t w[14];
        pt_from_abi(q, a + i);
        pt_deisogenize(s, q);
        gf_to_words(w, s);
        words_store56(out + 56 * i, w);
    }
};
struct LanePtDecode {
    abi_pt *out; int32_t *status; const uint8_t *ser; uint32_t allow_identity;
    GDM void operator()(size_t i) const {
        pt p; uint32_t w[14];
        words_load56(w, ser + 56 * i);
        gmask_t ok = pt_decode(p, w, allow_identity ? ~0u : 0u);
        pt_to_abi(out + i, p);
        status[i] = ST_OK(ok);
    }
};
template <bool UNIFORM>
struct LaneFromHash {
    abi_pt *out; const uint8_t *hashed;
    GDM void operator()(size_t i) const {
        pt p; uint32_t w[14];
        words_load56(w, hashed + (UNIFORM ? 112 : 56) * i);
        pt_from_hash_nonuniform(p, w);
        if (UNIFORM) { /* elligator.c:86-94 */
            pt p2;
            words_load56(w, hashed + 112 * i + 56);
            pt_from_hash_nonuniform(p2, w);
            pt_add(p, p, p2);
        }
        pt_to_abi(out + i, p);
    }
};
// Elligator inverses (elligator.c:104-164).  Uniform: hashed[112*i+56..] is the caller's second half, the
// first half is written (elligator.c:154-164).
template <bool UNIFORM>
struct LaneInvertElligator {
    uint8_t *hashed; int32_t *status; const abi_pt *a; const uint32_t *hint;
    GDM void operator()(size_t i) const {
        pt p; uint32_t w[14];
        pt_from_abi(p, a + i);
        if (UNIFORM) {
            pt p2;
            words_load56(w, hashed + 112 * i + 56);
            pt_from_hash_nonuniform(p2, w);
            pt_sub(p, p, p2);
        }
        gmask_t ok = pt_invert_elligator_nonuniform(w, p, hint[i]);
        words_store56(hashed + (UNIFORM ? 112 : 56) * i, w);
        status[i] = ST_OK(ok);
    }
};
struct LaneEncodeEddsa {
    uint8_t *out; const abi_pt *a;
    GDM void operator()(size_t i) const {
        pt q; uint32_t w[15], sign;
        pt_from_abi(q, a + i);
        pt_encode_like_eddsa(w, sign, q);
        w[14] = sign << 7;
        words_store_bytes(out + 57 * i, 57, w);
    }
};
struct LaneDecodeEddsa {
    abi_pt *out; int32_t *status; const uint8_t *enc;
    GDM void operator()(size_t i) const {
        pt p; uint32_t w[15];
        words_load_bytes(w, 15, enc + 57 * i, 57);
        gmask_t ok = pt_decode_like_eddsa(p, w, w[14] & 0xff);
        pt_to_abi(out + i, p);
        status[i] = ST_OK(ok);
    }
};
struct LaneEncodeX448 {
    uint8_t *out; const abi_pt *a;
    GDM void operator()(size_t i) const {
        pt q; uint32_t w[14];
        pt_from_abi(q, a + i);
        pt_encode_like_x448(w, q);
        words_store56(out + 56 * i, w);
    }
};

// ---- scalar multiplications ------------------------------------------------------------------
// goldilocks_448_precomputed_scalarmul / point_scalarmul / point_double_scalarmul /
// base_double_scalarmul_non_secret: SlotComb, SlotScalarmul, SlotDoubleScalarmul, SlotBaseDoubleScalarmul (slot_lanes.cuh)

// ---- scalars mod q ---------------------------------------------------------------------------
enum { SCOP_ADD, SCOP_SUB, SCOP_MUL, SCOP_HALVE };
template <int OP>
struct LaneSc {
    abi_sc *out; const abi_sc *a, *b;
    GDM void operator()(size_t i) const {
        sc x, y, z;
        sc_from_abi(x, a + i);
        if (OP != SCOP_HALVE) sc_from_abi(y, b + i);
        if (OP == SCOP_ADD) sc_add(z, x, y);
        if (OP == SCOP_SUB) sc_sub(z, x, y);
        if (OP == SCOP_MUL) sc_mul(z, x, y);
        if (OP == SCOP_HALVE) sc_halve(z, x);
        sc_to_abi(out + i, z);
    }
};
struct ByteAtPtr { const uint8_t *p; GDM uint8_t operator()(int k) const { return p[k]; } };
struct LaneScInvert { /* goldilocks_448_scalar_invert (scalar.c:107-166): SUCCESS iff the result is nonzero */
    abi_sc *out; int32_t *status; const abi_sc *a;
    GDM void operator()(size_t i) const {
        sc x, z;
        sc_from_abi(x, a + i);
        sc_invert(z, x);
        uint32_t any = 0;
#pragma unroll
        for (int k = 0; k < SC_WORDS; k++) any |= z.w[k];
        sc_to_abi(out + i, z);
        status[i] = any ? -1 : 0;
    }
};
struct LaneScDecodeLong {
    abi_sc *out; const uint8_t *ser; size_t len;
    GDM void operator()(size_t i) const {
        sc z;
        if (len == 114) {        /* the two EdDSA lengths take the folding reduction the verify / sign kernels use (sc.cuh) */
            uint32_t w[29];
            words_load_bytes(w, 29, ser + len * i, 114);
            sc_reduce_114(z, w);
        } else if (len == 57) {
            uint32_t w[15];
            words_load_bytes(w, 15, ser + len * i, 57);
            sc_reduce_57(z, w);
        } else {
            ByteAtPtr at = {ser + len * i};
            sc_decode_long(z, at, (int)len);
        }
        sc_to_abi(out + i, z);
    }
};

struct ByteAtWords { const uint32_t *w; GDM uint8_t operator()(int k) const { return (uint8_t)(w[k >> 2] >> (8 * (k & 3))); } };

// ---- streaming SHA-3 / SHAKE front end (reference shake.c:89-213) ------------------------------------
// The caller-owned sponge object of goldilocks/shake.h (26 x u64: 200 state bytes + 8 parameter bytes,
// keccak_internal.h) is copied to the device, one lane runs the reference's absorb / pad / squeeze loop
// with every Keccak-f on the device, and the object is copied back.  Bulk hashing belongs in
// goldilocks_shake256_hash_batch; this exists so prehash (Ed448ph) callers keep working.
struct sponge_abi { uint64_t w[25]; uint8_t position, flags, rate, start_round, pad, rate_pad, max_out, remaining; };
GD void sponge_permute(sponge_abi *s) { /* dokeccak (keccak_internal.h): start_round is 0 for every exported parameter set */
    keccak_state st;
#pragma unroll
    for (int i = 0; i < 25; i++) st.a[i] = s->w[i];
    keccak_f1600(st);
#pragma unroll
    for (int i = 0; i < 25; i++) s->w[i] = st.a[i];
    s->position = 0;
}
struct LaneSpongeUpdate { /* shake.c:89-112 */
    sponge_abi *sp; const uint8_t *in; size_t len;
    GDM void operator()(size_t) const {
        uint8_t *b = (uint8_t *)sp->w;
        const uint8_t *p = in;
        size_t left = len;
        while (left) {
            const size_t cando = (size_t)sp->rate - sp->position;
            uint8_t *state = b + sp->position;
            if (cando > left) {
                for (size_t i = 0; i < left; i++) state[i] ^= p[i];
                sp->position = (uint8_t)(sp->position + left);
                break;
            }
            for (size_t i = 0; i < cando; i++) state[i] ^= p[i];
            sponge_permute(sp);
            left -= cando;
            p += cando;
        }
    }
};
struct LaneSpongeOutput { /* shake.c:114-162; status = FAILURE when more than max_out bytes were asked of a fixed-length hash */
    sponge_abi *sp; uint8_t *out; size_t len; int32_t *status;
    GDM void operator()(size_t) const {
        int32_t ret = -1;
        if (sp->max_out != 0xFF) {
            if (sp->remaining >= len) sp->remaining = (uint8_t)(sp->remaining - len);
            else { sp->remaining = 0; ret = 0; }
        }
        uint8_t *b = (uint8_t *)sp->w;
        if (sp->flags == 'A') {
            b[sp->position] ^= sp->pad;
            b[sp->rate - 1] ^= sp->rate_pad;
            sponge_permute(sp);
            sp->flags = 'Z';
        }
        uint8_t *o = out;
        size_t left = len;
        while (left) {
            const size_t cando = (size_t)sp->rate - sp->position;
            const uint8_t *state = b + sp->position;
            if (cando > left) {
                for (size_t i = 0; i < left; i++) o[i] = state[i];
                sp->position = (uint8_t)(sp->position + left);
                break;
            }
            for (size_t i = 0; i < cando; i++) o[i] = state[i];
            sponge_permute(sp);
            left -= cando;
            o += cando;
        }
        status[0] = ret;
    }
};

// ---- EdDSA <-> X448 key conversions ----------------------------------------------------------------
struct LaneEdPkToX448 { /* goldilocks_ed448_convert_public_key_to_x448 (goldilocks.c:1079-1103): u = y^2 (1 - d y^2) / (1 - y^2) */
    uint8_t *x; const uint8_t *ed;
    GDM void operator()(size_t i) const {
        uint32_t w[15], wo[14];
        words_load_bytes(w, 15, ed + 57 * i, 57);   /* the 57th byte (sign) is not read by the reference either */
        gf y, n, d, one;
        (void)gf_from_words(y, w);
        gf_set_ui(one, 1);
        gf_sqr(n, y);
        gf_sub(d, one, n);
        gf_invert(d, d);
        gf_mul(y, n, d);
        gf_mulw_signed(d, n, GOLD_EDWARDS_D);
        gf_sub(d, one, d);
        gf_mul(n, y, d);
        gf_to_words(wo, n);
        words_store56(x + 56 * i, wo);
    }
};
struct LaneEdSkToX448 { /* goldilocks_ed448_convert_private_key_to_x448 (eddsa.c:83-95): SHAKE256(sk)[0..56) */
    uint8_t *x; const uint8_t *ed;
    GDM void operator()(size_t i) const {
        shake256_ctx h;
        shake256_init(h);
        for (int k = 0; k < 57; k++) shake256_absorb_byte(h, ed[57 * i + k]);
        shake256_finish_absorb(h);
        uint32_t w[14];
        shake256_out_words<14>(h, w);
        words_store_bytes(x + 56 * i, 56, w);
    }
};
// ---- caller-supplied fixed-base tables (goldilocks_448_precompute, goldilocks.c:757-818) -------------
// Host layout of precomputed_s: 80 niels x {a, b, c} x 8 u64 canonical radix-2^56 limbs (15 360 bytes).
struct abi_niels { abi_gf a, b, c; };
struct LanePrecompute { /* lane 5k + c builds comb c of table k */
    abi_niels *tables; const abi_pt *points; niels *scratch /* 16 per lane */;
    GDM void operator()(size_t lane) const {
        const size_t k = lane / COMB_N; const int c = (int)(lane % COMB_N);
        pt b;
        pt_from_abi(b, points + k);
        niels *mine = scratch + 16 * lane;
        build_comb(mine, b, c);
        for (int e = 0; e < 16; e++) {
            abi_niels *o = tables + (COMB_ENTRIES * k + 16 * c + e);
            gf_to_abi(&o->a, mine[e].a); gf_to_abi(&o->b, mine[e].b); gf_to_abi(&o->c, mine[e].c);
        }
    }
};
struct LaneNielsFromAbi { /* uploaded table -> device limbs */
    niels *out; const abi_niels *in;
    GDM void operator()(size_t e) const { gf_from_abi(out[e].a, &in[e].a); gf_from_abi(out[e].b, &in[e].b); gf_from_abi(out[e].c, &in[e].c); }
};

// ---- SHAKE256 one-shot ---------------------------------------------------------------------------
struct LaneShake256 {
    uint8_t *out; size_t outlen; const uint8_t *in; const size_t *off;
    GDM void operator()(size_t i) const {
        shake256_ctx h;
        shake256_init(h);
        for (size_t k = off[i]; k < off[i + 1]; k++) shake256_absorb_byte(h, in[k]);
        shake256_finish_absorb(h);
        for (size_t k = 0; k < outlen; k++) out[outlen * i + k] = shake256_squeeze_byte(h);
    }
};

// ---- EdDSA -----------------------------------------------------------------------------------------
struct CtxAt { const uint8_t *p; GDM uint8_t operator()(uint32_t k) const { return p[k]; } };

// secret scalar of a private key: SHAKE256(sk)[0..57) clamped, mod q  (eddsa.c:98-117).
// `h` is left squeezing at byte 57, so a signer can pull the 57 seed bytes straight out of it
// (eddsa.c:161-176: secret_scalar_ser and seed are the two halves of one 114-byte SHAKE output).
GD void ed448_secret_scalar(sc &secret, shake256_ctx &h, const uint8_t *sk) {
    shake256_init(h);
    for (int k = 0; k < 57; k++) shake256_absorb_byte(h, sk[k]);
    shake256_finish_absorb(h);
    uint32_t w[15];
    shake256_out_words<15>(h, w);   /* bytes 0 .. 56 of the 114-byte output; the clamp clears byte 56 and leaves 57 .. 59 out */
    w[14] &= 0xffu;
    ed448_clamp_words(w);
    sc_reduce_57(secret, w); /* folding reduction (sc.cuh): branch-free, same canonical value as scalar_decode_long */
}
struct LaneEdSecretScalar { /* goldilocks_ed448_derive_secret_scalar, eddsa.c:98-127 */
    abi_sc *out; const uint8_t *sk;
    GDM void operator()(size_t i) const {
        sc s, h1, h2; shake256_ctx hk;
        ed448_secret_scalar(s, hk, sk + 57 * i);
        sc_halve(h1, s);
        sc_halve(h2, h1);
        sc_to_abi(out + i, h2);
    }
};
// Signing is split in four launches so each keeps its own register budget and holds ONE sponge
// (nvcc 12.9 -O3 miscompiled the kernel that ran the key-expansion sponge and the nonce sponge
// back to back with the seed handed over in local memory; RFC 8032 vectors guard this on the GPU):
//   0) expand: secret scalar and seed from SHAKE256(sk)     (eddsa.c:161-171)
//   1) nonce: nonce scalar, nonce/4                          (eddsa.c:173-199)
//   2) R = encode(comb(nonce/4))                            (eddsa.c:201-205; SlotEdSignR, slot_lanes.cuh)
//   3) S = challenge * secret + nonce ; sig = R || S || 0   (eddsa.c:207-229)
struct LaneEdSignExpand { /* eddsa.c:161-171: SHAKE256(sk) -> clamped secret scalar || 57-byte seed (device scratch) */
    abi_sc *secret; uint8_t *seed; const uint8_t *sk;
    GDM void operator()(size_t i) const {
        sc s;
        shake256_ctx hk;
        ed448_secret_scalar(s, hk, sk + 57 * i);
        uint32_t w[29], sw[15];      /* seed = bytes 57 .. 113 of the same output block (eddsa.c:161-176) */
        shake256_out_words<29>(hk, w);
#pragma unroll
        for (int k = 0; k < 15; k++) sw[k] = k < 14 ? (w[14 + k] >> 8) | (w[15 + k] << 24) : (w[28] >> 8) & 0xffu;
        words_store_bytes(seed + 57 * i, 57, sw);
        sc_to_abi(secret + i, s);
    }
};
struct LaneEdSignNonce { /* eddsa.c:173-199: nonce = SHAKE256(dom || seed || msg) mod q, and nonce/4 for the comb */
    abi_sc *nonce, *nonce4; const uint8_t *seed, *msg; const size_t *off; uint32_t prehashed; const uint8_t *ctx; uint32_t ctx_len;
    GDM void operator()(size_t i) const {
        sc n, h1, h2;
        shake256_ctx h;
        CtxAt cat = {ctx};
        ed448_hash_init_with_dom(h, prehashed, cat, ctx_len);
        for (int k = 0; k < 57; k++) shake256_absorb_byte(h, seed[57 * i + k]);
        for (size_t k = off[i]; k < off[i + 1]; k++) shake256_absorb_byte(h, msg[k]);
        shake256_finish_absorb(h);
        uint32_t w[29]; /* 114 output bytes straight from the state words, reduced by folding (sc.cuh) */
        shake256_out_words<29>(h, w);
        w[28] &= 0xffffu;
        sc_reduce_114(n, w);
        sc_halve(h1, n);
        sc_halve(h2, h1);
        sc_to_abi(nonce + i, n);
        sc_to_abi(nonce4 + i, h2);
    }
};
GD void ed448_challenge(sc &c, const uint8_t *r57, const uint8_t *pk57, const uint8_t *msg, size_t lo, size_t hi,
                        uint32_t prehashed, const uint8_t *ctx, uint32_t ctx_len) {
    shake256_ctx h;
    CtxAt cat = {ctx};
    ed448_hash_init_with_dom(h, prehashed, cat, ctx_len);
    for (int k = 0; k < 57; k++) shake256_absorb_byte(h, r57[k]);
    for (int k = 0; k < 57; k++) shake256_absorb_byte(h, pk57[k]);
    for (size_t k = lo; k < hi; k++) shake256_absorb_byte(h, msg[k]);
    shake256_finish_absorb(h);
    uint32_t w[29]; /* 114 output bytes straight from the state words, reduced by folding (sc.cuh) */
    shake256_out_words<29>(h, w);
    w[28] &= 0xffffu;
    sc_reduce_114(c, w);
}
struct LaneEdSignFinish {
    uint8_t *sig; const abi_sc *secret, *nonce; const uint8_t *pk, *msg; const size_t *off; uint32_t prehashed; const uint8_t *ctx; uint32_t ctx_len;
    GDM void operator()(size_t i) const {
        sc c, s, n, t, r;
        ed448_challenge(c, sig + 114 * i, pk + 57 * i, msg, off[i], off[i + 1], prehashed, ctx, ctx_len);
        sc_from_abi(s, secret + i);
        sc_from_abi(n, nonce + i);
        sc_mul(t, c, s);
        sc_add(r, t, n);
        uint32_t w[15];
        for (int k = 0; k < 14; k++) w[k] = r.w[k];
        w[14] = 0;
        words_store_bytes(sig + 114 * i + 57, 57, w);
    }
};
// Verification is three launches (eddsa.c:253-306):
//   1) decode A and R (2n lanes, one isr each)            -> points + ok flags
//   2) challenge = -SHAKE256(dom || R || A || M) mod q, response = S mod q
//   3) combo = response*B + challenge*A ; accept iff combo == R (mod 2-torsion) and both decodes succeeded
//      (SlotEdVerifyFinish, slot_lanes.cuh)
struct LaneEdVerifyDecode {
    /* Without a plan: lane 2i = public key i, lane 2i+1 = R of signature i.  With the plan of a grouped batch
     * (verify_plan.cuh) only public keys are decoded, once per key, by the lanes from n on: the keys of the stand-alone
     * signatures, then one representative per key table; the remaining lanes retire at once.  R is not decoded for signatures
     * under a key table (slot_lanes.cuh s_verify_accept_prep); the lanes from 2n on decode the R of the stand-alone ones.
     * The result lands in pts[2i] (key of signature i) / pts[2i+1] (its R). */
    abi_pt *pts; int32_t *ok; const uint8_t *sig, *pk; size_t n; verify_plan plan; size_t lane0; /* first lane of this launch */
    GDM void operator()(size_t j0) const {
        const size_t j = j0 + lane0;
        size_t i = j >> 1, which = j & 1;
        if (plan.unique_sig) {
            if (j < n) return;
            {
                const size_t k = j - n, nu = plan.counts[1];
                which = 0;
                if (k >= n) {                                   /* lanes from 2n on: R of the stand-alone signatures (half-size path) */
                    if (k - n >= nu) return;
                    i = plan.unique_sig[k - n];
                    which = 1;
                } else if (k < nu) i = plan.unique_sig[k];
                else if (k - nu < plan.counts[2]) i = plan.tab_rep[k - nu];
                else return;
            }
        }
        const uint8_t *enc = which ? sig + 114 * i : pk + 57 * i;
        pt p; uint32_t w[15];
        words_load_bytes(w, 15, enc, 57);
        gmask_t good = pt_decode_like_eddsa(p, w, w[14] & 0xff);
        /* the third launch only needs TIGHT limbs back, so store weakly reduced (not canonical) limbs */
        abi_pt *o = pts + 2 * i + which;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            o->x.limb[k] = (uint64_t)p.x.v[2 * k] + ((uint64_t)p.x.v[2 * k + 1] << 28);
            o->y.limb[k] = (uint64_t)p.y.v[2 * k] + ((uint64_t)p.y.v[2 * k + 1] << 28);
            o->z.limb[k] = (uint64_t)p.z.v[2 * k] + ((uint64_t)p.z.v[2 * k + 1] << 28);
            o->t.limb[k] = (uint64_t)p.t.v[2 * k] + ((uint64_t)p.t.v[2 * k + 1] << 28);
        }
        ok[2 * i + which] = ST_OK(good);
    }
};
struct LaneEdVerifyScalars {
    abi_sc *challenge, *response; const uint8_t *sig, *pk, *msg; const size_t *off; uint32_t prehashed; const uint8_t *ctx; uint32_t ctx_len; size_t i0;
    const uint32_t *key_index; uint32_t n_keys; /* key set calls: the key of signature i is pk[key_index[i]] (out of range: key 0, rejected later) */
    GDM void operator()(size_t k) const {
        const size_t i = k + i0;
        size_t ki = i;
        if (key_index) { ki = key_index[i]; if (ki >= n_keys) ki = 0; }
        sc c, nc, r;
        ed448_challenge(c, sig + 114 * i, pk + 57 * ki, msg, off[i], off[i + 1], prehashed, ctx, ctx_len);
        sc_neg(nc, c);
        uint32_t sw[15];
        words_load_bytes(sw, 15, sig + 114 * i + 57, 57);
        sc_reduce_57(r, sw);         /* reduces mod q, no range check (eddsa.c:287-291) */
        /* GOLDILOCKS_448_EDDSA_DECODE_RATIO = 1: no doubling of the response */
        sc_to_abi(challenge + i, nc);
        sc_to_abi(response + i, r);
    }
};
// Stand-alone signatures (no key table to share) are verified with half-size multipliers (sc.cuh sc_half_gcd, slot_algos.cuh
// s_verify_half).  One lane per such signature, after LaneEdVerifyScalars: from the challenge c and the response s it leaves
//     challenge[i] <- u in words 0..6, |v| in words 7..13, the sign of v in bit 31 of word 13   (v c == u mod q)
//     response[i]  <- sB = v s mod q
// c = 0 keeps the reference's quirk (goldilocks.c:1281-1284: the combination is the identity whatever s is): u = 0, v = 1, sB = 0.
struct LaneVerifyHalf {
    abi_sc *challenge, *response; verify_plan plan;
    GDM void operator()(size_t j) const {
        size_t i = j;
        if (plan.unique_sig) {
            if (j >= plan.counts[1]) return;
            i = plan.unique_sig[j];
        }
        sc c, r, u, v, sB, packed;
        sc_from_abi(c, challenge + i);
        sc_from_abi(r, response + i);
        const gmask_t v_neg = sc_half_gcd(u, v, c);
        sc_mul(sB, v, r);
        if (v_neg) sc_neg(sB, sB);
        uint32_t any = 0;
#pragma unroll
        for (int k = 0; k < SC_WORDS; k++) any |= c.w[k];
        if (!any) sc_set_zero(sB);
#pragma unroll
        for (int k = 0; k < 7; k++) { packed.w[k] = u.w[k]; packed.w[7 + k] = v.w[k]; }
        packed.w[13] |= v_neg & 0x80000000u;
        sc_to_abi(challenge + i, packed);
        sc_to_abi(response + i, sB);
    }
};
// What the finish kernels leave per signature for the last step (slot_lanes.cuh s_verify_accept_prep): G D, H and flags.
// 256 bytes, so that the grouped path can keep it in the unused R half of its point array.
#define VAUX_FAST 1u  /* every other condition holds: accept iff lobit(H / (G D)) == sign bit */
#define VAUX_SLOW 2u  /* degenerate case already decided: accept */
#define VAUX_LOW  4u  /* the sign bit of the encoding */
struct verify_aux { abi_gf gd, h, prefix; uint32_t flags; uint32_t pad[15]; };
// Sign check of the square-root-free R comparison, VSIGN_BATCH signatures per lane and inversion (Montgomery's trick:
// prefix products out, one inversion, back-substitution).  aux record of signature i = aux[i * stride].
#define VSIGN_BATCH 16
struct LaneVerifySign {
    int32_t *status; verify_aux *aux; size_t stride, n;
    GDM void operator()(size_t l) const {
        const size_t lo = l * VSIGN_BATCH, hi = lo + VSIGN_BATCH < n ? lo + VSIGN_BATCH : n;
        gf acc, v, t;
        gf_set_ui(acc, 1);
        for (size_t i = lo; i < hi; i++) {
            verify_aux *a = aux + i * stride;
            gf_from_abi(v, &a->gd);
            gf_mul(acc, acc, v);
#pragma unroll
            for (int k = 0; k < 8; k++) a->prefix.limb[k] = (uint64_t)acc.v[2 * k] + ((uint64_t)acc.v[2 * k + 1] << 28);
        }
        gf inv;
        gf_invert(inv, acc);
        for (size_t i = hi; i-- > lo;) {
            verify_aux *a = aux + i * stride;
            if (i > lo) { gf_from_abi(t, &aux[(i - 1) * stride].prefix); gf_mul(t, inv, t); } /* 1 / (G D)_i */
            else gf_copy(t, inv);
            gf_from_abi(v, &a->gd);
            gf_mul(inv, inv, v);
            gf_from_abi(v, &a->h);
            gf_mul(t, t, v);                                  /* x = H / (G D) */
            const uint32_t f = a->flags;
            const uint32_t sign_ok = ((gf_lobit(t) & 1u) == ((f & VAUX_LOW) ? 1u : 0u)) ? 1u : 0u;
            status[i] = (((f & VAUX_FAST) && sign_ok) || (f & VAUX_SLOW)) ? -1 : 0;
        }
    }
};
// ---- set lookup by bytes (goldilocks_ed448_verify_keyset_lookup_batch, DESIGN.md decision 23; goldilocks_x448_peerset_lookup_batch,
// decision 24).  Public data only, variable time.
template <int W>
GD int key_cmp(const uint8_t *a, const uint8_t *b) { /* memcmp order of two W-byte keys */
    for (int k = 0; k < W; k++)
        if (a[k] != b[k]) return a[k] < b[k] ? -1 : 1;
    return 0;
}
// Lane j: key_index[j] = the lowest index of the set whose W bytes equal key j, or m.  `sorted` holds the set's indices ordered by
// key bytes, ties by index (made on the host at creation), so the lower bound of key j in it is its lowest equal index.  A byte
// order rather than a hash order: ceil(log2 m) + 1 comparisons whatever keys the set holds.
template <int W>
struct LaneSetLookup {
    uint32_t *key_index; const uint8_t *pk, *set_pk; const uint32_t *sorted; uint32_t m;
    GDM void operator()(size_t j) const {
        const uint8_t *q = pk + W * j;
        uint32_t lo = 0, hi = m;
        while (lo < hi) {
            const uint32_t mid = lo + (hi - lo) / 2;
            if (key_cmp<W>(set_pk + W * (size_t)sorted[mid], q) < 0) lo = mid + 1;
            else hi = mid;
        }
        key_index[j] = (lo < m && key_cmp<W>(set_pk + W * (size_t)sorted[lo], q) == 0) ? sorted[lo] : m;
    }
};
using LaneKeysetLookup = LaneSetLookup<57>;    /* Ed448 public keys of a key set */
using LaneX448PeerLookup = LaneSetLookup<56>;  /* u-coordinates of an X448 peer set */
// *hits = the number of sort keys below m (keys_s: the looked-up indices, clamped to m and sorted; LaneDecafPeerKeys).  One lane
// writes: the first miss, or the last lane when there is none.
struct LaneKeysetHits {
    uint32_t *hits; const uint32_t *keys_s; uint32_t m; size_t n;
    GDM void operator()(size_t j) const {
        const bool miss = keys_s[j] >= m;
        if (miss && (j == 0 || keys_s[j - 1] < m)) *hits = (uint32_t)j;
        if (!miss && j + 1 == n) *hits = (uint32_t)n;
    }
};
// The misses (elements order[hits + q], q < misses) packed for goldilocks_ed448_verify_batch's path: their message lengths (lane
// `misses` writes 0, so an exclusive scan over misses + 1 entries gives the new offsets and the total) ...
struct LaneKeysetMissLengths {
    size_t *len; const size_t *off; const uint32_t *order; size_t hits, misses;
    GDM void operator()(size_t q) const {
        if (q >= misses) { len[q] = 0; return; }
        const size_t i = order[hits + q];
        len[q] = off[i + 1] - off[i];
    }
};
// ... then their signatures, keys and messages
struct LaneKeysetMissGather {
    uint8_t *sig2, *pk2, *msg2; const size_t *off2; const uint8_t *sig, *pk, *msg; const size_t *off; const uint32_t *order; size_t hits;
    GDM void operator()(size_t q) const {
        const size_t i = order[hits + q];
        for (int k = 0; k < 114; k++) sig2[114 * q + k] = sig[114 * i + k];
        for (int k = 0; k < 57; k++) pk2[57 * q + k] = pk[57 * i + k];
        const size_t lo = off[i], len = off[i + 1] - lo;
        uint8_t *d = msg2 + off2[q];
        for (size_t k = 0; k < len; k++) d[k] = msg[lo + k];
    }
};
// status[order[j]] = st_sorted[j]: the hits' statuses (j < hits) and the misses' (j >= hits) back to the caller's positions
struct LaneKeysetScatter {
    int32_t *status; const int32_t *st_sorted; const uint32_t *order;
    GDM void operator()(size_t j) const { status[order[j]] = st_sorted[j]; }
};
struct LaneBuildWide { /* verification table, WIDE_LANES lanes */
    niels *wide; pniels *tmp; gf *pre; const fixed_tables *ft;
    GDM void operator()(size_t lane) const { build_wide_lane(wide, tmp, pre, ft->comb, (int)lane); }
};
struct LaneBuildTables {
    fixed_tables *ft;
    GDM void operator()(size_t lane) const { build_tables_lane(ft, (int)lane); }
};
