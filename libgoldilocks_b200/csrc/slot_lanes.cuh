// slot_lanes.cuh -- functors of the slot-machine kernels (slots.cuh): `operator()(i, base)` processes
// element i with this lane's shared-memory slots starting at handle `base`.
#pragma once
#include <type_traits>
#include "lanes.cuh"
#include "slot_algos.cuh"
#include "verify_plan.cuh"

struct SlotX448 { /* goldilocks_x448 (goldilocks.c:1006-1076) */
    static constexpr int NSLOTS = X448_NSLOTS;
    uint8_t *out; int32_t *status; const uint8_t *base, *scalar;
    GDM void operator()(size_t i, sref sb, bool live) const {
        uint32_t wb[14], ws[14], wo[14];
        words_load56(wb, base + 56 * i);
        words_load56(ws, scalar + 56 * i);
        gmask_t nz = x448_ladder_slots(wo, wb, ws, sb);
        if (!live) return;
        words_store56(out + 56 * i, wo);
        status[i] = ST_OK(nz);
    }
};

GD void s_pt_from_abi(sref sb, const abi_pt *a) { /* slots 0..3 = X, Y, Z, T */
    gf v;
    gf_from_abi(v, &a->x); s_st(s_slot(sb, 0), v);
    gf_from_abi(v, &a->y); s_st(s_slot(sb, 1), v);
    gf_from_abi(v, &a->z); s_st(s_slot(sb, 2), v);
    gf_from_abi(v, &a->t); s_st(s_slot(sb, 3), v);
}
// Reference quirk kept for bit-exact parity: when scalar2 == 0 its wNAF is empty and
// goldilocks.c:1281-1284 returns the identity WITHOUT adding scalar1*B.
GD void s_bdsm_quirk(sref sb, const sc &scalar2) {
    uint32_t any2 = 0;
#pragma unroll
    for (int k = 0; k < SC_WORDS; k++) any2 |= scalar2.w[k];
    const gmask_t z2 = (gmask_t)(((uint64_t)any2 - 1) >> 32);
    gf v, zero, one;
    gf_set_zero(zero);
    gf_set_ui(one, 1);
    s_ld(v, s_slot(sb, 0)); gf_cond_sel(v, v, zero, z2); s_st(s_slot(sb, 0), v);
    s_ld(v, s_slot(sb, 1)); gf_cond_sel(v, v, one, z2); s_st(s_slot(sb, 1), v);
    s_ld(v, s_slot(sb, 2)); gf_cond_sel(v, v, one, z2); s_st(s_slot(sb, 2), v);
    s_ld(v, s_slot(sb, 3)); gf_cond_sel(v, v, zero, z2); s_st(s_slot(sb, 3), v);
}
struct SlotBaseDoubleScalarmul { /* goldilocks_448_base_double_scalarmul_non_secret (goldilocks.c:1260-1330) */
    static constexpr int NSLOTS = BDSM_NSLOTS;
    abi_pt *out; const abi_sc *scalar1; const abi_pt *base2; const abi_sc *scalar2; const niels *wide; uint4 *scratch;
    GDM void operator()(size_t i, sref sb, size_t slot) const {
        sc s1, s2;
        sc_from_abi(s1, scalar1 + i); sc_from_abi(s2, scalar2 + i);
        s_pt_from_abi(sb, base2 + i);
        s_base_double_scalarmul(sb, s1, s2, wide, wtab_of<1>(scratch, slot));
        s_bdsm_quirk(sb, s2);
        gf v;
        s_ld(v, s_slot(sb, 0)); gf_to_abi(&out[i].x, v);
        s_ld(v, s_slot(sb, 1)); gf_to_abi(&out[i].y, v);
        s_ld(v, s_slot(sb, 2)); gf_to_abi(&out[i].z, v);
        s_ld(v, s_slot(sb, 3)); gf_to_abi(&out[i].t, v);
    }
};
// Verification under a repeated key (eddsa.c:293-305): combo = response*B + challenge*A from the key's tables, accept iff
// combo == R on the quotient group (goldilocks.c:644-653) and both decodes succeeded --
// that accept bit WITHOUT the square root of the R decode (goldilocks.c:949-1004 needs isr(N D), 446 squarings).
// With y = the encoded coordinate of R, N = 1 - y^2, D = 1 - d y^2 (never 0: d is a non-square), the reference decodes
// x = +-sqrt(N/D) with lobit(x) = the sign bit, maps (x, y) through the 4-isogeny to (X_R : Y_R) and accepts iff
// Y_c X_R == Y_R X_c.  Multiplied by D^2 that equation is linear in W = x D (W^2 = N D):
//     G W == H,   G = 2 y (2D - N - y^2 D) Y_c,   H = (y^2 D - N)(N + y^2 D) X_c.
// If G != 0 the reference accepts iff N D != 0, H^2 == G^2 N D (then N D is a square and W = +-H/G) and
// lobit(H / (G D)) == sign bit (W = H/G picks the root the decoder picks; the two roots have different low bits).
// That needs one INVERSION, not a square root, and inversions batch (Montgomery's trick): this step leaves G D, H and
// the flags in the signature's `aux` record and LaneVerifySign (lanes.cuh) finishes 16 signatures per inversion.
// If G == 0 (y = 0, Y_c = 0, ... : never on honest data) the lane takes the reference's own route here and now:
// accept iff N D is a non-zero square (s_isr) and H == 0.  The other decode conditions (y < p, low seven bits of the
// last byte clear) are checked as the reference checks them.
// On entry slots 0, 1 hold X_c, Y_c; all seven slots are clobbered.
SFN void s_verify_accept_prep(verify_aux *aux, sref sb, const uint8_t *r_enc, gmask_t key_ok) {
    const sref s0 = s_slot(sb, 0), s1 = s_slot(sb, 1), s2 = s_slot(sb, 2), s3 = s_slot(sb, 3), s4 = s_slot(sb, 4), s5 = s_slot(sb, 5), s6 = s_slot(sb, 6);
    gf a, b, one, N, D, E;
    uint32_t w[15];
    gf_set_ui(one, 1);
    words_load_bytes(w, 15, r_enc, 57);
    gmask_t good = gf_from_words(a, w);                      /* y < p (f_generic.c:48-68) */
    good &= ((w[14] & 0x7f) == 0) ? ~0u : 0u;                /* goldilocks.c:965 */
    good &= key_ok;
    const uint32_t low = (w[14] >> 7) & 1u;
    s_st(s2, a);                                             /* y */
    s_sqr(s3, s2);                                           /* y^2 */
    s_ld(b, s3);
    gf_sub(N, one, b);
    gf_mulw_signed(a, b, GOLD_EDWARDS_D);
    gf_sub(D, one, a);
    s_st(s4, N); s_st(s5, D);
    s_mul(s6, s3, s5);                                       /* E = y^2 D */
    s_ld(E, s6); s_ld(N, s4); s_ld(D, s5);
    gf_add(a, D, D); gf_sub(a, a, N); gf_sub(a, a, E);       /* 2D - N - E */
    s_st(s3, a);
    s_mul(s3, s2, s3);
    s_mul(s3, s3, s1);                                       /* y (2D - N - E) Y_c = G / 2 */
    s_ld(N, s4); s_ld(E, s6);
    gf_sub(a, E, N); s_st(s1, a);
    gf_add(a, N, E); s_st(s2, a);
    s_mul(s6, s1, s2);
    s_mul(s6, s6, s0);                                       /* H */
    s_mul(s4, s4, s5);                                       /* N D */
    s_ld(a, s3); gf_add(a, a, a); s_st(s3, a);               /* G */
    s_sqr(s0, s6);
    s_sqr(s2, s3);
    s_mul(s2, s2, s4);
    s_ld(a, s0); s_ld(b, s2);
    gmask_t fast = gf_eq(a, b);                              /* H^2 == G^2 N D */
    s_ld(a, s4);
    fast &= ~gf_is_zero(a);                                  /* N D != 0 (y = +-1 is rejected: isr(0) fails, goldilocks.c:974) */
    s_ld(a, s3);
    const gmask_t g_zero = gf_is_zero(a);
    fast &= ~g_zero;
    gmask_t slow = 0;
    if (g_zero) {                                            /* degenerate: the reference's own route */
        const gmask_t square = s_isr(s0, s2, s4);
        s_ld(a, s6);
        slow = square & gf_is_zero(a);
    }
    s_mul(s5, s3, s5);                                       /* G D (1 where it is 0: it only feeds the batched inversion) */
    s_ld(a, s5);
    gf_cond_sel(a, a, one, g_zero);
    s_ld(b, s6);
#pragma unroll
    for (int k = 0; k < 8; k++) {                            /* weakly reduced limbs: the next kernel only multiplies them */
        aux->gd.limb[k] = (uint64_t)a.v[2 * k] + ((uint64_t)a.v[2 * k + 1] << 28);
        aux->h.limb[k] = (uint64_t)b.v[2 * k] + ((uint64_t)b.v[2 * k + 1] << 28);
    }
    aux->flags = ((good & fast) ? VAUX_FAST : 0u) | ((good & slow) ? VAUX_SLOW : 0u) | (low ? VAUX_LOW : 0u);
}
// A stand-alone signature with half-size multipliers (slot_algos.cuh s_verify_half): key2[0], key2[1] = the decoded public key and R,
// *challenge / *response as LaneVerifyHalf (lanes.cuh) left them; two window tables per lane in `scratch`.  All-ones iff
// response B + challenge A == R on the quotient group (eddsa.c:293-305, goldilocks.c:644-653): the combination's x is 0.
GD gmask_t s_verify_half_item(sref sb, const abi_pt *key2, const abi_sc *challenge, const abi_sc *response, const niels *wide, uint4 *scratch, size_t slot) {
    const spt p = {s_slot(sb, 0), s_slot(sb, 1), s_slot(sb, 2), s_slot(sb, 3)};
    const swk w = {s_slot(sb, 4), s_slot(sb, 5), s_slot(sb, 6)};
    sc packed, sB, u, v;
    sc_from_abi(packed, challenge);
    sc_from_abi(sB, response);
    sc_set_zero(u);
    sc_set_zero(v);
#pragma unroll
    for (int k = 0; k < 7; k++) { u.w[k] = packed.w[k]; v.w[k] = packed.w[7 + k]; }
    const gmask_t v_neg = (gmask_t)0 - (v.w[6] >> 31);
    v.w[6] &= 0x7fffffffu;
    sc_half_bias(u, u);
    sc_half_bias(v, v);
    const wtab<1> ta = wtab_of<1>(scratch, 2 * slot), tr = wtab_of<1>(scratch, 2 * slot + 1);
    s_pt_from_abi(sb, key2);
    s_prepare_signed_window<1>(p, w, ta);
    s_pt_from_abi(sb, key2 + 1);
    s_prepare_signed_window<1>(p, w, tr);
    s_verify_half(sb, sB, u, v, v_neg, wide, ta, tr);
    gf x;
    s_ld(x, p.x);
    return gf_is_zero(x);
}
struct SlotEdVerifyFinish {
    static constexpr int NSLOTS = BDSM_NSLOTS;
    int32_t *status; const abi_pt *pts; const int32_t *ok; const abi_sc *challenge, *response; const niels *wide; uint4 *scratch;
    GDM void operator()(size_t i, sref sb, size_t slot) const {
        const gmask_t eq = s_verify_half_item(sb, pts + 2 * i, challenge + i, response + i, wide, scratch, slot);
        status[i] = ST_OK(eq & (gmask_t)ok[2 * i] & (gmask_t)ok[2 * i + 1]);
    }
};
// The per-key tables of a batch, in two launches (slot_algos.cuh s_key_column_bases / s_build_key_column): one lane per key walks the doubling
// chain, then one lane per (key, column) -- work item chunks * t + c -- fills a column.  The column shape (10 x 9 or 15 x 6) comes from
// the plan's counts (vsh_pick, slot_algos.cuh).
struct SlotKeyChain {
    static constexpr int NSLOTS = BDSM_NSLOTS;
    const abi_pt *pts; uint4 *ktabs; verify_plan plan;
    GDM void operator()(size_t t, sref sb, size_t slot) const {
        (void)slot;
        if (t >= plan.counts[2]) return;
        const vsh_shape sh = vsh_pick(plan.counts);
        s_pt_from_abi(sb, pts + 2 * (size_t)plan.tab_rep[t]);
        s_key_column_bases(sb, ktab_of(ktabs, t, sh.quads), sh.chunks, sh.rows * WINDOW_BITS);
    }
};
struct SlotKeyColumns {
    static constexpr int NSLOTS = BDSM_NSLOTS;
    uint4 *ktabs; uint4 *scratch; verify_plan plan;
    GDM void operator()(size_t item, sref sb, size_t slot) const {
        const vsh_shape sh = vsh_pick(plan.counts);
        const size_t t = item / (size_t)sh.chunks;
        if (t >= plan.counts[2]) return;
        s_build_key_column(sb, ktab_of(ktabs, t, sh.quads), (int)(item % (size_t)sh.chunks), wtab_of<1>(scratch, slot));
    }
};
// The finish kernel of a grouped batch.  Work items [0, counts[1]) are the stand-alone signatures, verified exactly like
// SlotEdVerifyFinish (own window table in `scratch`); items [counts[1], counts[1] + counts[0]) are signatures whose
// public key (byte-identical) occurs more than once: the multiples of the key come from the table its group built.
// One launch for both; the expensive stand-alone items go first and the items are handed out dynamically
// (k_slots_persist, slots.cuh), so the cheap ones fill in behind them.  The shared items never decode R: s_verify_accept_prep
// works from its bytes and leaves the sign check to LaneVerifySign; the stand-alone items (half-size multipliers, R decoded by
// LaneVerifyHalf) leave their verdict in the same record.
struct SlotEdVerifyFinishShared {
    static constexpr int NSLOTS = BDSM_NSLOTS;
    abi_pt *pts; const int32_t *ok; const abi_sc *challenge, *response; const niels *wide; uint4 *ktabs; uint4 *scratch;
    verify_plan plan; const uint8_t *sig;
    GDM void operator()(size_t j, sref sb, size_t slot) const {
        const size_t nu = plan.counts[1];
        size_t i;
        gmask_t key_ok;
        sc c, r;
        if (j >= nu) {
            if (j - nu >= plan.counts[0]) return;
            const size_t t = plan.shared_tab[j - nu];
            i = plan.shared_sig[j - nu];
            sc_from_abi(c, challenge + i);
            sc_from_abi(r, response + i);
            const vsh_shape sh = vsh_pick(plan.counts);
            s_verify_shared_key(sb, r, c, wide, ktab_of(ktabs, t, sh.quads), sh.rows, sh.chunks);
            key_ok = (gmask_t)ok[2 * (size_t)plan.tab_rep[t]]; /* the key bytes are the representative's, so is the decode flag */
        } else {
            i = plan.unique_sig[j];
            const gmask_t eq = s_verify_half_item(sb, pts + 2 * i, challenge + i, response + i, wide, scratch, slot);
            verify_aux *aux = (verify_aux *)(pts + 2 * i + 1);   /* the decoded R has been consumed */
            const abi_gf one = {{1, 0, 0, 0, 0, 0, 0, 0}};
            aux->gd = one; aux->h = one;
            aux->flags = (eq & (gmask_t)ok[2 * i] & (gmask_t)ok[2 * i + 1]) ? VAUX_SLOW : 0u;
            return;
        }
        s_bdsm_quirk(sb, c);
        s_verify_accept_prep((verify_aux *)(pts + 2 * i + 1), sb, sig + 114 * i, key_ok); /* the R slot of pts is free: R is never decoded */
    }
};

// Key sets (include/goldilocks_b200.h, goldilocks_b200_keyset_*): the same per-key tables, built once by
// goldilocks_b200_keyset_create and kept in HBM across calls (SURVEY 8(f)4).
struct SlotKeysetTables { /* one lane per key: decoded key t -> table t */
    static constexpr int NSLOTS = BDSM_NSLOTS;
    const abi_pt *pts; uint4 *ktabs;
    GDM void operator()(size_t t, sref sb, size_t slot) const {
        (void)slot;
        s_pt_from_abi(sb, pts + t);
        s_build_key_tables(sb, ktab_of(ktabs, t));
    }
};
// A key set's tables serve many calls, so their entries are made affine once: niels = pniels.n / pniels.z (goldilocks.c:280-288 has
// z = 2Z; the reference normalises its fixed-base tables the same way, precompute in goldilocks.c:765-815).  One lane per (key, column):
// Montgomery's trick over the column's 16 entries, one inversion.  Every addition under the key then costs 7 multiplications, not 8.
struct LaneKeysetNormalize {
    uint4 *ktabs; uint32_t ncols, quads_per_key;       /* 10 columns of KTAB_QUADS, or the flat layout's 90 of KSET_QUADS */
    GDM void operator()(size_t item) const {
        wtab<1> kt;
        kt.base = ktabs + (item / ncols) * (size_t)quads_per_key;
        const int e0 = (int)(item % ncols) * WINDOW_NTABLE;
        gf pre[WINDOW_NTABLE], acc, z, zi, x;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (int e = 0; e < WINDOW_NTABLE; e++) {
            gq_ld<false, 1>(z, kt.coord(e0 + e, 3));
            if (e == 0) gf_copy(acc, z);
            else gf_mul(acc, acc, z);
            gf_copy(pre[e], acc);
        }
        gf_invert(acc, acc);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (int e = WINDOW_NTABLE - 1; e >= 0; e--) {
            if (e > 0) gf_mul(zi, acc, pre[e - 1]);          /* 1 / z_e */
            else gf_copy(zi, acc);
            gq_ld<false, 1>(z, kt.coord(e0 + e, 3));
            gf_mul(acc, acc, z);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
            for (int j = 0; j < 3; j++) {
                gq_ld<false, 1>(x, kt.coord(e0 + e, j));
                gf_mul(x, x, zi);
                gq_st<1>(kt.coord(e0 + e, j), x);
            }
        }
    }
};
// The flat layout of a key set (slot_algos.cuh s_verify_flat_key): chain of 89 x 5 doublings per key, one lane per (key, digit position)
// for the 90 column tables, then the same normalisation.
struct SlotKeysetChain {
    static constexpr int NSLOTS = BDSM_NSLOTS;
    const abi_pt *pts; uint4 *ktabs;
    GDM void operator()(size_t t, sref sb, size_t slot) const {
        (void)slot;
        s_pt_from_abi(sb, pts + t);
        s_key_column_bases(sb, kset_of(ktabs, t), KSET_COLS, WINDOW_BITS);
    }
};
struct SlotKeysetColumns {
    static constexpr int NSLOTS = BDSM_NSLOTS;
    uint4 *ktabs; uint4 *scratch;
    GDM void operator()(size_t item, sref sb, size_t slot) const {
        s_build_key_column(sb, kset_of(ktabs, item / KSET_COLS), (int)(item % KSET_COLS), wtab_of<1>(scratch, slot));
    }
};
struct SlotEdVerifyFinishKeysetFlat { /* signature i under key key_index[i] of a flat-layout set: no doublings */
    static constexpr int NSLOTS = BDSM_NSLOTS;
    verify_aux *aux; const int32_t *key_ok; const abi_sc *challenge, *response; const niels *wide; const uint4 *ktabs;
    const uint32_t *key_index; uint32_t n_keys; const uint8_t *sig;
    GDM void operator()(size_t i, sref sb, size_t slot) const {
        (void)slot;
        const uint32_t t = key_index[i];
        if (t >= n_keys) { /* no such key: FAILURE */
            abi_gf one = {{1, 0, 0, 0, 0, 0, 0, 0}};
            aux[i].gd = one; aux[i].h = one; aux[i].flags = 0;
            return;
        }
        sc c, r;
        sc_from_abi(c, challenge + i);
        sc_from_abi(r, response + i);
        s_verify_flat_key(sb, r, c, wide, kset_of(const_cast<uint4 *>(ktabs), t));
        s_bdsm_quirk(sb, c);
        s_verify_accept_prep(aux + i, sb, sig + 114 * i, (gmask_t)key_ok[t]);
    }
};
struct SlotEdVerifyFinishKeyset { /* signature i under key key_index[i] of the set */
    static constexpr int NSLOTS = BDSM_NSLOTS;
    verify_aux *aux; const int32_t *key_ok; const abi_sc *challenge, *response; const niels *wide; const uint4 *ktabs;
    const uint32_t *key_index; uint32_t n_keys; const uint8_t *sig;
    GDM void operator()(size_t i, sref sb, size_t slot) const {
        (void)slot;
        const uint32_t t = key_index[i];
        if (t >= n_keys) { /* no such key: FAILURE */
            abi_gf one = {{1, 0, 0, 0, 0, 0, 0, 0}};
            aux[i].gd = one; aux[i].h = one; aux[i].flags = 0;
            return;
        }
        sc c, r;
        sc_from_abi(c, challenge + i);
        sc_from_abi(r, response + i);
        s_verify_shared_key<true>(sb, r, c, wide, ktab_of(const_cast<uint4 *>(ktabs), t));   /* affine entries */
        s_bdsm_quirk(sb, c);
        s_verify_accept_prep(aux + i, sb, sig + 114 * i, (gmask_t)key_ok[t]);
    }
};
/* the finish kernel of a set's layout, for host code that picks it with one flag (both keep their own kernel names) */
template <bool FLAT>
using SlotEdVerifyFinishKeysetLayout = std::conditional_t<FLAT, SlotEdVerifyFinishKeysetFlat, SlotEdVerifyFinishKeyset>;
// Key-set lookup calls (goldilocks_ed448_verify_keyset_lookup_batch; DESIGN.md decision 23): lane j < hits verifies element
// i = order[j] (the batch sorted by looked-up key, so the lanes of a warp read one or two tables) under key key_index[i] < m of a
// set of either layout, with the evaluations of the two kernels above, and leaves its aux record at aux[j].
template <bool FLAT>
struct SlotEdVerifyFinishKeysetOrdered {
    static constexpr int NSLOTS = BDSM_NSLOTS;
    verify_aux *aux; const int32_t *key_ok; const abi_sc *challenge, *response; const niels *wide; const uint4 *ktabs;
    const uint32_t *key_index, *order; const uint8_t *sig;
    GDM void operator()(size_t j, sref sb, size_t slot) const {
        (void)slot;
        const size_t i = order[j];
        const uint32_t t = key_index[i];
        sc c, r;
        sc_from_abi(c, challenge + i);
        sc_from_abi(r, response + i);
        if (FLAT) s_verify_flat_key(sb, r, c, wide, kset_of(const_cast<uint4 *>(ktabs), t));
        else s_verify_shared_key<true>(sb, r, c, wide, ktab_of(const_cast<uint4 *>(ktabs), t));   /* affine entries */
        s_bdsm_quirk(sb, c);
        s_verify_accept_prep(aux + j, sb, sig + 114 * i, (gmask_t)key_ok[t]);
    }
};

GD void s_pt_to_abi(abi_pt *o, sref sb) { /* slots 0..3 -> canonical host limbs */
    gf v;
    s_ld(v, s_slot(sb, 0)); gf_to_abi(&o->x, v);
    s_ld(v, s_slot(sb, 1)); gf_to_abi(&o->y, v);
    s_ld(v, s_slot(sb, 2)); gf_to_abi(&o->z, v);
    s_ld(v, s_slot(sb, 3)); gf_to_abi(&o->t, v);
}
struct SlotComb { /* goldilocks_448_precomputed_scalarmul (goldilocks.c:830-877) */
    static constexpr int NSLOTS = COMB_NSLOTS;
    abi_pt *out; const abi_sc *scalar; const fixed_tables *ft;
    GDM void operator()(size_t i, sref sb, bool live) const {
        sc s;
        sc_from_abi(s, scalar + i);
        s_comb_scalarmul(sb, ft->win, s);
        if (live) s_pt_to_abi(out + i, sb);
    }
};

struct SlotX448DerivePk { /* goldilocks.c:1117-1141 */
    static constexpr int NSLOTS = COMB_NSLOTS;
    uint8_t *out; const uint8_t *scalar; const fixed_tables *ft;
    GDM void operator()(size_t i, sref sb, bool live) const {
        uint32_t ws[14], wo[14];
        words_load56(ws, scalar + 56 * i);
        ws[0] &= ~3u;
        ws[13] |= 0x80000000u; /* X_PRIVATE_BITS = 448: top byte keeps all its bits, bit 447 is set */
        sc s, h;
        ByteAtWords at = {ws};
        sc_decode_long(s, at, 56);
        sc_halve(h, s);        /* GOLDILOCKS_X448_ENCODE_RATIO = 2 */
        s_comb_scalarmul(sb, ft->win, h);
        s_encode_like_x448(wo, sb);
        if (live) words_store56(out + 56 * i, wo);
    }
};
// X448 peer sets (include/goldilocks_b200.h, goldilocks_b200_x448_peerset_*; DESIGN.md decision 20).  A recurring public u gets
// the reference's (5,5,18) comb table (LanePrecompute) of an Edwards point Q with X448(u, k) = encode_like_x448((k / 8) Q):
// 17 doublings and 90 additions instead of 448 ladder steps.  The dual of RFC 7748's 4-isogeny sends (u, v) on curve448 to
// edwards448 with a y that depends on u alone,
//     y = -(u^5 - 2u^3 - 4u v^2 + u) / (u^5 - 2u^2 v^2 - 2u^3 - 2v^2 + u),   v^2 = u^3 + 156326 u^2 + u,
// and Q = that y decoded like an EdDSA key with sign 0 (the sign of x never reaches a u-coordinate).  psi_hat(psi) = [4], the
// decode has ratio 1 and the X448 encoder ratio 2: the composite is [+-8], hence k / 8, and it kills the torsion of u as the
// clamped k does in the ladder.  A peer takes the table only if v^2 is a non-zero square (checked here, not left to the
// decoder), u mod p is neither 0 (the denominator vanishes and gf_invert(0) = 0 would hide it) nor p - 1 (y = 1, which the
// decoder rejects), and the decode succeeds; every other peer keeps the ladder.  The flag is public.
struct LaneX448PeerLift {
    abi_pt *pts; int32_t *table_ok; const uint8_t *peers;
    GDM void operator()(size_t i) const {
        uint32_t w[14];
        words_load56(w, peers + 56 * i);
        gf u, u2, v2, a, b, num, den, one;
        (void)gf_from_words(u, w);                       /* u >= p is taken mod p, like the ladder does */
        gf_set_ui(one, 1);
        gf_sqr(u2, u);
        gf_mulw(a, u, 156326);
        gf_add(a, a, u2);
        gf_add(a, a, one);
        gf_mul(v2, a, u);                                /* v^2 = u (u^2 + 156326 u + 1) */
        gf_sub(a, u2, one);
        gf_sqr(a, a);                                    /* (u^2 - 1)^2 */
        gf_add(b, v2, v2);
        gf_add(b, b, b);
        gf_sub(num, a, b);
        gf_mul(num, num, u);                             /* u ((u^2 - 1)^2 - 4 v^2) */
        gf_mul(den, a, u);
        gf_add(b, u2, one);
        gf_mul(b, b, v2);
        gf_add(b, b, b);
        gf_sub(den, den, b);                             /* u (u^2 - 1)^2 - 2 v^2 (u^2 + 1) */
        gmask_t ok = gf_isr(a, v2);                      /* v^2 a non-zero square: u is on the curve, not on its twist */
        ok &= ~gf_is_zero(u);
        gf_add(b, u, one);
        ok &= ~gf_is_zero(b);                            /* u != p - 1 */
        ok &= ~gf_is_zero(den);
        gf_invert(den, den);
        gf_mul(a, num, den);
        gf_neg(a, a);
        uint32_t yw[14];
        gf_to_words(yw, a);
        pt q;
        ok &= pt_decode_like_eddsa(q, yw, 0);
        if (!ok) pt_set_identity(q);                     /* a ladder peer's table is built from the identity and never read */
        pt_to_abi(pts + i, q);
        table_ok[i] = ST_OK(ok);
    }
};
// The comb half of an X448 against a peer with a table: the scalar words ws clamped exactly as the ladder clamps them
// (SlotX448DerivePk), k / 8 through table t of the set, and the fraction num / den = (y^2, x^2) of the result.
GD void s_x448_peer_comb(sref num, sref den, uint32_t ws[14], sref sb, const niels *tables, uint32_t t) {
    ws[0] &= ~3u;
    ws[13] |= 0x80000000u;
    sc s, h;
    ByteAtWords at = {ws};
    sc_decode_long(s, at, 56);
    sc_halve(h, s);
    sc_halve(s, h);
    sc_halve(h, s);                                      /* k / 8 */
    s_comb_scalarmul_table(sb, tables + (size_t)COMB_ENTRIES * t, h);
    s_sqr(num, s_slot(sb, 1));
    s_sqr(den, s_slot(sb, 0));
}
// Element i = goldilocks_x448(peers[peer_index[i]], scalar i): the comb over the peer's table or the ladder, by the peer's
// public flag.  Both leave a fraction num / den -- (y^2, x^2) of the comb result (goldilocks.c:1104-1115 u = (y/x)^2), the
// ladder's (x2, z2) -- and meet in ONE x448_finish, because its inversion is shared across the block (s_block_invert4) and
// every lane has to reach it, whichever branch its warp took.  A missing peer is 0 / 0: zeros and FAILURE.
struct SlotX448Peer {
    static constexpr int NSLOTS = 7;
    static_assert(COMB_NSLOTS == NSLOTS && X448_NSLOTS == NSLOTS, "the comb and the ladder share the slots");
    uint8_t *out; int32_t *status; const niels *tables; const int32_t *table_ok; const uint8_t *peers;
    const uint32_t *peer_index; const uint8_t *scalar; uint32_t n_peers;
    GDM void operator()(size_t i, sref sb, bool live) const {
        uint32_t ws[14], wo[14];
        words_load56(ws, scalar + 56 * i);
        const uint32_t t = peer_index[i];
        sref num = s_slot(sb, 6), den = s_slot(sb, 5);
        if (t >= n_peers) {
            gf z;
            gf_set_zero(z);
            s_st(num, z);
            s_st(den, z);
        } else if (table_ok[t]) {
            s_x448_peer_comb(num, den, ws, sb, tables, t);
        } else {
            uint32_t wu[14];
            words_load56(wu, peers + 56 * (size_t)t);
            x448_ladder_xz(num, den, wu, ws, sb);
        }
        const gmask_t nz = x448_finish(wo, sb, num, den);
        if (!live) return;
        words_store56(out + 56 * i, wo);
        status[i] = ST_OK(nz);
    }
};
// X448 against a peer set by the peer's bytes (goldilocks_x448_peerset_lookup_batch; DESIGN.md decision 24).  Lane j handles
// element i = order[j] (the batch sorted by looked-up peer, LaneDecafPeerKeys: hits grouped by peer, the misses as one tail) in
// place, with t = peer_index[i] (LaneX448PeerLookup: the lowest set index with base i's bytes, or m).  A hit on a peer with a
// table runs its comb; every other element -- a miss, or a peer that keeps the ladder -- runs the ladder on its own base bytes,
// which on a hit are the set's.  Both meet in the one x448_finish every lane has to reach, as in SlotX448Peer.
struct SlotX448PeerLookup {
    static constexpr int NSLOTS = 7;
    static_assert(COMB_NSLOTS == NSLOTS && X448_NSLOTS == NSLOTS, "the comb and the ladder share the slots");
    uint8_t *out; int32_t *status; const niels *tables; const int32_t *table_ok;
    const uint32_t *peer_index, *order; const uint8_t *base, *scalar; uint32_t n_peers;
    GDM void operator()(size_t j, sref sb, bool live) const {
        const size_t i = order[j];
        const uint32_t t = peer_index[i];
        uint32_t ws[14], wo[14];
        words_load56(ws, scalar + 56 * i);
        sref num = s_slot(sb, 6), den = s_slot(sb, 5);
        if (t < n_peers && table_ok[t]) {
            s_x448_peer_comb(num, den, ws, sb, tables, t);
        } else {
            uint32_t wu[14];
            words_load56(wu, base + 56 * i);
            x448_ladder_xz(num, den, wu, ws, sb);
        }
        const gmask_t nz = x448_finish(wo, sb, num, den);
        if (!live) return;
        words_store56(out + 56 * i, wo);
        status[i] = ST_OK(nz);
    }
};
// Decaf peer sets (include/goldilocks_b200.h, goldilocks_b200_decaf_peerset_*; DESIGN.md decision 21): a recurring peer of
// goldilocks_448_direct_scalarmul (goldilocks.c:888-903) is decoded once and gets the reference's (5,5,18) comb table, so a call
// runs the comb instead of the signed-window multiplication.  Both recode the scalar with the same sc_recode_signed and add up
// the same signed digits (every one of the 450 bit positions contributes +-2^k), so they multiply the point by the same
// integer 2 s' - (2^450 - 1): the same point, and the same encoding.  Lane t < m decodes peer t; a peer that fails to decode
// is the base point with FAILURE, exactly as SlotDirectScalarmul selects it.  Entry m is the base point with FAILURE: an index
// >= m is clamped to it, which is what 56 undecodable bytes give.  The status is public.
struct LaneDecafPeerDecode {
    abi_pt *pts; int32_t *peer_ok; const uint8_t *peers; const fixed_tables *ft; uint32_t m, allow_identity;
    GDM void operator()(size_t t) const {
        pt p;
        pt_set_identity(p);
        gmask_t ok = 0;
        if (t < m) {
            uint32_t wd[14];
            words_load56(wd, peers + 56 * t);
            ok = pt_decode(p, wd, allow_identity ? ~0u : 0u);
        }
        pt q; /* point_cond_sel(basep, point_base, basep, succ) */
        gf_cond_sel(q.x, ft->base.x, p.x, ok);
        gf_cond_sel(q.y, ft->base.y, p.y, ok);
        gf_cond_sel(q.z, ft->base.z, p.z, ok);
        gf_cond_sel(q.t, ft->base.t, p.t, ok);
        pt_to_abi(pts + t, q);
        peer_ok[t] = ST_OK(ok);
    }
};
// The sort keys of a call: (min(peer_index[j], m), j).  Sorted by peer, the values are the order SlotDecafPeer takes the
// elements in, so the lanes of a warp read one or two tables instead of up to 32.  Only public data goes through the sort.
struct LaneDecafPeerKeys {
    uint32_t *keys, *vals; const uint32_t *peer_index; uint32_t m;
    GDM void operator()(size_t j) const {
        const uint32_t t = peer_index[j];
        keys[j] = t < m ? t : m;
        vals[j] = (uint32_t)j;
    }
};
// Lane j: element i = order[j] of goldilocks_448_direct_scalarmul(scaled_i, peers[peer_index[i]], scalar i, allow_identity of
// the set, short_circuit).  The comb over table min(peer_index[i], m), the decaf encoding, the peer's status; with short_circuit
// a failed element keeps the caller's bytes through SlotDirectScalarmul's masked merge.  Reads and writes element i in place.
struct SlotDecafPeer {
    static constexpr int NSLOTS = COMB_NSLOTS;
    uint8_t *scaled; int32_t *status; const niels *tables; const int32_t *peer_ok; const uint32_t *peer_index; const uint32_t *order;
    const abi_sc *scalar; uint32_t n_peers, short_circuit;
    GDM void operator()(size_t j, sref sb, bool live) const {
        const size_t i = order[j];
        const uint32_t ti = peer_index[i];
        const size_t t = ti < n_peers ? ti : n_peers;
        sc s;
        sc_from_abi(s, scalar + i);
        s_comb_scalarmul_table(sb, tables + (size_t)COMB_ENTRIES * t, s);
        pt q;
        s_ld(q.x, s_slot(sb, 0)); s_ld(q.y, s_slot(sb, 1)); s_ld(q.z, s_slot(sb, 2)); s_ld(q.t, s_slot(sb, 3));
        gf e;
        pt_deisogenize(e, q);
        uint32_t wd[14];
        gf_to_words(wd, e);
        if (!live) return;
        const int32_t st = peer_ok[t];
        status[i] = st;
        uint32_t keep[14];
        words_load56(keep, scaled + 56 * i);
        const gmask_t wr = (gmask_t)st | (short_circuit ? 0u : ~0u);
#pragma unroll
        for (int k = 0; k < 14; k++) wd[k] = (wd[k] & wr) | (keep[k] & ~wr);
        words_store56(scaled + 56 * i, wd);
    }
};
// Point sets (include/goldilocks_b200.h, goldilocks_b200_pointset_*; DESIGN.md decision 22): goldilocks_448_base_double_scalarmul_non_secret
// (goldilocks.c:1260-1330) against a recurring point, from the tables a key set keeps for its keys (flat: FLAT = true, or the compact
// ten-column layout).  Both evaluations add the same sc_recode_signed digits of scalar2 times the same multiples of the point as
// s_base_double_scalarmul, and scalar1 B from the same fixed-base tables, so they give the same point, torsion included.  Table m of
// the set is the identity's: an index >= m is clamped to it, so the kernel never branches on the index.  Lane j handles element
// i = order[j] (the batch sorted by point, LaneDecafPeerKeys) and writes out[i] in place.  Variable time, like the reference's _non_secret.
template <bool FLAT>
struct SlotPointset {
    static constexpr int NSLOTS = BDSM_NSLOTS;
    abi_pt *out; const abi_sc *scalar1, *scalar2; const niels *wide; const uint4 *ktabs; const uint32_t *point_index, *order; uint32_t n_points;
    GDM void operator()(size_t j, sref sb, size_t slot) const {
        (void)slot;
        const size_t i = order[j];
        const uint32_t ti = point_index[i];
        const size_t t = ti < n_points ? ti : n_points;
        sc s1, s2;
        sc_from_abi(s1, scalar1 + i);
        sc_from_abi(s2, scalar2 + i);
        if (FLAT) s_verify_flat_key(sb, s1, s2, wide, kset_of(const_cast<uint4 *>(ktabs), t), true);
        else s_verify_shared_key<true>(sb, s1, s2, wide, ktab_of(const_cast<uint4 *>(ktabs), t), VSH_ROWS, VSH_CHUNKS, true);   /* affine entries */
        s_bdsm_quirk(sb, s2);
        s_pt_to_abi(out + i, sb);
    }
};
struct SlotEdDerivePk { /* eddsa.c:129-144 */
    static constexpr int NSLOTS = COMB_NSLOTS;
    uint8_t *pk; const uint8_t *sk; const fixed_tables *ft;
    GDM void operator()(size_t i, sref sb, bool live) const {
        sc s, h1, h2; uint32_t w[15], sign; shake256_ctx hk;
        ed448_secret_scalar(s, hk, sk + 57 * i);
        sc_halve(h1, s);
        sc_halve(h2, h1);      /* GOLDILOCKS_448_EDDSA_ENCODE_RATIO = 4 */
        s_comb_scalarmul(sb, ft->win, h2);
        s_encode_like_eddsa(w, sign, sb);
        w[14] = sign << 7;
        if (live) words_store_bytes(pk + 57 * i, 57, w);
    }
};
struct SlotEdSignR { /* eddsa.c:201-205: R = encode(comb(nonce / 4)) */
    static constexpr int NSLOTS = COMB_NSLOTS;
    uint8_t *sig; const abi_sc *nonce4; const fixed_tables *ft;
    GDM void operator()(size_t i, sref sb, bool live) const {
        sc s; uint32_t w[15], sign;
        sc_from_abi(s, nonce4 + i);
        s_comb_scalarmul(sb, ft->win, s);
        s_encode_like_eddsa(w, sign, sb);
        w[14] = sign << 7;
        if (live) words_store_bytes(sig + 114 * i, 57, w);
    }
};

struct SlotScalarmul { /* goldilocks_448_point_scalarmul (goldilocks.c:405-465); `slot` indexes per-thread HBM scratch */
    static constexpr int NSLOTS = WINDOW_NSLOTS;
    abi_pt *out; const abi_pt *base; const abi_sc *scalar; uint4 *scratch;
    GDM void operator()(size_t i, sref sb, size_t slot) const {
        sc s;
        sc_from_abi(s, scalar + i);
        s_pt_from_abi(sb, base + i);
        s_window_scalarmul(sb, s, wtab_of<32>(scratch, slot));
        s_pt_to_abi(out + i, sb);
    }
};
struct LoadAbiPt { const abi_pt *p; GDM void operator()(sref sb) const { s_pt_from_abi(sb, p); } };
struct SlotDoubleScalarmul { /* goldilocks_448_point_double_scalarmul (goldilocks.c:467-541) */
    static constexpr int NSLOTS = WINDOW_NSLOTS;
    abi_pt *out; const abi_pt *base1; const abi_sc *scalar1; const abi_pt *base2; const abi_sc *scalar2; uint4 *scratch; size_t nthreads; /* scratch = two tables per thread */
    GDM void operator()(size_t i, sref sb, size_t slot) const {
        sc s1, s2;
        sc_from_abi(s1, scalar1 + i); sc_from_abi(s2, scalar2 + i);
        s_pt_from_abi(sb, base1 + i);
        LoadAbiPt load2 = {base2 + i};
        s_window_double_scalarmul(sb, s1, s2, load2, wtab_of<32>(scratch, slot), wtab_of<32>(scratch + nthreads * WTAB_QUADS_PER_LANE, slot));
        s_pt_to_abi(out + i, sb);
    }
};

struct SlotDualScalarmul { /* goldilocks_448_point_dual_scalarmul (goldilocks.c:543-642): a1 = scalar1*b, a2 = scalar2*b, one table */
    static constexpr int NSLOTS = WINDOW_NSLOTS;
    abi_pt *out1, *out2; const abi_pt *base; const abi_sc *scalar1, *scalar2; uint4 *scratch;
    GDM void operator()(size_t i, sref sb, size_t slot) const {
        const spt p = {s_slot(sb, 0), s_slot(sb, 1), s_slot(sb, 2), s_slot(sb, 3)};
        const swk w = {s_slot(sb, 4), s_slot(sb, 5), s_slot(sb, 6)};
        const wtab<32> t = wtab_of<32>(scratch, slot);
        sc s, sx;
        s_pt_from_abi(sb, base + i);
        s_prepare_fixed_window<32>(p, w, t);
        sc_from_abi(s, scalar1 + i);
        sc_recode_signed(sx, s);
        s_window_mainloop(p, w, sx, t);
        s_pt_to_abi(out1 + i, sb);
        sc_from_abi(s, scalar2 + i);
        sc_recode_signed(sx, s);
        s_window_mainloop(p, w, sx, t);
        s_pt_to_abi(out2 + i, sb);
    }
};
// goldilocks_448_direct_scalarmul (goldilocks.c:888-903): decode, (base point when the decode failed),
// constant-time scalarmul, encode.  status = the decode's; with short_circuit a failed element is not written.
struct SlotDirectScalarmul {
    static constexpr int NSLOTS = WINDOW_NSLOTS;
    uint8_t *scaled; int32_t *status; const uint8_t *base; const abi_sc *scalar; uint32_t allow_identity, short_circuit;
    const fixed_tables *ft; uint4 *scratch;
    GDM void operator()(size_t i, sref sb, size_t slot) const {
        uint32_t wd[14];
        words_load56(wd, base + 56 * i);
        gmask_t ok;
        {
            pt p;
            ok = pt_decode(p, wd, allow_identity ? ~0u : 0u);
            gf v; /* point_cond_sel(basep, point_base, basep, succ) */
            gf_cond_sel(v, ft->base.x, p.x, ok); s_st(s_slot(sb, 0), v);
            gf_cond_sel(v, ft->base.y, p.y, ok); s_st(s_slot(sb, 1), v);
            gf_cond_sel(v, ft->base.z, p.z, ok); s_st(s_slot(sb, 2), v);
            gf_cond_sel(v, ft->base.t, p.t, ok); s_st(s_slot(sb, 3), v);
        }
        sc s;
        sc_from_abi(s, scalar + i);
        s_window_scalarmul(sb, s, wtab_of<32>(scratch, slot));
        pt q;
        s_ld(q.x, s_slot(sb, 0)); s_ld(q.y, s_slot(sb, 1)); s_ld(q.z, s_slot(sb, 2)); s_ld(q.t, s_slot(sb, 3));
        gf e;
        pt_deisogenize(e, q);
        gf_to_words(wd, e);
        status[i] = ST_OK(ok);
        /* short-circuited elements keep the caller's bytes (goldilocks.c:896): a masked merge, not a branch on the decode's verdict */
        uint32_t keep[14];
        words_load56(keep, scaled + 56 * i);
        const gmask_t wr = ok | (short_circuit ? 0u : ~0u);
#pragma unroll
        for (int k = 0; k < 14; k++) wd[k] = (wd[k] & wr) | (keep[k] & ~wr);
        words_store56(scaled + 56 * i, wd);
    }
};
struct SlotCombTable { /* goldilocks_448_precomputed_scalarmul over a caller-supplied table (goldilocks.c:830-877) */
    static constexpr int NSLOTS = COMB_NSLOTS;
    abi_pt *out; const abi_sc *scalar; const niels *table;
    GDM void operator()(size_t i, sref sb, bool live) const {
        sc s;
        sc_from_abi(s, scalar + i);
        s_comb_scalarmul_table(sb, table, s);
        if (live) s_pt_to_abi(out + i, sb);
    }
};

// ---- direct access to the mixed additions (SURVEY 8(a) row a9; goldilocks.c:271-380) -- test entry point only -------------------
// The reference keeps pt_to_pniels / pniels_to_pt / niels_to_pt / add_niels_to_pt / sub_niels_from_pt / add_pniels_to_pt /
// sub_pniels_from_pt static, so every caller reaches them through a scalar multiplication.  goldilocks_b200_debug_niels_batch runs ONE of
// them per element, in both shapes the kernels use -- by value (point.cuh, the lane kernels) and on the slot machine (slot_algos.cuh,
// the scalar-multiplication kernels) -- so that all four output coordinates can be pinned to the reference's formulas.
//   op 0: pniels_to_pt(pt_to_pniels(q))      1 / 2: p +/- pniels(q), by value        3 / 4: p +/- comb[which], by value
//   op 5: niels_to_pt(comb[which])           6 / 7: p +/- pniels(q), slot machine    8 / 9: p +/- comb[which], slot machine
//   op 10 (internal): recs[i] = the projective-niels record of q the slot machine adds from (y - x, y + x, -2 d' t, 2 z)
struct LanePtNiels {
    abi_pt *out; pt *recs; const abi_pt *p, *q; const niels *comb; const uint32_t *which; uint32_t op;
    GDM void operator()(size_t i) const {
        pt P, Q, R;
        pt_from_abi(P, p + i);
        pt_from_abi(Q, q + i);
        pniels pn;
        pt_to_pniels(pn, Q);
        niels e;
        const niels *src = comb + which[i] % COMB_ENTRIES;
        gf_ld<false>(e.a, &src->a); gf_ld<false>(e.b, &src->b); gf_ld<false>(e.c, &src->c);
        pt_copy(R, P);
        if (op == 0) pniels_to_pt(R, pn);
        else if (op == 1) pt_addsub_pniels<false>(R, pn, false);
        else if (op == 2) pt_addsub_pniels<true>(R, pn, false);
        else if (op == 3) pt_addsub_niels<false>(R, e, false);
        else if (op == 4) pt_addsub_niels<true>(R, e, false);
        else if (op == 5) niels_to_pt(R, e);
        else {
            pt rec;
            gf_copy(rec.x, pn.n.a); gf_copy(rec.y, pn.n.b); gf_neg(rec.z, pn.n.c); gf_copy(rec.t, pn.z);
            gf_copy(recs[i].x, rec.x); gf_copy(recs[i].y, rec.y); gf_copy(recs[i].z, rec.z); gf_copy(recs[i].t, rec.t);
        }
        pt_to_abi(out + i, R);
    }
};
struct SlotNielsDebug {
    static constexpr int NSLOTS = 7;
    abi_pt *out; const abi_pt *p; const pt *recs; const niels *comb; const uint32_t *which; uint32_t op;
    GDM void operator()(size_t i, sref sb, bool live) const {
        const spt P = {s_slot(sb, 0), s_slot(sb, 1), s_slot(sb, 2), s_slot(sb, 3)};
        const swk w = {s_slot(sb, 4), s_slot(sb, 5), s_slot(sb, 6)};
        s_pt_from_abi(sb, p + i);
        const gmask_t sub = (op & 1u) ? ~0u : 0u;
        if (op < 8) {
            wtab<1> t;
            t.base = reinterpret_cast<uint4 *>(const_cast<pt *>(recs + i));
            s_pt_add_pniels_g<1>(P, w, t, 0, sub, ~sub, false);      /* the record holds -c: an addition negates it back */
        } else {
            const niels *e = comb + which[i] % COMB_ENTRIES;
            s_pt_add_niels_g<1>(P, w, gq(&e->a), gq(&e->b), gq(&e->c), sub, sub, false);
        }
        if (live) s_pt_to_abi(out + i, sb);
    }
};
