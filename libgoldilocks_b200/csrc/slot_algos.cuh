// slot_algos.cuh -- the long-running scalar multiplications written against the slot machine
// (slots.cuh): X448 ladder, verification double-scalar multiplication, fixed-base comb.
// Formula-for-formula the same group law as point.cuh / algos.cuh (which cite the reference);
// only the storage discipline differs: operands are slot handles, conditional swaps are handle
// selections, table entries are multiplied straight out of global memory.
#pragma once
#include "slots.cuh"
#include "algos.cuh"

#if defined(__CUDA_ARCH__)
// Block-shared inversion (Montgomery's trick across lanes; the reference does the same thing across table
// entries in goldilocks.c:703-726).  Every lane of the block has a NONZERO field element in slot `zin`;
// on return its inverse is in slot `zout`.  Warp 0 does the work for the four lanes (w, l), w = 0..3, that
// share lane index l: 3 prefix products, ONE inversion chain, 6 multiplications -- the other three warps
// wait at the barrier (other resident blocks keep the multiplier busy).  All 128 lanes of the block must
// call it (k_slots keeps out-of-range lanes alive for this); slots 0..2 and `zout` of every lane are clobbered.
// Constant time: the schedule is fixed, operands are only multiplied.
GD void s_block_invert4(sref sb, int zin, int zout) {
    __syncthreads();
    if (threadIdx.x < 32) {
        sref t[4]; /* slot 0 of the four lanes served by this lane */
#pragma unroll
        for (int w = 0; w < 4; w++) t[w] = s_lane_shift(sb, 32u * w);
        const sref z0 = s_slot(t[0], zin), z1 = s_slot(t[1], zin), z2 = s_slot(t[2], zin), z3 = s_slot(t[3], zin);
        const sref p1 = s_slot(t[0], 0), p2 = s_slot(t[0], 1), p3 = s_slot(t[0], 2), inv = s_slot(t[1], 0);
        s_mul(p1, z0, z1);
        s_mul(p2, p1, z2);
        s_mul(p3, p2, z3);
        s_invert(inv, p3, s_slot(t[1], 1), s_slot(t[1], 2));
        s_mul(s_slot(t[3], zout), inv, p2);
        s_mul(inv, inv, z3);
        s_mul(s_slot(t[2], zout), inv, p1);
        s_mul(inv, inv, z2);
        s_mul(s_slot(t[1], zout), inv, z0);
        s_mul(s_slot(t[0], zout), inv, z1);
    }
    __syncthreads();
}
#endif

// ---------------------------------------------------------------------------------------------
// X448 (RFC 7748) -- reference goldilocks.c:1006-1076.  Per bit: 3 addsub, 5 M, 4 S, 1 sub,
// 1 mulw+add = 14 slot operations on 7 slots; the two conditional swaps exchange handles only.
// ---------------------------------------------------------------------------------------------
#define X448_NSLOTS 7
// The ladder proper: on return x_out / z_out name the slots (two of 1..4) that hold the projective result.
GD void x448_ladder_xz(sref &x_out, sref &z_out, const uint32_t base[14], const uint32_t scalar[14], sref sb) {
    sref x1 = s_slot(sb, 0), x2 = s_slot(sb, 1), z2 = s_slot(sb, 2), x3 = s_slot(sb, 3), z3 = s_slot(sb, 4), t1 = s_slot(sb, 5), t2 = s_slot(sb, 6);
    {
        gf v;
        (void)gf_from_words(v, base); /* u >= p is accepted mod p, like the reference's ignored result */
        s_st(x1, v); s_st(x3, v);
        gf_set_ui(v, 1);
        s_st(x2, v); s_st(z3, v);
        gf_set_zero(v);
        s_st(z2, v);
    }
    gmask_t swap = 0;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int w = 13; w >= 0; w--) {
        uint32_t word = 0;
#pragma unroll
        for (int i = 0; i < 14; i++) word |= (i == w) ? scalar[i] : 0u;
        if (w == 0) word &= ~3u;            /* clear the cofactor bits */
        if (w == 13) word |= 0x80000000u;   /* force bit 447 */
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (int b = 31; b >= 0; b--) {
            const gmask_t k_t = (gmask_t)(-(int32_t)((word >> b) & 1u));
            swap ^= k_t;
            { /* cswap(x2,x3), cswap(z2,z3): the lane renames its slots, no data moves */
                const sref nx2 = s_sel(x2, x3, swap), nx3 = s_sel(x3, x2, swap);
                const sref nz2 = s_sel(z2, z3, swap), nz3 = s_sel(z3, z2, swap);
                x2 = nx2; x3 = nx3; z2 = nz2; z3 = nz3;
            }
            swap = k_t;
            s_addsub(t1, t2, x2, z2);          /* A = x2+z2, B = x2-z2 */
            s_addsub(x2, z2, x3, z3);          /* C = x3+z3, D = x3-z3 */
            s_mul(x3, z2, t1);                 /* DA */
            s_mul(z3, x2, t2);                 /* CB */
            s_addsub(x2, z2, x3, z3);          /* DA+CB, DA-CB */
            s_sqr(x3, x2);                     /* x3 = (DA+CB)^2 */
            s_sqr(z3, z2);
            s_mul(z3, x1, z3);                 /* z3 = x1 (DA-CB)^2 */
            s_sqr(x2, t1);                     /* AA */
            s_sqr(z2, t2);                     /* BB */
            s_sub(t2, x2, z2);                 /* E = AA-BB */
            s_mulw_add(t1, t2, (uint32_t)(-GOLD_EDWARDS_D), x2); /* a24*E + AA */
            s_mul(x2, x2, z2);                 /* x2 = AA*BB */
            s_mul(z2, t2, t1);                 /* z2 = E (AA + a24 E) */
        }
    }
    {
        const sref nx2 = s_sel(x2, x3, swap), nx3 = s_sel(x3, x2, swap);
        const sref nz2 = s_sel(z2, z3, swap), nz3 = s_sel(z3, z2, swap);
        x2 = nx2; x3 = nx3; z2 = nz2; z3 = nz3;
    }
    x_out = x2;
    z_out = z2;
}
// out = canonical bytes of num / den, 0 for den = 0 (goldilocks.c:69-80 gf_invert(0) = 0); all-ones iff out != 0.
// num: any slot but 5, den: any slot; every slot is clobbered.  On the device the inversion is
// shared by the four lanes of a block that have the same lane index (s_block_invert4 below): one addition chain
// per four elements instead of one per element -- so every lane of the block has to get here.
GD gmask_t x448_finish(uint32_t out[14], sref sb, sref num, sref den) {
    const sref zi = s_slot(sb, 5), xs = s_slot(sb, 6), res = s_slot(sb, 0);
    gmask_t nz;
    {
        gf z, one;
        s_ld(z, den);
        nz = ~gf_is_zero(z);
        gf_set_ui(one, 1);
        gf_cond_sel(z, one, z, nz);             /* 0 -> 1 so it cannot poison the shared product */
        s_st(zi, z);
        s_copy(xs, num);
    }
#if defined(__CUDA_ARCH__)
    s_block_invert4(sb, 5, 4);                  /* slot 5 -> its inverse in slot 4 */
    s_mul(res, xs, s_slot(sb, 4));
#else
    s_invert(s_slot(sb, 4), zi, s_slot(sb, 1), s_slot(sb, 2));
    s_mul(res, xs, s_slot(sb, 4));
#endif
    gf r, zero;
    s_ld(r, res);
    gf_set_zero(zero);
    gf_cond_sel(r, zero, r, nz);
    gf_to_words(out, r);
    return ~gf_is_zero(r);
}
GD gmask_t x448_ladder_slots(uint32_t out[14], const uint32_t base[14], const uint32_t scalar[14], sref sb) {
    sref x2, z2;
    x448_ladder_xz(x2, z2, base, scalar, sb);
    return x448_finish(out, sb, x2, z2);
}

// ---------------------------------------------------------------------------------------------
// Group law on slots.  A point occupies four slots (X, Y, Z, T); `w` names three scratch slots.
// Same formulas as point.cuh (goldilocks.c:232-254, 315-380); sign handling of table entries is a
// per-lane handle/pointer selection instead of a data swap.
// ---------------------------------------------------------------------------------------------
struct spt { sref x, y, z, t; };
struct swk { sref t0, t1, t2; };

// p = 2p.  4S + 3M (+1M for T).  (goldilocks.c:232-254 point_double_internal)  T is dead on entry
// and serves as the fourth temporary.
GD void s_pt_double(const spt &p, const swk &w, bool before_double) { /* 9 (10 with T) slot operations */
    s_sqr_sum(w.t2, p.y, p.x);          /* (x+y)^2 */
    s_sqr2_addsub(p.t, w.t1, p.x, p.y); /* d = y^2 + x^2 ; e = y^2 - x^2 (one pass: -0.6 % on verify) */
    s_sub(w.t2, w.t2, p.t);            /* b = (x+y)^2 - d  (fusing this into the square above: no gain) */
    s_sqr2_sub(w.t0, p.z, w.t1);       /* a' = 2 z^2 - e */
    s_mul(p.x, w.t0, w.t2);
    s_mul(p.z, w.t1, w.t0);
    s_mul(p.y, w.t1, p.t);
    if (!before_double) s_mul(p.t, w.t2, p.t);
}

// A lane's window table of pniels in global memory (coordinate order a, b, c, z), in one of the two
// layouts of slots.cuh: QS = 1 lane-contiguous (256 B per entry; public-index gathers of verification),
// QS = 32 warp-interleaved (constant-time scans are fully coalesced).
template <int QS>
struct wtab {
    uint4 *base; /* this lane's quad 0 of coordinate 0 of entry 0 */
    GDM uint4 *coord(int e, int c) const { return base + (size_t)(e * 4 + c) * 4 * QS; }
    static constexpr int ESTRIDE = 16 * QS; /* quads between the same coordinate of consecutive entries */
};
#define WTAB_ENTRIES 17 /* 16 odd multiples + pniels(2P) while the table is being built */
#define WTAB_QUADS_PER_LANE (WTAB_ENTRIES * 16)
template <int QS>
GD wtab<QS> wtab_of(uint4 *scratch, size_t thread) { /* thread = global thread index (device) or worker index (host) */
    wtab<QS> t;
    if (QS == 1) t.base = scratch + thread * WTAB_QUADS_PER_LANE;
    else t.base = scratch + (thread / 32) * (size_t)(WTAB_QUADS_PER_LANE * 32) + (thread % 32);
    return t;
}

// p += (+-) e for an affine niels e = (a, b, c) in global memory.  7M (6M without T).
//   swap_ab : use (b, a) instead of (a, b)       \\  a negated entry is swap_ab = neg_c = all-ones
//   neg_c   : the stored c is minus the real one  /  (goldilocks.c:271-278 cond_neg_niels)
// (goldilocks.c:315-359 add_niels_to_pt / sub_niels_from_pt)
template <int QS>
GD void s_pt_add_niels_g(const spt &p, const swk &w, const uint4 *ea, const uint4 *eb, const uint4 *ec, gmask_t swap_ab, gmask_t neg_c, bool before_double) {
    const uint4 *pa = swap_ab ? eb : ea, *pb = swap_ab ? ea : eb; /* per-lane select of two addresses: no divergence */
    s_addsub(w.t1, w.t0, p.y, p.x);    /* y+x ; y-x */
    s_mulg<QS>(w.t0, w.t0, pa);        /* a  = e.a (y-x) */
    s_mulg<QS>(w.t1, w.t1, pb);        /* dy = e.b (y+x) */
    s_mulg<QS>(p.x, p.t, ec);          /* x  = e.c t */
    s_addsub(w.t2, w.t1, w.t1, w.t0);  /* c = dy + a ; b = dy - a */
    s_addsub(w.t0, p.y, p.z, p.x);     /* v = z + x ; u = z - x */
    s_mul(p.z, w.t0, p.y);             /* z = u v */
    s_mul(p.x, s_sel(p.y, w.t0, neg_c), w.t1);   /* x = (neg ? v : u) b */
    s_mul(p.y, s_sel(w.t0, p.y, neg_c), w.t2);   /* y = (neg ? u : v) c */
    if (!before_double) s_mul(p.t, w.t1, w.t2);  /* t = b c */
}
// entry e of a window table: z first (goldilocks.c:361-380)
template <int QS>
GD void s_pt_add_pniels_g(const spt &p, const swk &w, const wtab<QS> &t, int e, gmask_t swap_ab, gmask_t neg_c, bool before_double) {
    s_mulg<QS>(p.z, p.z, t.coord(e, 3));
    s_pt_add_niels_g<QS>(p, w, t.coord(e, 0), t.coord(e, 1), t.coord(e, 2), swap_ab, neg_c, before_double);
}
// table[e] = pniels(p) with c stored NEGATED (c' = +2*39082*t = -(2 d' t), saves a negation per entry;
// readers pass neg_c = ~sign).  a TIGHT, b and z LOOSE (they only ever feed multiplications).
// (goldilocks.c:280-288 pt_to_pniels)
template <int QS>
GD void s_pt_to_pniels_negc_g(const wtab<QS> &t, int e, const spt &p, const swk &w) {
    s_addsub(w.t1, w.t0, p.y, p.x);
    s_stg<QS>(t.coord(e, 0), w.t0);
    s_stg<QS>(t.coord(e, 1), w.t1);
    s_mulw(w.t0, p.t, (uint32_t)(-2 * GOLD_TWISTED_D));
    s_stg<QS>(t.coord(e, 2), w.t0);
    s_add(w.t0, p.z, p.z);
    s_stg<QS>(t.coord(e, 3), w.t0);
}
// table[0..15] = odd multiples 1P..31P of the point in slots 0..3; table[16] is scratch.  Clobbers the
// point: P, then 2P + P, then += 2P.  (goldilocks.c:382-403 prepare_fixed_window)
template <int QS>
GD void s_prepare_fixed_window(const spt &p, const swk &w, const wtab<QS> &t) {
    s_pt_to_pniels_negc_g<QS>(t, 0, p, w);
    s_pt_double(p, w, false);
    s_pt_to_pniels_negc_g<QS>(t, 16, p, w);
    s_pt_add_pniels_g<QS>(p, w, t, 0, 0, ~0u, false);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int i = 1; i < WINDOW_NTABLE; i++) {
        s_pt_to_pniels_negc_g<QS>(t, i, p, w);
        if (i != WINDOW_NTABLE - 1) s_pt_add_pniels_g<QS>(p, w, t, 16, 0, ~0u, false);
    }
}
GD void s_pt_set_identity(const spt &p) {
    gf v;
    gf_set_zero(v); s_st(p.x, v); s_st(p.t, v);
    gf_set_ui(v, 1); s_st(p.y, v); s_st(p.z, v);
}

// p += scalar1 * B for the recoded scalar s1x (sc_recode_signed): its WIDE_TABLES signed WIDE_BITS-bit digits against the init-time
// tables of odd multiples of 2^(WIDE_BITS m) B (algos.cuh) -- additions only, no doublings.  T of the result only on request.
GD void s_add_fixed_base(const spt &p, const swk &w, const sc &s1x, const niels *wide, bool need_t) {
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int m = 0; m < WIDE_TABLES; m++) {
        uint32_t bits1 = sc_bits(s1x, m * WIDE_BITS, WIDE_BITS);
        const gmask_t inv1 = (gmask_t)((int32_t)(bits1 >> (WIDE_BITS - 1)) - 1);
        bits1 ^= inv1;
        const niels *e = wide + (size_t)m * WIDE_ENTRIES + (bits1 & (WIDE_ENTRIES - 1));
        s_pt_add_niels_g<1>(p, w, gq(&e->a), gq(&e->b), gq(&e->c), inv1, inv1, m == WIDE_TABLES - 1 && !need_t);
    }
}

#define BDSM_NSLOTS 7
// combo = scalar1*B + scalar2*base2 for PUBLIC inputs, warp-uniform schedule -- see the comment on
// "combo = scalar1*B + scalar2*base2" in algos.cuh, which defines the digits and the tables.
// On entry the slots X,Y,Z,T (0..3) hold base2; on exit they hold the result (X, Y, Z valid, T valid).
// `multiples` = this lane's window table (lane-contiguous layout: the digits are public, entries are gathered).
GD void s_base_double_scalarmul(sref sb, const sc &scalar1, const sc &scalar2, const niels *wide_base, const wtab<1> &multiples) {
    const spt p = {s_slot(sb, 0), s_slot(sb, 1), s_slot(sb, 2), s_slot(sb, 3)};
    const swk w = {s_slot(sb, 4), s_slot(sb, 5), s_slot(sb, 6)};
    sc s1x, s2x;
    sc_recode_signed(s1x, scalar1);
    sc_recode_signed(s2x, scalar2);
    s_prepare_fixed_window<1>(p, w, multiples);   /* odd multiples 1P, 3P, ..., 31P */
    s_pt_set_identity(p);                      /* the unified addition law takes it from there */
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int k = 89; k >= 0; k--) {
        const int i = k * WINDOW_BITS;
        if (k != 89) {
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
            for (int j = 0; j < WINDOW_BITS - 1; j++) s_pt_double(p, w, true);
            s_pt_double(p, w, false);
        }
        uint32_t bits2 = sc_window5(s2x, i);
        const gmask_t inv2 = (gmask_t)((int32_t)(bits2 >> (WINDOW_BITS - 1)) - 1);
        bits2 ^= inv2;
        s_pt_add_pniels_g<1>(p, w, multiples, (int)(bits2 & (WINDOW_NTABLE - 1)), inv2, ~inv2, k != 0);
    }
    s_add_fixed_base(p, w, s1x, wide_base, true);
}

// ---------------------------------------------------------------------------------------------
// Stand-alone verification with half-size multipliers (sc.cuh sc_half_gcd): instead of combo = s B + c A, compared with R,
//     slots 0..3  <-  sB * B  +  u * A  -+  |v| * R          (sB = v s mod q,  v c == u mod q,  u, |v| < 2^223),
// which is the identity of the quotient group exactly when combo == R there (v is a unit mod q and the quotient group has
// prime order q; goldilocks.c:644-653 point_eq is equality in that group).  u and |v| are 45 signed 5-bit digits each
// (sc_half_bias), so there are 44 x 5 doublings instead of 89 x 5; the full-size sB goes to the doubling-free init-time tables
// of the fixed base (s_add_fixed_base).
// Window tables: entry e = (e + 1) P for e = 0..15, entry 16 = the identity (digit 0) -- 15 additions per table.
// ---------------------------------------------------------------------------------------------
template <int QS>
GD void s_prepare_signed_window(const spt &p, const swk &w, const wtab<QS> &t) {
    s_pt_to_pniels_negc_g<QS>(t, 0, p, w);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int i = 1; i < WINDOW_NTABLE; i++) {
        s_pt_add_pniels_g<QS>(p, w, t, 0, 0, ~0u, false);
        s_pt_to_pniels_negc_g<QS>(t, i, p, w);
    }
    s_pt_set_identity(p);
    s_pt_to_pniels_negc_g<QS>(t, WINDOW_NTABLE, p, w);       /* a = b = 1, c = 0, z = 2 */
}
// p += d * P for the signed digit d = biased - 16 of a window table built by s_prepare_signed_window; `flip` negates the term
GD void s_pt_add_signed_digit(const spt &p, const swk &w, const wtab<1> &t, uint32_t biased, gmask_t flip, bool before_double) {
    const int32_t d = (int32_t)biased - 16;
    const uint32_t mag = (uint32_t)(d < 0 ? -d : d);
    const gmask_t neg = (d < 0 ? ~0u : 0u) ^ flip;
    s_pt_add_pniels_g<1>(p, w, t, mag ? (int)mag - 1 : WINDOW_NTABLE, neg, ~neg, before_double);
}
// On entry ta and tr hold the window tables of A and R; ub, vb are the biased multipliers (sc_half_bias), v_neg the sign of v.
GD void s_verify_half(sref sb, const sc &sB, const sc &ub, const sc &vb, gmask_t v_neg, const niels *wide, const wtab<1> &ta, const wtab<1> &tr) {
    const spt p = {s_slot(sb, 0), s_slot(sb, 1), s_slot(sb, 2), s_slot(sb, 3)};
    const swk w = {s_slot(sb, 4), s_slot(sb, 5), s_slot(sb, 6)};
    sc s1x;
    sc_recode_signed(s1x, sB);
    s_pt_set_identity(p);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int k = HALF_WINDOWS - 1; k >= 0; k--) {
        if (k != HALF_WINDOWS - 1) {
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
            for (int j = 0; j < WINDOW_BITS - 1; j++) s_pt_double(p, w, true);
            s_pt_double(p, w, false);
        }
        s_pt_add_signed_digit(p, w, ta, sc_window5(ub, k * WINDOW_BITS), 0, false);
        s_pt_add_signed_digit(p, w, tr, sc_window5(vb, k * WINDOW_BITS), ~v_neg, k != 0);   /* - v R */
    }
    s_add_fixed_base(p, w, s1x, wide, false);
}

// ---------------------------------------------------------------------------------------------
// Verification under a repeated public key (SURVEY 8(f)4; same group element as s_base_double_scalarmul).
// The 90 signed 5-bit digits d_k of scalar2 (the very recoding above) are regrouped by column: k = R c + r with
// R = VSH_ROWS (9) rows and VSH_CHUNKS (10) columns, so
//     combo = sum_r 2^(5r) * sum_c d_(Rc+r) * A_c   +   scalar1 * B,
// with A_c = 2^(5Rc) A from a table built ONCE PER KEY (s_build_key_tables: 9 x 45 doublings + ten
// 16-entry tables of odd multiples, shared read-only by every signature under that key) and scalar1 * B from the
// doubling-free init-time tables (s_add_fixed_base: 25 signed 18-bit digits).  One signature then costs 8 x 5 doublings
// + 90 + 25 additions.
// Table layout: KTAB_ENTRIES pniels, entry 16c + e = (2e+1) A_c; the last two entries are build scratch.
// ---------------------------------------------------------------------------------------------
#define KTAB_ENTRIES (VSH_CHUNKS * WINDOW_NTABLE + 2)
#define KTAB_QUADS (KTAB_ENTRIES * 16)
GD wtab<1> ktab_of(uint4 *ktabs, size_t table, uint32_t quads_per_key = KTAB_QUADS) { wtab<1> t; t.base = ktabs + table * (size_t)quads_per_key; return t; }
// The column shape of a BATCH's per-key tables is picked on the device, from the work lists the grouping pass leaves (no host round
// trip).  More columns = fewer rows = fewer doublings per signature, for more column tables per key:
//     columns x rows      doublings / signature     MAC32 / key table     taken from (signatures per key table)
//       10 x 9                   40                      659 k                  --
//       15 x 6                   25                      792 k                   9      (B200, 16 per key: step 45.2 -> 44.3 ms)
//       30 x 3                   10                    1 176 k                  32
//       90 x 1                    0                    2 659 k                 256      (one signer for the whole batch: additions only)
// Every shape fits the buffer sized for n/4 + 1 tables of the narrow one, because it is only taken when the tables are that few.
struct vsh_shape { int rows, chunks; uint32_t quads; };
#define VSH_MAX_CHUNKS_PER_SIG_NUM 15 /* columns built per signature, at most: 15 / 9 for the 15 x 6 shape (launch bound of the column kernel) */
#define VSH_MAX_CHUNKS_PER_SIG_DEN 9
GD vsh_shape vsh_make(int rows, int chunks) { vsh_shape s; s.rows = rows; s.chunks = chunks; s.quads = (uint32_t)chunks * WINDOW_NTABLE * 16; return s; }
GD vsh_shape vsh_pick(const uint32_t *counts) { /* counts[0] = signatures under key tables, counts[2] = key tables (verify_plan.cuh) */
    const uint64_t sigs = counts[0], tabs = counts[2];
    if (sigs >= 256 * tabs) return vsh_make(1, 90);
    if (sigs >= 32 * tabs) return vsh_make(3, 30);
    if (sigs >= 9 * tabs) return vsh_make(6, 15);
    vsh_shape s = vsh_make(VSH_ROWS, VSH_CHUNKS);
    s.quads = KTAB_QUADS;
    return s;
}
// On entry slots 0..3 hold A (all four coordinates valid).
GD void s_build_key_tables(sref sb, const wtab<1> &t) {
    const spt p = {s_slot(sb, 0), s_slot(sb, 1), s_slot(sb, 2), s_slot(sb, 3)};
    const swk w = {s_slot(sb, 4), s_slot(sb, 5), s_slot(sb, 6)};
    const int save = VSH_CHUNKS * WINDOW_NTABLE + 1;       /* A_c parked here while its table is built (the builder clobbers p) */
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int c = 0; c < VSH_CHUNKS; c++) {
        s_stg<1>(t.coord(save, 0), p.x); s_stg<1>(t.coord(save, 1), p.y); s_stg<1>(t.coord(save, 2), p.z); s_stg<1>(t.coord(save, 3), p.t);
        wtab<1> tc;
        tc.base = t.base + (size_t)c * WINDOW_NTABLE * 16;  /* its scratch entry 16 is entry 0 of the next column, written later */
        s_prepare_fixed_window<1>(p, w, tc);
        if (c == VSH_CHUNKS - 1) break;
        s_ldg<1>(p.x, t.coord(save, 0)); s_ldg<1>(p.y, t.coord(save, 1)); s_ldg<1>(p.z, t.coord(save, 2));
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (int j = 0; j < VSH_SHIFT - 1; j++) s_pt_double(p, w, true);
        s_pt_double(p, w, false);
    }
}
// The same tables in two steps, for batches (verify_dev): the doubling chain is inherently serial -- one lane per key -- but the ten
// column tables are independent once their base points A_c exist, so they are built by ten lanes per key.
//   step 1 (s_key_column_bases): A_c = 2^(45c) A for c = 0..9, parked as raw X, Y, Z, T in the LAST entry of column c
//   step 2 (s_build_key_column): one lane per (key, column) loads A_c and fills the column's 16 entries (the parked point is
//          overwritten last); pniels(2 A_c), which the builder reads back, goes to the lane's own scratch table.
GD void s_key_column_bases(sref sb, const wtab<1> &t, int ncols = VSH_CHUNKS, int shift = VSH_SHIFT) {
    const spt p = {s_slot(sb, 0), s_slot(sb, 1), s_slot(sb, 2), s_slot(sb, 3)};
    const swk w = {s_slot(sb, 4), s_slot(sb, 5), s_slot(sb, 6)};
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int c = 0; c < ncols; c++) {
        const int park = c * WINDOW_NTABLE + WINDOW_NTABLE - 1;
        s_stg<1>(t.coord(park, 0), p.x); s_stg<1>(t.coord(park, 1), p.y); s_stg<1>(t.coord(park, 2), p.z); s_stg<1>(t.coord(park, 3), p.t);
        if (c == ncols - 1) break;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (int j = 0; j < shift - 1; j++) s_pt_double(p, w, true);
        s_pt_double(p, w, false);
    }
}
GD void s_build_key_column(sref sb, const wtab<1> &t, int c, const wtab<1> &scratch) {
    const spt p = {s_slot(sb, 0), s_slot(sb, 1), s_slot(sb, 2), s_slot(sb, 3)};
    const swk w = {s_slot(sb, 4), s_slot(sb, 5), s_slot(sb, 6)};
    wtab<1> tc;
    tc.base = t.base + (size_t)c * WINDOW_NTABLE * 16;
    const int park = WINDOW_NTABLE - 1;
    s_ldg<1>(p.x, tc.coord(park, 0)); s_ldg<1>(p.y, tc.coord(park, 1)); s_ldg<1>(p.z, tc.coord(park, 2)); s_ldg<1>(p.t, tc.coord(park, 3));
    s_pt_to_pniels_negc_g<1>(tc, 0, p, w);
    s_pt_double(p, w, false);
    s_pt_to_pniels_negc_g<1>(scratch, 0, p, w);               /* pniels(2 A_c) */
    s_pt_add_pniels_g<1>(p, w, tc, 0, 0, ~0u, false);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int i = 1; i < WINDOW_NTABLE; i++) {
        s_pt_to_pniels_negc_g<1>(tc, i, p, w);
        if (i != WINDOW_NTABLE - 1) s_pt_add_pniels_g<1>(p, w, scratch, 0, 0, ~0u, false);
    }
}
// Key sets, flat layout (goldilocks_b200_keyset_policy): a key that serves many calls can afford a table PER DIGIT POSITION -- 90 columns
// of 16 affine entries, entry 16 k + e = (2e+1) 2^(5k) A, 369 KB per key -- and then a signature under it costs 90 + 25 additions and not
// one doubling: what decision 17 does for the fixed base, done for the key.
#define KSET_COLS 90
#define KSET_QUADS (KSET_COLS * WINDOW_NTABLE * 16)
GD wtab<1> kset_of(uint4 *ktabs, size_t table) { wtab<1> t; t.base = ktabs + table * KSET_QUADS; return t; }
// need_t: T of the result too (point sets return the point; verification only compares it).
GD void s_verify_flat_key(sref sb, const sc &scalar1, const sc &scalar2, const niels *wide, const wtab<1> &kt, bool need_t = false) {
    const spt p = {s_slot(sb, 0), s_slot(sb, 1), s_slot(sb, 2), s_slot(sb, 3)};
    const swk w = {s_slot(sb, 4), s_slot(sb, 5), s_slot(sb, 6)};
    sc s1x, s2x;
    sc_recode_signed(s1x, scalar1);
    sc_recode_signed(s2x, scalar2);
    s_pt_set_identity(p);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int k = 0; k < KSET_COLS; k++) {
        uint32_t bits2 = sc_window5(s2x, k * WINDOW_BITS);
        const gmask_t inv2 = (gmask_t)((int32_t)(bits2 >> (WINDOW_BITS - 1)) - 1);
        bits2 ^= inv2;
        const int e2 = k * WINDOW_NTABLE + (int)(bits2 & (WINDOW_NTABLE - 1));
        s_pt_add_niels_g<1>(p, w, kt.coord(e2, 0), kt.coord(e2, 1), kt.coord(e2, 2), inv2, ~inv2, false);
    }
    s_add_fixed_base(p, w, s1x, wide, need_t);
}
// combo (slots 0..3) = scalar1*B + scalar2*A with A's tables in `kt`; `wide` = the init-time tables of the fixed base.
// AFFINE: the entries have been divided by their z (key sets, LaneKeysetNormalize): 7 multiplications per addition instead of 8.
// need_t as in s_verify_flat_key.
template <bool AFFINE = false>
GD void s_verify_shared_key(sref sb, const sc &scalar1, const sc &scalar2, const niels *wide, const wtab<1> &kt, int rows = VSH_ROWS, int chunks = VSH_CHUNKS,
                            bool need_t = false) {
    const spt p = {s_slot(sb, 0), s_slot(sb, 1), s_slot(sb, 2), s_slot(sb, 3)};
    const swk w = {s_slot(sb, 4), s_slot(sb, 5), s_slot(sb, 6)};
    sc s1x, s2x;
    sc_recode_signed(s1x, scalar1);
    sc_recode_signed(s2x, scalar2);
    s_pt_set_identity(p);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int r = rows - 1; r >= 0; r--) {
        if (r != rows - 1) {
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
            for (int j = 0; j < WINDOW_BITS - 1; j++) s_pt_double(p, w, true);
            s_pt_double(p, w, false);
        }
        int c_last = (89 - r) / rows;                       /* last column with a digit in this row */
        if (c_last > chunks - 1) c_last = chunks - 1;
        const int last_k = rows * c_last + r;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (int c = 0; c < chunks; c++) {
            const int k = rows * c + r;
            if (k > 89) break;
            const bool row_ends = r != 0 && k == last_k;    /* a doubling follows: T is not needed */
            uint32_t bits2 = sc_window5(s2x, k * WINDOW_BITS);
            const gmask_t inv2 = (gmask_t)((int32_t)(bits2 >> (WINDOW_BITS - 1)) - 1);
            bits2 ^= inv2;
            const int e2 = c * WINDOW_NTABLE + (int)(bits2 & (WINDOW_NTABLE - 1));
            if (AFFINE) s_pt_add_niels_g<1>(p, w, kt.coord(e2, 0), kt.coord(e2, 1), kt.coord(e2, 2), inv2, ~inv2, row_ends);
            else s_pt_add_pniels_g<1>(p, w, kt, e2, inv2, ~inv2, row_ends);
        }
    }
    s_add_fixed_base(p, w, s1x, wide, need_t);
}

// ---------------------------------------------------------------------------------------------
// Fixed-base signed comb, constant time -- reference goldilocks.c:830-877 (same digits, table and
// operation order as comb_scalarmul in algos.cuh).  7 slots: X,Y,Z,T and three temporaries; the three
// coordinates of the selected entry are fetched just in time (a and b, then c) into slots that are dead at
// that point, the conditional negation of the entry is a handle selection (goldilocks.c:271-278).
// ---------------------------------------------------------------------------------------------
#define COMB_NSLOTS 7
// p += (+-) entry idx of a 16-entry row of affine niels, constant time in idx and the sign.  No extra
// slots: once y+x and y-x are taken, X and Y are dead until the end and receive the looked-up a and b
// (then c); (goldilocks.c:315-359 with the sign as a handle selection, 271-278).
GD void s_pt_add_niels_ct(const spt &p, const swk &w, const niels *row, uint32_t idx, gmask_t neg, bool before_double) {
    const int stride = (int)(sizeof(niels) / sizeof(uint4));
    s_addsub(w.t1, w.t0, p.y, p.x);                      /* y+x ; y-x */
    s_lookup_ct<true, 1>(p.x, gq(&row->a), stride, 1 << (COMB_T - 1), idx);
    s_lookup_ct<true, 1>(p.y, gq(&row->b), stride, 1 << (COMB_T - 1), idx);
    s_mul(w.t0, w.t0, s_sel(p.x, p.y, neg));             /* a  = e.a (y-x) */
    s_mul(w.t1, w.t1, s_sel(p.y, p.x, neg));             /* dy = e.b (y+x) */
    s_lookup_ct<true, 1>(p.y, gq(&row->c), stride, 1 << (COMB_T - 1), idx);
    s_mul(p.x, p.t, p.y);                                /* x  = e.c t */
    s_addsub(w.t2, w.t1, w.t1, w.t0);                    /* c = dy + a ; b = dy - a */
    s_addsub(w.t0, p.y, p.z, p.x);                       /* v = z + x ; u = z - x */
    s_mul(p.z, w.t0, p.y);
    s_mul(p.x, s_sel(p.y, w.t0, neg), w.t1);
    s_mul(p.y, s_sel(w.t0, p.y, neg), w.t2);
    if (!before_double) s_mul(p.t, w.t1, w.t2);
}
// out = scalar * B over the doubling-free table `win` (WIN_ROWS rows of 16, algos.cuh): 90 constant-time
// additions, no doublings.  Digit j of the signed recoding = bits [5j, 5j+5) of (scalar + adj)/2.
GD void s_comb_scalarmul(sref sb, const niels *win, const sc &scalar) {
    const spt p = {s_slot(sb, 0), s_slot(sb, 1), s_slot(sb, 2), s_slot(sb, 3)};
    const swk w = {s_slot(sb, 4), s_slot(sb, 5), s_slot(sb, 6)};
    sc s1x;
    sc_recode_signed(s1x, scalar);
    { /* accumulator = identity; the unified addition law takes the first entry from there */
        gf v;
        gf_set_zero(v); s_st(p.x, v); s_st(p.t, v);
        gf_set_ui(v, 1); s_st(p.y, v); s_st(p.z, v);
    }
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int j = 0; j < WIN_ROWS; j++) {
        uint32_t tab = sc_bits(s1x, COMB_T * j, COMB_T);
        const gmask_t invert = (gmask_t)((int32_t)(tab >> (COMB_T - 1)) - 1);
        tab ^= invert;
        tab &= (1u << (COMB_T - 1)) - 1;
        s_pt_add_niels_ct(p, w, win + 16 * j, tab, invert, false);
    }
}

// ---------------------------------------------------------------------------------------------
// Encoders that follow a comb multiplication (slots 0..3 = the point, 9 slots available).  The one
// inversion each needs is shared by four lanes on the device (s_block_invert4); inverse of 0 is 0 as in
// the reference's gf_invert (goldilocks.c:69-80).
// ---------------------------------------------------------------------------------------------
// slot `zin` <- z or 1 when z == 0; returns the nonzero mask
GD gmask_t s_nonzero_or_one(sref zin, sref z) {
    gf v, one;
    s_ld(v, z);
    const gmask_t nz = ~gf_is_zero(v);
    gf_set_ui(one, 1);
    gf_cond_sel(v, one, v, nz);
    s_st(zin, v);
    return nz;
}
// slot 4 <- 1 / slot 5 (slot 5 nonzero); slots 0..2 are scratch, slots 3 and 6 are preserved
GD void s_invert_5_to_4(sref sb) {
#if defined(__CUDA_ARCH__)
    s_block_invert4(sb, 5, 4);
#else
    s_invert(s_slot(sb, 4), s_slot(sb, 5), s_slot(sb, 1), s_slot(sb, 2));
#endif
}
// RFC 8032 encoding after the 4-isogeny back to the untwisted curve (goldilocks.c:905-946):
// yw = canonical y words, xsign = low bit of x.
GD void s_encode_like_eddsa(uint32_t yw[14], uint32_t &xsign, sref sb) {
    const spt p = {s_slot(sb, 0), s_slot(sb, 1), s_slot(sb, 2), s_slot(sb, 3)};
    const sref t0 = s_slot(sb, 4), t1 = s_slot(sb, 5), t2 = s_slot(sb, 6), xs = s_slot(sb, 6), ys = s_slot(sb, 3);
    s_sqr(t0, p.x);                    /* x^2 */
    s_sqr(t1, p.y);                    /* y^2 */
    s_sqr_sum(t2, p.y, p.x);
    s_addsub(p.t, t1, t1, t0);         /* u = y^2 + x^2 ; z = y^2 - x^2 */
    s_sub(t2, t2, p.t);                /* 2xy */
    s_sqr2_sub(t0, p.z, t1);           /* t = 2 z^2 - (y^2 - x^2) */
    s_mul(xs, t0, t2);                 /* x = t * 2xy        (t2 = slot 6 is read before it is written) */
    s_mul(p.z, p.t, t0);               /* z = u t */
    s_mul(ys, t1, p.t);                /* y = (y^2 - x^2) u  (in place over u, slot 3) */
    const gmask_t nz = s_nonzero_or_one(s_slot(sb, 5), p.z);
    s_invert_5_to_4(sb);
    s_mul(xs, xs, s_slot(sb, 4));      /* affine x */
    s_mul(ys, ys, s_slot(sb, 4));      /* affine y */
    gf x, y, zero;
    gf_set_zero(zero);
    s_ld(x, xs); gf_cond_sel(x, zero, x, nz);
    s_ld(y, ys); gf_cond_sel(y, zero, y, nz);
    gf_to_words(yw, y);
    xsign = gf_lobit(x) & 1u;
}
// u = (y/x)^2 (goldilocks.c:1104-1115)
GD void s_encode_like_x448(uint32_t uw[14], sref sb) {
    const sref xs = s_slot(sb, 6);
    s_copy(xs, s_slot(sb, 1));         /* y survives the inversion in slot 6 */
    const gmask_t nz = s_nonzero_or_one(s_slot(sb, 5), s_slot(sb, 0));
    s_invert_5_to_4(sb);
    s_mul(xs, xs, s_slot(sb, 4));
    s_sqr(xs, xs);
    gf u, zero;
    gf_set_zero(zero);
    s_ld(u, xs); gf_cond_sel(u, zero, u, nz);
    gf_to_words(uw, u);
}

// ---------------------------------------------------------------------------------------------
// Variable-base scalar multiplication, constant time -- reference goldilocks.c:405-465 (and 467-541
// for two bases): signed 5-bit fixed windows over this lane's own table of 16 odd multiples in global
// memory; every lookup scans the whole table with masks (s_lookup_ct_rw), the sign is a handle
// selection.  7 slots; the accumulator starts from the identity (unified addition law) instead of
// pniels_to_pt of the first digit -- same group element.
// ---------------------------------------------------------------------------------------------
#define WINDOW_NSLOTS 7
// p += (+-) table[idx], constant time in idx and the sign (`neg` all-ones = subtract).  The table is in
// the warp-interleaved layout, so each of the 4 x 16 x 4 loads of the scan is one coalesced 512-byte row.
GD void s_pt_add_pniels_ct(const spt &p, const swk &w, const wtab<32> &t, uint32_t idx, gmask_t neg, bool before_double) {
    const int es = wtab<32>::ESTRIDE;
    s_lookup_ct<false, 32>(w.t2, t.coord(0, 3), es, WINDOW_NTABLE, idx);
    s_mul(p.z, p.z, w.t2);
    s_addsub(w.t1, w.t0, p.y, p.x);                      /* X and Y are dead from here: they hold a and b, then c */
    s_lookup_ct<false, 32>(p.x, t.coord(0, 0), es, WINDOW_NTABLE, idx);
    s_lookup_ct<false, 32>(p.y, t.coord(0, 1), es, WINDOW_NTABLE, idx);
    s_mul(w.t0, w.t0, s_sel(p.x, p.y, neg));
    s_mul(w.t1, w.t1, s_sel(p.y, p.x, neg));
    s_lookup_ct<false, 32>(p.y, t.coord(0, 2), es, WINDOW_NTABLE, idx);   /* stored negated: neg_c = ~neg */
    s_mul(p.x, p.t, p.y);
    s_addsub(w.t2, w.t1, w.t1, w.t0);
    s_addsub(w.t0, p.y, p.z, p.x);
    s_mul(p.z, w.t0, p.y);
    s_mul(p.x, s_sel(w.t0, p.y, neg), w.t1);             /* x = (neg_c ? v : u) b, neg_c = ~neg */
    s_mul(p.y, s_sel(p.y, w.t0, neg), w.t2);
    if (!before_double) s_mul(p.t, w.t1, w.t2);
}
GD void s_window_digit(uint32_t &idx, gmask_t &neg, const sc &s1x, int i) {
    uint32_t bits = sc_window5(s1x, i);
    neg = (gmask_t)((int32_t)(bits >> (WINDOW_BITS - 1)) - 1);
    bits ^= neg;
    idx = bits & (WINDOW_NTABLE - 1);
}
// slots 0..3 <- sum of the signed 5-bit digits of s1x (already recoded) times the table's odd multiples
GD void s_window_mainloop(const spt &p, const swk &w, const sc &s1x, const wtab<32> &multiples) {
    s_pt_set_identity(p);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int k = 89; k >= 0; k--) {
        if (k != 89) {
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
            for (int j = 0; j < WINDOW_BITS - 1; j++) s_pt_double(p, w, true);
            s_pt_double(p, w, false);
        }
        uint32_t idx; gmask_t neg;
        s_window_digit(idx, neg, s1x, k * WINDOW_BITS);
        s_pt_add_pniels_ct(p, w, multiples, idx, neg, k != 0);
    }
}
// slots 0..3: base on entry, scalar * base on exit
GD void s_window_scalarmul(sref sb, const sc &scalar, const wtab<32> &multiples) {
    const spt p = {s_slot(sb, 0), s_slot(sb, 1), s_slot(sb, 2), s_slot(sb, 3)};
    const swk w = {s_slot(sb, 4), s_slot(sb, 5), s_slot(sb, 6)};
    sc s1x;
    sc_recode_signed(s1x, scalar);
    s_prepare_fixed_window<32>(p, w, multiples);
    s_window_mainloop(p, w, s1x, multiples);
}
// slots 0..3: base b on entry and the result scalarb*b + scalarc*c on exit; `c_abi` is loaded when needed
template <class LoadC>
GD void s_window_double_scalarmul(sref sb, const sc &scalarb, const sc &scalarc, LoadC load_c, const wtab<32> &multiples1, const wtab<32> &multiples2) {
    const spt p = {s_slot(sb, 0), s_slot(sb, 1), s_slot(sb, 2), s_slot(sb, 3)};
    const swk w = {s_slot(sb, 4), s_slot(sb, 5), s_slot(sb, 6)};
    sc s1x, s2x;
    sc_recode_signed(s1x, scalarb);
    sc_recode_signed(s2x, scalarc);
    s_prepare_fixed_window<32>(p, w, multiples1);
    load_c(sb);
    s_prepare_fixed_window<32>(p, w, multiples2);
    s_pt_set_identity(p);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int k = 89; k >= 0; k--) {
        if (k != 89) {
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
            for (int j = 0; j < WINDOW_BITS - 1; j++) s_pt_double(p, w, true);
            s_pt_double(p, w, false);
        }
        uint32_t idx; gmask_t neg;
        s_window_digit(idx, neg, s1x, k * WINDOW_BITS);
        s_pt_add_pniels_ct(p, w, multiples1, idx, neg, false);
        s_window_digit(idx, neg, s2x, k * WINDOW_BITS);
        s_pt_add_pniels_ct(p, w, multiples2, idx, neg, k != 0);
    }
}

// ---------------------------------------------------------------------------------------------
// Fixed-base comb over a caller-supplied (5,5,18) table (goldilocks_448_precompute output), constant
// time -- reference goldilocks.c:830-877 verbatim: 18 rounds x 5 combs, 17 doublings + 90 additions.
// The library's own base-point path uses the doubling-free table instead (s_comb_scalarmul).
// ---------------------------------------------------------------------------------------------
GD void s_comb_scalarmul_table(sref sb, const niels *table, const sc &scalar) {
    const spt p = {s_slot(sb, 0), s_slot(sb, 1), s_slot(sb, 2), s_slot(sb, 3)};
    const swk w = {s_slot(sb, 4), s_slot(sb, 5), s_slot(sb, 6)};
    sc s1x;
    sc_recode_signed(s1x, scalar);
    s_pt_set_identity(p);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    for (int i = COMB_S - 1; i >= 0; i--) {
        if (i != COMB_S - 1) s_pt_double(p, w, false);
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (int j = 0; j < COMB_N; j++) {
            uint32_t tab = 0;
#pragma unroll
            for (int k = 0; k < COMB_T; k++) {
                const int bit = i + COMB_S * (k + j * COMB_T);
                if (bit < GOLDILOCKS_SCALAR_BITS_) tab |= sc_bit(s1x, bit) << k;
            }
            const gmask_t invert = (gmask_t)((int32_t)(tab >> (COMB_T - 1)) - 1);
            tab ^= invert;
            tab &= (1u << (COMB_T - 1)) - 1;
            s_pt_add_niels_ct(p, w, table + (j << (COMB_T - 1)), tab, invert, j == COMB_N - 1 && i != 0);
        }
    }
}
