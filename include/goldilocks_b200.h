/*
 * goldilocks_b200.h -- C ABI of the B200-native batched Ed448-Goldilocks engine.
 *
 * This is the drop-in boundary (SURVEY.md section 8(b)).  It has two halves:
 *
 *  1. LEGACY single-element entry points with exactly the names, argument order, struct sizes
 *     and return conventions of libgoldilocks' own public headers
 *     (reference: src/public_include/goldilocks/{common,point_448,ed448}.h).  Each one runs a
 *     batch of one on the GPU; there is no CPU fallback.
 *
 *  2. `*_batch` entry points: the same operation over n independent elements.  Every
 *     per-element argument of the legacy call becomes a packed array (element i at
 *     base + i*sizeof(element)), `n` is appended, fallible operations gain a per-element
 *     `goldilocks_error_t status[n]`, and variable-length messages are passed as one arena plus
 *     `msg_off[n+1]` byte offsets.  All pointers are HOST pointers unless the function name ends
 *     in `_dev`.  A batch call returns GOLDILOCKS_SUCCESS when the device executed the batch and
 *     GOLDILOCKS_FAILURE on a CUDA error (see goldilocks_b200_last_error()).
 *
 * Types below are layout-compatible with the reference's x86_64 ABI (GOLDILOCKS_WORD_BITS 64):
 *   gf_448_s       64 bytes, 8 x u64 limbs radix 2^56, aligned(32)   (reference f_field.h:23-27)
 *   point_s        256 bytes = x,y,z,t                                (reference point_448.h:66-70)
 *   scalar_s       56 bytes, 7 x u64, value < q                       (reference point_448.h:82-86)
 * Field limbs are only defined mod p: the library accepts any limb values below 2^60 and always
 * emits canonical limbs (< 2^56, value < p).
 *
 * The header is self-contained C99/C++ and pulls in no CUDA or torch types.
 */
#ifndef GOLDILOCKS_B200_H
#define GOLDILOCKS_B200_H 1

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GOLDILOCKS_B200_API __attribute__((visibility("default")))

/* ---- scalar types and sizes (reference common.h:51-85, point_448.h:23-63, ed448.h:24-52) ---- */
typedef uint64_t goldilocks_word_t;
typedef uint64_t goldilocks_bool_t;           /* all-ones = true, 0 = false */
typedef enum { GOLDILOCKS_SUCCESS = -1, GOLDILOCKS_FAILURE = 0 } goldilocks_error_t;

#define GOLDILOCKS_448_SCALAR_LIMBS 7
#define GOLDILOCKS_448_SCALAR_BITS 446
#define GOLDILOCKS_448_SER_BYTES 56
#define GOLDILOCKS_448_HASH_BYTES 56
#define GOLDILOCKS_448_SCALAR_BYTES 56
#define GOLDILOCKS_X448_PUBLIC_BYTES 56
#define GOLDILOCKS_X448_PRIVATE_BYTES 56
#define GOLDILOCKS_EDDSA_448_PUBLIC_BYTES 57
#define GOLDILOCKS_EDDSA_448_PRIVATE_BYTES 57
#define GOLDILOCKS_EDDSA_448_SIGNATURE_BYTES 114

typedef struct gf_448_s { goldilocks_word_t limb[8]; } __attribute__((aligned(32))) gf_448_s;
typedef struct goldilocks_448_point_s { gf_448_s x, y, z, t; } goldilocks_448_point_s, goldilocks_448_point_p[1];
typedef struct goldilocks_448_scalar_s { goldilocks_word_t limb[GOLDILOCKS_448_SCALAR_LIMBS]; } goldilocks_448_scalar_s, goldilocks_448_scalar_p[1];
/* Fixed-base table handle (reference goldilocks.c:59-66).  goldilocks_448_precomputed_base selects the
 * library's device-resident base-point tables; any other pointer must address a caller-allocated table of
 * goldilocks_448_sizeof_precomputed_s bytes filled by goldilocks_448_precompute(), byte-compatible with
 * the reference's (80 affine niels, canonical radix-2^56 limbs). */
typedef struct goldilocks_448_precomputed_s goldilocks_448_precomputed_s;
GOLDILOCKS_B200_API extern const size_t goldilocks_448_sizeof_precomputed_s, goldilocks_448_alignof_precomputed_s; /* point_448.h:79 */

GOLDILOCKS_B200_API extern const goldilocks_448_precomputed_s *goldilocks_448_precomputed_base;
GOLDILOCKS_B200_API extern const goldilocks_448_point_p goldilocks_448_point_base;       /* reference point_448.h:283 */
GOLDILOCKS_B200_API extern const goldilocks_448_point_p goldilocks_448_point_identity;   /* reference goldilocks.c:83 */
GOLDILOCKS_B200_API extern const goldilocks_448_scalar_p goldilocks_448_scalar_one, goldilocks_448_scalar_zero;
GOLDILOCKS_B200_API extern const uint8_t goldilocks_x448_base_point[GOLDILOCKS_X448_PUBLIC_BYTES]; /* goldilocks.c:39 */

/* ======================================================================================
 * 1. Legacy single-element entry points (batch of one on the GPU)
 * ====================================================================================== */
/* reference point_448.h:303-334 / goldilocks.c:178-258 */
GOLDILOCKS_B200_API void goldilocks_448_point_add(goldilocks_448_point_p sum, const goldilocks_448_point_p a, const goldilocks_448_point_p b);
GOLDILOCKS_B200_API void goldilocks_448_point_sub(goldilocks_448_point_p diff, const goldilocks_448_point_p a, const goldilocks_448_point_p b);
GOLDILOCKS_B200_API void goldilocks_448_point_double(goldilocks_448_point_p two_a, const goldilocks_448_point_p a);
GOLDILOCKS_B200_API void goldilocks_448_point_negate(goldilocks_448_point_p nega, const goldilocks_448_point_p a);
/* reference point_448.h:241-264 / goldilocks.c:136-176 */
GOLDILOCKS_B200_API void goldilocks_448_point_encode(uint8_t ser[56], const goldilocks_448_point_p pt);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_decode(goldilocks_448_point_p pt, const uint8_t ser[56], goldilocks_bool_t allow_identity);
/* reference point_448.h:270-281,555-563 / goldilocks.c:644-673 */
GOLDILOCKS_B200_API goldilocks_bool_t goldilocks_448_point_eq(const goldilocks_448_point_p a, const goldilocks_448_point_p b);
GOLDILOCKS_B200_API goldilocks_bool_t goldilocks_448_point_valid(const goldilocks_448_point_p a);
/* reference point_448.h:355-359 / goldilocks.c:405-465 (constant time) */
GOLDILOCKS_B200_API void goldilocks_448_point_scalarmul(goldilocks_448_point_p scaled, const goldilocks_448_point_p base, const goldilocks_448_scalar_p scalar);
/* reference point_448.h:477-481 / goldilocks.c:830-877 (constant time fixed-base comb) */
GOLDILOCKS_B200_API void goldilocks_448_precomputed_scalarmul(goldilocks_448_point_p scaled, const goldilocks_448_precomputed_s *base, const goldilocks_448_scalar_p scalar);
/* reference point_448.h:494-500 / goldilocks.c:467-541 (constant time) */
GOLDILOCKS_B200_API void goldilocks_448_point_double_scalarmul(goldilocks_448_point_p combo, const goldilocks_448_point_p base1, const goldilocks_448_scalar_p scalar1, const goldilocks_448_point_p base2, const goldilocks_448_scalar_p scalar2);
/* reference point_448.h:542-547 / goldilocks.c:1260-1330 (variable time, public inputs only) */
GOLDILOCKS_B200_API void goldilocks_448_base_double_scalarmul_non_secret(goldilocks_448_point_p combo, const goldilocks_448_scalar_p scalar1, const goldilocks_448_point_p base2, const goldilocks_448_scalar_p scalar2);
/* reference point_448.h:510-531 / goldilocks.c:543-642 (constant time): a1 = scalar1*base, a2 = scalar2*base */
GOLDILOCKS_B200_API void goldilocks_448_point_dual_scalarmul(goldilocks_448_point_p a1, goldilocks_448_point_p a2, const goldilocks_448_point_p base, const goldilocks_448_scalar_p scalar1, const goldilocks_448_scalar_p scalar2);
/* reference point_448.h:371-384 / goldilocks.c:888-903: decode, scalarmul, encode; a failed decode multiplies the base point
 * (or, with short_circuit, returns at once without writing `scaled`) */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_direct_scalarmul(uint8_t scaled[56], const uint8_t base[56], const goldilocks_448_scalar_p scalar, goldilocks_bool_t allow_identity, goldilocks_bool_t short_circuit);
/* reference point_448.h:455-466,483-486 / goldilocks.c:757-818,1337-1343 */
GOLDILOCKS_B200_API void goldilocks_448_precompute(goldilocks_448_precomputed_s *table, const goldilocks_448_point_p base);
GOLDILOCKS_B200_API void goldilocks_448_precomputed_destroy(goldilocks_448_precomputed_s *table);
/* reference point_448.h:565-594 / goldilocks.c:675-702,879-886 */
GOLDILOCKS_B200_API void goldilocks_448_point_debugging_torque(goldilocks_448_point_p q, const goldilocks_448_point_p p);
GOLDILOCKS_B200_API void goldilocks_448_point_debugging_pscale(goldilocks_448_point_p q, const goldilocks_448_point_p p, const uint8_t factor[56]);
GOLDILOCKS_B200_API void goldilocks_448_point_cond_sel(goldilocks_448_point_p out, const goldilocks_448_point_p a, const goldilocks_448_point_p b, goldilocks_bool_t pick_b);
GOLDILOCKS_B200_API void goldilocks_448_point_destroy(goldilocks_448_point_p point);
/* reference point_448.h:647-664 / elligator.c:32-94 */
GOLDILOCKS_B200_API void goldilocks_448_point_from_hash_nonuniform(goldilocks_448_point_p pt, const uint8_t hashed_data[56]);
GOLDILOCKS_B200_API void goldilocks_448_point_from_hash_uniform(goldilocks_448_point_p pt, const uint8_t hashed_data[112]);
/* reference point_448.h:666-709 / elligator.c:104-164: one preimage of pt under the maps above, chosen by `which`
 * (bit 0 sign of s, bit 1 alternative x, bit 2 sign of r0); FAILURE when that branch has no preimage.  The uniform
 * variant reads partial_hash[56..111] and writes partial_hash[0..55]. */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_invert_elligator_nonuniform(uint8_t recovered_hash[56], const goldilocks_448_point_p pt, uint32_t which);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_invert_elligator_uniform(uint8_t partial_hash[112], const goldilocks_448_point_p pt, uint32_t which);
/* reference ed448.h:215-232 / goldilocks.c:905-1004 ; point_448.h:430-434 / goldilocks.c:1104-1115 */
GOLDILOCKS_B200_API void goldilocks_448_point_mul_by_ratio_and_encode_like_eddsa(uint8_t enc[57], const goldilocks_448_point_p p);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_decode_like_eddsa_and_mul_by_ratio(goldilocks_448_point_p p, const uint8_t enc[57]);
GOLDILOCKS_B200_API void goldilocks_448_point_mul_by_ratio_and_encode_like_x448(uint8_t out[56], const goldilocks_448_point_p p);
/* reference point_448.h:398-402,445-448 / goldilocks.c:1006-1076,1117-1141 */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_x448(uint8_t out[56], const uint8_t base[56], const uint8_t scalar[56]);
GOLDILOCKS_B200_API void goldilocks_x448_derive_public_key(uint8_t out[56], const uint8_t scalar[56]);
/* reference ed448.h:61-165 / eddsa.c:98-306 */
GOLDILOCKS_B200_API void goldilocks_ed448_derive_secret_scalar(goldilocks_448_scalar_p secret, const uint8_t privkey[57]);
GOLDILOCKS_B200_API void goldilocks_ed448_derive_public_key(uint8_t pubkey[57], const uint8_t privkey[57]);
GOLDILOCKS_B200_API void goldilocks_ed448_sign(uint8_t signature[114], const uint8_t privkey[57], const uint8_t pubkey[57], const uint8_t *message, size_t message_len, uint8_t prehashed, const uint8_t *context, uint8_t context_len);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_ed448_verify(const uint8_t signature[114], const uint8_t pubkey[57], const uint8_t *message, size_t message_len, uint8_t prehashed, const uint8_t *context, uint8_t context_len);
/* reference ed448.h:234-262 / goldilocks.c:1079-1103, eddsa.c:83-95 */
GOLDILOCKS_B200_API void goldilocks_ed448_convert_public_key_to_x448(uint8_t x[56], const uint8_t ed[57]);
GOLDILOCKS_B200_API void goldilocks_ed448_convert_private_key_to_x448(uint8_t x[56], const uint8_t ed[57]);
/* Streaming SHA-3 / SHAKE objects (reference shake.h:27-120, keccak_internal.h, shake.c:89-250) and the Ed448ph
 * entry points built on them (ed448.h:36-46,107-137,170-190 / eddsa.c:76-80,232-251,309-329).  The sponge object
 * is the reference's (26 x u64, caller-owned); every Keccak-f runs on the device, one round trip per call --
 * bulk hashing belongs in goldilocks_shake256_hash_batch. */
typedef struct goldilocks_keccak_sponge_s { uint64_t opaque[26]; } goldilocks_keccak_sponge_s, goldilocks_keccak_sponge_p[1];
struct goldilocks_kparams_s { uint8_t position, flags, rate, start_round, pad, rate_pad, max_out, remaining; };
GOLDILOCKS_B200_API extern const struct goldilocks_kparams_s GOLDILOCKS_SHAKE128_params_s, GOLDILOCKS_SHAKE256_params_s,
    GOLDILOCKS_SHA3_224_params_s, GOLDILOCKS_SHA3_256_params_s, GOLDILOCKS_SHA3_384_params_s, GOLDILOCKS_SHA3_512_params_s;
GOLDILOCKS_B200_API void goldilocks_sha3_init(goldilocks_keccak_sponge_p sponge, const struct goldilocks_kparams_s *params);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_sha3_update(struct goldilocks_keccak_sponge_s *sponge, const uint8_t *in, size_t len);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_sha3_output(goldilocks_keccak_sponge_p sponge, uint8_t *out, size_t len);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_sha3_final(goldilocks_keccak_sponge_p sponge, uint8_t *out, size_t len);
GOLDILOCKS_B200_API void goldilocks_sha3_reset(goldilocks_keccak_sponge_p sponge);
GOLDILOCKS_B200_API void goldilocks_sha3_destroy(goldilocks_keccak_sponge_p sponge);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_sha3_hash(uint8_t *out, size_t outlen, const uint8_t *in, size_t inlen, const struct goldilocks_kparams_s *params);
GOLDILOCKS_B200_API size_t goldilocks_sha3_default_output_bytes(const goldilocks_keccak_sponge_p sponge);
GOLDILOCKS_B200_API size_t goldilocks_sha3_max_output_bytes(const goldilocks_keccak_sponge_p sponge);
/* Sponge-based CSPRNG (reference spongerng.h:22-87 / spongerng.c:92-205): a SHAKE256 object that is re-keyed after every
 * request.  Host-side composition of the streaming calls above, so its Keccak-f permutations run on the device too.  A
 * deterministic generator reproduces the reference's byte stream exactly (the reference's tests draw their inputs from it);
 * a non-deterministic one stirs in 32 bytes of OS entropy before each request. */
typedef struct { goldilocks_keccak_sponge_p sponge; } goldilocks_keccak_prng_s;
typedef goldilocks_keccak_prng_s goldilocks_keccak_prng_p[1];
GOLDILOCKS_B200_API void goldilocks_spongerng_init_from_buffer(goldilocks_keccak_prng_p prng, const uint8_t *in, size_t len, int deterministic);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_spongerng_init_from_file(goldilocks_keccak_prng_p prng, const char *file, size_t len, int deterministic);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_spongerng_init_from_dev_urandom(goldilocks_keccak_prng_p prng);
GOLDILOCKS_B200_API void goldilocks_spongerng_next(goldilocks_keccak_prng_p prng, uint8_t *out, size_t len);
GOLDILOCKS_B200_API void goldilocks_spongerng_stir(goldilocks_keccak_prng_p prng, const uint8_t *in, size_t len);
GOLDILOCKS_B200_API void goldilocks_ed448_prehash_init(goldilocks_keccak_sponge_p hash);
GOLDILOCKS_B200_API void goldilocks_ed448_sign_prehash(uint8_t signature[114], const uint8_t privkey[57], const uint8_t pubkey[57], const goldilocks_keccak_sponge_p hash, const uint8_t *context, uint8_t context_len);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_ed448_verify_prehash(const uint8_t signature[114], const uint8_t pubkey[57], const goldilocks_keccak_sponge_p hash, const uint8_t *context, uint8_t context_len);
/* reference point_448.h:113-233 / scalar.c */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_scalar_invert(goldilocks_448_scalar_p out, const goldilocks_448_scalar_p a);
GOLDILOCKS_B200_API goldilocks_bool_t goldilocks_448_scalar_eq(const goldilocks_448_scalar_p a, const goldilocks_448_scalar_p b);
GOLDILOCKS_B200_API void goldilocks_448_scalar_cond_sel(goldilocks_448_scalar_p out, const goldilocks_448_scalar_p a, const goldilocks_448_scalar_p b, goldilocks_bool_t pick_b);
GOLDILOCKS_B200_API void goldilocks_448_scalar_set_unsigned(goldilocks_448_scalar_p out, uint64_t a);
GOLDILOCKS_B200_API void goldilocks_448_scalar_destroy(goldilocks_448_scalar_p scalar);
/* reference common.h:98-114 / utils.c */
GOLDILOCKS_B200_API void goldilocks_bzero(void *data, size_t size);
GOLDILOCKS_B200_API goldilocks_bool_t goldilocks_memeq(const void *data1, const void *data2, size_t size);
GOLDILOCKS_B200_API void goldilocks_448_scalar_add(goldilocks_448_scalar_p out, const goldilocks_448_scalar_p a, const goldilocks_448_scalar_p b);
GOLDILOCKS_B200_API void goldilocks_448_scalar_sub(goldilocks_448_scalar_p out, const goldilocks_448_scalar_p a, const goldilocks_448_scalar_p b);
GOLDILOCKS_B200_API void goldilocks_448_scalar_mul(goldilocks_448_scalar_p out, const goldilocks_448_scalar_p a, const goldilocks_448_scalar_p b);
GOLDILOCKS_B200_API void goldilocks_448_scalar_halve(goldilocks_448_scalar_p out, const goldilocks_448_scalar_p a);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_scalar_decode(goldilocks_448_scalar_p out, const uint8_t ser[56]);
GOLDILOCKS_B200_API void goldilocks_448_scalar_decode_long(goldilocks_448_scalar_p out, const uint8_t *ser, size_t ser_len);
GOLDILOCKS_B200_API void goldilocks_448_scalar_encode(uint8_t ser[56], const goldilocks_448_scalar_p s);

/* ======================================================================================
 * 2. Batched entry points (host pointers; element i at base + i*sizeof(element))
 * ====================================================================================== */
/* Field level, canonical 56-byte little-endian elements (BASELINE config 1).  Replaces the
 * reference's hidden gf_448_{mul,sqr,add,sub,isr} (f_field.h:66-84) composed with
 * gf_deserialize/gf_serialize (f_generic.c:19-68): out = serialize(op(deserialize(a), deserialize(b))).
 * Inputs >= p are taken mod p, like gf_deserialize's ignored-result callers. */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_gf_mul_batch(uint8_t *out, const uint8_t *a, const uint8_t *b, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_gf_sqr_batch(uint8_t *out, const uint8_t *a, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_gf_add_batch(uint8_t *out, const uint8_t *a, const uint8_t *b, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_gf_sub_batch(uint8_t *out, const uint8_t *a, const uint8_t *b, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_gf_mulw_batch(uint8_t *out, const uint8_t *a, uint32_t w, size_t n);
/* out = x^((p-3)/4), status = SUCCESS iff out^2 * x == 1 (f_arithmetic.c:14-47) */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_gf_isr_batch(uint8_t *out, goldilocks_error_t *status, const uint8_t *x, size_t n);
/* out = 1/x (0 for x = 0) (goldilocks.c:69-80) */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_gf_invert_batch(uint8_t *out, const uint8_t *x, size_t n);

/* Group level */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_add_batch(goldilocks_448_point_s *out, const goldilocks_448_point_s *a, const goldilocks_448_point_s *b, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_sub_batch(goldilocks_448_point_s *out, const goldilocks_448_point_s *a, const goldilocks_448_point_s *b, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_double_batch(goldilocks_448_point_s *out, const goldilocks_448_point_s *a, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_negate_batch(goldilocks_448_point_s *out, const goldilocks_448_point_s *a, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_eq_batch(goldilocks_bool_t *out, const goldilocks_448_point_s *a, const goldilocks_448_point_s *b, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_valid_batch(goldilocks_bool_t *out, const goldilocks_448_point_s *a, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_encode_batch(uint8_t *ser /*n*56*/, const goldilocks_448_point_s *pts, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_decode_batch(goldilocks_448_point_s *pts, goldilocks_error_t *status, const uint8_t *ser /*n*56*/, goldilocks_bool_t allow_identity, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_from_hash_nonuniform_batch(goldilocks_448_point_s *pts, const uint8_t *hashed /*n*56*/, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_from_hash_uniform_batch(goldilocks_448_point_s *pts, const uint8_t *hashed /*n*112*/, size_t n);
/* which[i] selects the branch of element i; the bytes of a failed element are written all the same (like the reference) */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_invert_elligator_nonuniform_batch(uint8_t *recovered /*n*56*/, goldilocks_error_t *status, const goldilocks_448_point_s *pts, const uint32_t *which, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_invert_elligator_uniform_batch(uint8_t *partial /*n*112, in/out*/, goldilocks_error_t *status, const goldilocks_448_point_s *pts, const uint32_t *which, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_scalarmul_batch(goldilocks_448_point_s *out, const goldilocks_448_point_s *base, const goldilocks_448_scalar_s *scalar, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_double_scalarmul_batch(goldilocks_448_point_s *out, const goldilocks_448_point_s *base1, const goldilocks_448_scalar_s *scalar1, const goldilocks_448_point_s *base2, const goldilocks_448_scalar_s *scalar2, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_precomputed_scalarmul_batch(goldilocks_448_point_s *out, const goldilocks_448_precomputed_s *base, const goldilocks_448_scalar_s *scalar, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_base_double_scalarmul_non_secret_batch(goldilocks_448_point_s *out, const goldilocks_448_scalar_s *scalar1, const goldilocks_448_point_s *base2, const goldilocks_448_scalar_s *scalar2, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_dual_scalarmul_batch(goldilocks_448_point_s *out1, goldilocks_448_point_s *out2, const goldilocks_448_point_s *base, const goldilocks_448_scalar_s *scalar1, const goldilocks_448_scalar_s *scalar2, size_t n);
/* status[i] = the decode's; with short_circuit the bytes of a failed element are left as the caller passed them */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_direct_scalarmul_batch(uint8_t *scaled /*n*56*/, goldilocks_error_t *status, const uint8_t *base /*n*56*/, const goldilocks_448_scalar_s *scalar, goldilocks_bool_t allow_identity, goldilocks_bool_t short_circuit, size_t n);
/* tables = n consecutive tables of goldilocks_448_sizeof_precomputed_s bytes */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_precompute_batch(goldilocks_448_precomputed_s *tables, const goldilocks_448_point_s *points, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_debugging_torque_batch(goldilocks_448_point_s *out, const goldilocks_448_point_s *a, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_debugging_pscale_batch(goldilocks_448_point_s *out, const goldilocks_448_point_s *a, const uint8_t *factor /*n*56*/, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_mul_by_ratio_and_encode_like_eddsa_batch(uint8_t *enc /*n*57*/, const goldilocks_448_point_s *pts, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_decode_like_eddsa_and_mul_by_ratio_batch(goldilocks_448_point_s *pts, goldilocks_error_t *status, const uint8_t *enc /*n*57*/, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_mul_by_ratio_and_encode_like_x448_batch(uint8_t *out /*n*56*/, const goldilocks_448_point_s *pts, size_t n);

/* Scalars mod q */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_scalar_add_batch(goldilocks_448_scalar_s *out, const goldilocks_448_scalar_s *a, const goldilocks_448_scalar_s *b, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_scalar_sub_batch(goldilocks_448_scalar_s *out, const goldilocks_448_scalar_s *a, const goldilocks_448_scalar_s *b, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_scalar_mul_batch(goldilocks_448_scalar_s *out, const goldilocks_448_scalar_s *a, const goldilocks_448_scalar_s *b, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_scalar_halve_batch(goldilocks_448_scalar_s *out, const goldilocks_448_scalar_s *a, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_scalar_invert_batch(goldilocks_448_scalar_s *out, goldilocks_error_t *status, const goldilocks_448_scalar_s *a, size_t n);
/* every element has the same serialized length ser_len (any length, reduced mod q; scalar.c:257-293) */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_scalar_decode_long_batch(goldilocks_448_scalar_s *out, const uint8_t *ser /*n*ser_len*/, size_t ser_len, size_t n);

/* CFRG cryptosystems */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_x448_batch(uint8_t *out /*n*56*/, goldilocks_error_t *status, const uint8_t *base /*n*56*/, const uint8_t *scalar /*n*56*/, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_x448_derive_public_key_batch(uint8_t *out /*n*56*/, const uint8_t *scalar /*n*56*/, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_ed448_convert_public_key_to_x448_batch(uint8_t *x /*n*56*/, const uint8_t *ed /*n*57*/, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_ed448_convert_private_key_to_x448_batch(uint8_t *x /*n*56*/, const uint8_t *ed /*n*57*/, size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_ed448_derive_public_key_batch(uint8_t *pubkey /*n*57*/, const uint8_t *privkey /*n*57*/, size_t n);
/* message i = msg[msg_off[i] .. msg_off[i+1]); prehashed/context are shared by the whole batch,
 * exactly the per-call arguments of the reference (eddsa.c:146-155,253-261). */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_ed448_sign_batch(uint8_t *signature /*n*114*/, const uint8_t *privkey /*n*57*/, const uint8_t *pubkey /*n*57*/, const uint8_t *msg, const size_t *msg_off /*n+1*/, uint8_t prehashed, const uint8_t *context, uint8_t context_len, size_t n);
/* status[i] is exactly what goldilocks_ed448_verify (eddsa.c:253-306) returns for element i.  Batches of 64 or more are
 * grouped by public key on the device: signatures whose 57 key bytes are identical share one decode of the key and one
 * table of its multiples (SURVEY 8(f)4), which only changes the cost, never the accept bit. */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_ed448_verify_batch(goldilocks_error_t *status, const uint8_t *signature /*n*114*/, const uint8_t *pubkey /*n*57*/, const uint8_t *msg, const size_t *msg_off /*n+1*/, uint8_t prehashed, const uint8_t *context, uint8_t context_len, size_t n);
/* Key sets (our extension; SURVEY 8(f)4, "precomputed per-public-key tables for repeated verification under the same key").
 * goldilocks_ed448_verify_batch already shares one table among the byte-identical keys of ONE batch; a key set keeps the
 * tables of m public keys in HBM (41 KB per key) ACROSS calls, so a verifier that sees the same signers again pays neither
 * the key decode nor the table build again.  status[i] is what goldilocks_ed448_verify(signature i, pubkeys[key_index[i]],
 * message i, ...) returns; an undecodable key is accepted into the set and rejects its signatures, like the reference;
 * key_index[i] >= m yields FAILURE for element i.  The handle belongs to the CUDA device that was current at creation. */
typedef struct goldilocks_b200_keyset_s goldilocks_b200_keyset;
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_b200_keyset_create(goldilocks_b200_keyset **keyset, const uint8_t *pubkeys /*m*57*/, size_t m);
GOLDILOCKS_B200_API void goldilocks_b200_keyset_destroy(goldilocks_b200_keyset *keyset);
GOLDILOCKS_B200_API size_t goldilocks_b200_keyset_size(const goldilocks_b200_keyset *keyset);
/* Table layout of the key sets and point sets created from now on: a set whose FLAT tables -- 369 KB per key or point, one 16-entry
 * table of affine multiples per digit position, so a multiplication by the key costs additions only and no doubling -- fit
 * max_table_bytes gets them (default 32 GB: sets of up to 93 000 keys or points); larger sets keep the 41 KB per key layout (ten
 * columns, forty doublings per call).  0 = never flat. */
GOLDILOCKS_B200_API void goldilocks_b200_keyset_policy(unsigned long long max_table_bytes);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_ed448_verify_keyset_batch(goldilocks_error_t *status, const goldilocks_b200_keyset *keyset, const uint32_t *key_index /*n*/, const uint8_t *signature /*n*114*/, const uint8_t *msg, const size_t *msg_off /*n+1*/, uint8_t prehashed, const uint8_t *context, uint8_t context_len, size_t n);
/* Verification by public-key bytes against a key set (our extension; DESIGN.md decision 23): the arguments of
 * goldilocks_ed448_verify_batch plus a key set, for a verifier that knows most of its signers but gets (signature, key, message)
 * rather than key indices.  status[i] is exactly what goldilocks_ed448_verify(signature i, pubkey i, message i, prehashed,
 * context) returns, for every i.  Signatures whose 57 key bytes equal a key of the set use its tables; the others go through
 * goldilocks_ed448_verify_batch's path (grouped by key within the call when there are 64 or more of them).  key_index (may be
 * NULL) receives, per element, the lowest set index whose 57 bytes equal pubkey i, or m when there is none.  A key of the set
 * that does not decode is still a hit and rejects its signatures, as goldilocks_ed448_verify does; duplicate keys in a set are
 * allowed.  The lookup is a binary search over the set's keys in byte order (kept by goldilocks_b200_keyset_create, 4 bytes per
 * key), so its cost does not depend on which keys the set holds.  Everything is public and the call is variable time.  The
 * handle belongs to the CUDA device that was current at creation (another device gets FAILURE) and is never sharded over
 * goldilocks_b200_set_devices.  An empty set is valid: every element misses and the result is goldilocks_ed448_verify_batch's.
 * n = 0 succeeds, n < 2^31. */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_ed448_verify_keyset_lookup_batch(goldilocks_error_t *status, uint32_t *key_index /*n, or NULL*/, const goldilocks_b200_keyset *keyset, const uint8_t *signature /*n*114*/, const uint8_t *pubkey /*n*57*/, const uint8_t *msg, const size_t *msg_off /*n+1*/, uint8_t prehashed, const uint8_t *context, uint8_t context_len, size_t n);
/* X448 peer sets (our extension; the 2014 API's "ECDH with a precomputed partner key", BASELINE.md section 1).  A caller whose
 * fresh secret scalars keep meeting the same public u-coordinates -- HPKE / ECIES to a known recipient, onion packets to a fixed
 * relay set -- builds a set of m peers once: each peer on the curve gets the reference's (5,5,18) comb table of a point that
 * multiplies like u (15 KB per peer in HBM), and an X448 against it costs a comb instead of a ladder.  Any 56 bytes are accepted as
 * a peer, exactly as goldilocks_x448 accepts them (u >= p is taken mod p; twist points, u = 0 and u = p - 1 keep the ladder).  out[i], status[i] are
 * exactly what goldilocks_x448(out, peers[peer_index[i]], scalar + 56 i) returns; peer_index[i] >= m yields FAILURE and 56 zero
 * bytes.  Constant time in the scalars; the peer indices are public.  The handle belongs to the CUDA device that was current at
 * creation and is never sharded over goldilocks_b200_set_devices.  Order a batch by peer: the lanes of a
 * warp then read one table (with many peers in random order goldilocks_x448_batch's ladder is faster; DESIGN.md decision 20).
 * goldilocks_x448_peerset_lookup_batch below takes the peers' bytes and orders the batch on the device. */
typedef struct goldilocks_b200_x448_peerset_s goldilocks_b200_x448_peerset;
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_b200_x448_peerset_create(goldilocks_b200_x448_peerset **set, const uint8_t *peers /*m*56*/, size_t m);
GOLDILOCKS_B200_API void goldilocks_b200_x448_peerset_destroy(goldilocks_b200_x448_peerset *set);
GOLDILOCKS_B200_API size_t goldilocks_b200_x448_peerset_size(const goldilocks_b200_x448_peerset *set);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_x448_peerset_batch(uint8_t *out /*n*56*/, goldilocks_error_t *status, const goldilocks_b200_x448_peerset *set,
                                                                     const uint32_t *peer_index /*n*/, const uint8_t *scalar /*n*56*/, size_t n);
/* X448 against a peer set by the peer's bytes (our extension; DESIGN.md decision 24): the arguments of goldilocks_x448_batch plus a
 * peer set, for a caller that holds each peer's 56 public bytes rather than its index in the set.
 *   Results: out[i], status[i] are exactly what goldilocks_x448(out, base + 56 i, scalar + 56 i) returns, for every i and any 56 bytes.
 *   Lookup: by raw bytes.  peer_index (may be NULL) receives, per element, the lowest set index whose 56 bytes equal base + 56 i, or m
 *   when there is none.  A u of the set encoded differently (u + p) misses and takes the ladder; its result is still goldilocks_x448's.
 *   Duplicate peers are allowed, an empty set is valid (every element misses), n = 0 succeeds, n < 2^31.  The search runs over the
 *   set's peers in byte order (kept by goldilocks_b200_x448_peerset_create, 4 bytes per peer), so its cost does not depend on which
 *   peers the set holds.
 *   Work: the call orders the batch by looked-up peer on the device (a radix sort of the indices, never of the scalars), so the lanes
 *   of a warp read one table whatever order the caller used; hits on peers with a comb table run the comb, every other element the
 *   ladder, in the same launch.
 *   Timing: constant time in the scalars; the bytes, the indices and the order are public.
 *   Devices: the handle belongs to the CUDA device that was current at creation (another device gets FAILURE) and is never sharded
 *   over goldilocks_b200_set_devices. */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_x448_peerset_lookup_batch(uint8_t *out /*n*56*/, goldilocks_error_t *status, uint32_t *peer_index /*n, or NULL*/,
                                                                            const goldilocks_b200_x448_peerset *set, const uint8_t *base /*n*56*/,
                                                                            const uint8_t *scalar /*n*56*/, size_t n);
/* Decaf peer sets (our extension): the same idea for goldilocks_448_direct_scalarmul, the decaf Diffie-Hellman.  A set of m
 * peer encodings is decoded once under allow_identity, and each peer gets the reference's (5,5,18) comb table (15 KB per peer
 * in HBM), so a multiplication against it costs a comb instead of a decode and a window multiplication.  scaled[i], status[i]
 * are exactly what goldilocks_448_direct_scalarmul(scaled + 56 i, peers + 56 peer_index[i], scalar + i, allow_identity,
 * short_circuit) returns, for scalars below q: a peer that does not decode multiplies the base point and reports FAILURE, and
 * with short_circuit that element keeps the caller's bytes.  peer_index[i] >= m behaves like 56 bytes that do not decode.
 * Constant time in the scalars; the peer indices are public.  The call orders the batch by peer on the device (a radix sort of
 * the indices, never of the scalars), so the lanes of a warp read one table whatever order the caller used.  The handle
 * belongs to the CUDA device that was current at creation and is never sharded over goldilocks_b200_set_devices; an empty set
 * is valid.  n < 2^31.  Measured on a B200, 2^20 scalars in any order against 1 to 2^16 peers: 3.5x goldilocks_448_direct_scalarmul_batch
 * (DESIGN.md decision 21). */
typedef struct goldilocks_b200_decaf_peerset_s goldilocks_b200_decaf_peerset;
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_b200_decaf_peerset_create(goldilocks_b200_decaf_peerset **set, const uint8_t *peers /*m*56*/,
                                                                            goldilocks_bool_t allow_identity, size_t m);
GOLDILOCKS_B200_API void goldilocks_b200_decaf_peerset_destroy(goldilocks_b200_decaf_peerset *set);
GOLDILOCKS_B200_API size_t goldilocks_b200_decaf_peerset_size(const goldilocks_b200_decaf_peerset *set);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_direct_scalarmul_peerset_batch(uint8_t *scaled /*n*56*/, goldilocks_error_t *status,
                                                                                     const goldilocks_b200_decaf_peerset *set, const uint32_t *peer_index /*n*/,
                                                                                     const goldilocks_448_scalar_s *scalar, goldilocks_bool_t short_circuit, size_t n);
/* Point sets (our extension): goldilocks_448_base_double_scalarmul_non_secret, s1 B + s2 P on public inputs, against recurring
 * points P -- the participant keys a FROST coordinator checks signature shares against, an OPRF server's public key, the long-term
 * keys of ring and SMP proofs.  A set of m points gets the tables a key set keeps for its keys (goldilocks_b200_keyset_policy
 * picks the layout: flat, 369 KB per point and no doubling per call, or 41 KB per point and forty doublings), so a call costs
 * additions against them instead of a window table and 445 doublings.
 *   Result: out[i] is the group element goldilocks_448_base_double_scalarmul_non_secret(scalar1 + i, points[point_index[i]],
 *   scalar2 + i) returns: goldilocks_448_point_eq holds and goldilocks_448_point_encode gives the same bytes.  out[i] has canonical
 *   limbs and all four coordinates valid.  Scalars are below q, as goldilocks_448_scalar_s requires.  The reference's scalar2 = 0
 *   case is kept: the result is the identity, without scalar1 B.
 *   Indices: point_index[i] >= m behaves as if the point were the identity (scalar1 B, or the identity when scalar2 = 0).
 *   Variable time in all of its inputs, like the reference's _non_secret; never pass secrets.
 *   Points passed to create must satisfy goldilocks_448_point_valid; weakly reduced limbs below 2^60 are accepted.
 * The call orders the batch by point on the device (a radix sort of the indices), so the lanes of a warp read one table whatever
 * order the caller used.  The handle belongs to the CUDA device that was current at creation and is never sharded over
 * goldilocks_b200_set_devices; another device gets FAILURE.  An empty set is valid, n = 0 succeeds, m < 2^32 - 1, n < 2^31
 * (DESIGN.md decision 22). */
typedef struct goldilocks_b200_pointset_s goldilocks_b200_pointset;
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_b200_pointset_create(goldilocks_b200_pointset **set, const goldilocks_448_point_s *points /*m*/, size_t m);
GOLDILOCKS_B200_API void goldilocks_b200_pointset_destroy(goldilocks_b200_pointset *set);
GOLDILOCKS_B200_API size_t goldilocks_b200_pointset_size(const goldilocks_b200_pointset *set);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_base_double_scalarmul_non_secret_pointset_batch(goldilocks_448_point_s *out, const goldilocks_b200_pointset *set,
                                                                                                      const uint32_t *point_index /*n*/, const goldilocks_448_scalar_s *scalar1,
                                                                                                      const goldilocks_448_scalar_s *scalar2, size_t n);
/* Random-linear-combination batch verification (SURVEY 8(f)3; csrc/rlc.cuh): an OPTIONAL fast path for batches in which
 * (nearly) every signature is expected to be valid.  Same arguments and per-element statuses as
 * goldilocks_ed448_verify_batch (eddsa.c:253-306).  Signatures whose R or public key does not decode are rejected up
 * front like the reference does; the rest are checked by ONE multi-scalar multiplication with fresh secret 128-bit
 * weights.  If that equation holds every remaining signature is reported valid (wrong with probability < 2^-127 per
 * call); if it does not, the ordinary per-signature path runs over the batch, so the statuses are the reference's
 * either way.  When the whole-batch equation fails the call localises the damage: the equations are evaluated again per
 * chunk of ~4096 consecutive signatures (same R decodes, challenges and weights), chunks whose equation holds are decided,
 * and only the signatures of the failing chunks go through the per-signature path (packed into one batch).  If more than
 * half of the chunks fail, the per-signature path runs over everything and the next calls on this device skip the equation
 * (see goldilocks_b200_rlc_policy).  *fast_path (may be NULL) receives 1 when the whole-batch equation decided the call,
 * 2 when the per-chunk equations did (failing chunks re-verified one signature at a time), 0 when the per-signature path ran
 * over everything. */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_ed448_verify_rlc_batch(goldilocks_error_t *status, const uint8_t *signature /*n*114*/, const uint8_t *pubkey /*n*57*/, const uint8_t *msg, const size_t *msg_off /*n+1*/, uint8_t prehashed, const uint8_t *context, uint8_t context_len, size_t n, int *fast_path);
/* After a call in which most chunks failed, the next `reprobe` - 1 calls of goldilocks_ed448_verify_rlc_batch on that device go
 * straight to the per-signature path and the one after tries the equation again (default 16; 0 = always try).  Setting the
 * policy also clears the remembered outcomes. */
GOLDILOCKS_B200_API void goldilocks_b200_rlc_policy(unsigned reprobe);
/* Concurrent single-element calls gathered into one batch (csrc/coalesce.h).  The reference's own entry points
 * goldilocks_ed448_verify (ed448.h:157-165; also reached through goldilocks_ed448_verify_prehash), goldilocks_ed448_sign
 * (ed448.h:108-118) and goldilocks_x448 (point_448.h) take one element; called from many host threads at once they are
 * independent, so with window_us > 0 the first caller of a kind waits up to window_us microseconds (or until max_batch calls
 * are in; 0 = 4096) for others, runs ONE batch launch for all of them on its own thread and current device, and every caller
 * gets exactly the result its own call would have produced.  Calls that differ in (prehashed, context) are batched separately.
 * At most three gathered batches run at a time; while the device is that busy a gathering keeps collecting, so batches grow with the load.
 * window_us = 0 (the default) turns it off: a lone caller would only pay the window as latency.  The environment variables
 * GOLDILOCKS_B200_COALESCE_US / GOLDILOCKS_B200_COALESCE_MAX set the same thing for unmodified programs.
 * goldilocks_b200_coalesce_stats: calls that went through a gathering, batches launched for them, largest batch (any may be NULL). */
GOLDILOCKS_B200_API void goldilocks_b200_coalesce(unsigned window_us, unsigned max_batch);
GOLDILOCKS_B200_API void goldilocks_b200_coalesce_stats(unsigned long long *calls, unsigned long long *batches, unsigned long long *largest);
/* SHAKE256 one-shot over n inputs, each squeezed to outlen bytes (shake.c:177-190, SHAKE256 params 211-213) */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_shake256_hash_batch(uint8_t *out /*n*outlen*/, size_t outlen, const uint8_t *in, const size_t *in_off /*n+1*/, size_t n);

/* ======================================================================================
 * 3. Device-resident variants of the headline paths: every pointer is a DEVICE pointer on the
 *    current CUDA device, `stream` is a cudaStream_t passed as void* (NULL = default stream).
 *    Calls are asynchronous on that stream; `scratch` must hold goldilocks_b200_*_scratch_bytes(n).
 * ====================================================================================== */
/* scratch of a device-resident verification on the CURRENT device: decoded points and scalars, the key-grouping work
 * lists, room for n/4 + 1 per-key tables (41 KB each) and the per-lane window tables of the finish kernel; about 11 KB
 * per signature.  Everything the call writes lives in this scratch, so calls in flight on different streams with
 * different scratch buffers are independent.  Returns 0 without a usable GPU. */
GOLDILOCKS_B200_API size_t goldilocks_b200_verify_scratch_bytes(size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_ed448_verify_batch_dev(goldilocks_error_t *status, const uint8_t *signature, const uint8_t *pubkey, const uint8_t *msg, const size_t *msg_off, uint8_t prehashed, const uint8_t *context /*device or NULL*/, uint8_t context_len, size_t n, void *scratch, void *stream);
/* device-pointer form of goldilocks_ed448_verify_rlc_batch: scratch comes from the library's own arena and the call
 * synchronises `stream` (it needs the number of distinct keys and the verdict on the host) */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_ed448_verify_rlc_batch_dev(goldilocks_error_t *status, const uint8_t *signature, const uint8_t *pubkey, const uint8_t *msg, const size_t *msg_off, uint8_t prehashed, const uint8_t *context /*device or NULL*/, uint8_t context_len, size_t n, void *stream, int *fast_path);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_x448_batch_dev(uint8_t *out, goldilocks_error_t *status, const uint8_t *base, const uint8_t *scalar, size_t n, void *stream);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_x448_peerset_batch_dev(uint8_t *out, goldilocks_error_t *status, const goldilocks_b200_x448_peerset *set,
                                                                         const uint32_t *peer_index, const uint8_t *scalar, size_t n, void *stream);
/* scratch of a device-resident X448 peer-set lookup call: the looked-up indices, the sort keys, the order and the sort's temporary
 * storage, about 20 bytes per element.  It holds public data only (indices and order), so it needs no wipe; the secrets stay in
 * out and scalar.  Returns 0 without a usable GPU. */
GOLDILOCKS_B200_API size_t goldilocks_b200_x448_peerset_scratch_bytes(size_t n);
/* device-pointer form of goldilocks_x448_peerset_lookup_batch; scratch >= goldilocks_b200_x448_peerset_scratch_bytes(n).  Fully
 * asynchronous on `stream`: unlike goldilocks_ed448_verify_keyset_lookup_batch_dev it never synchronises it.  It writes only into
 * scratch, out, status and peer_index, so calls in flight on different streams with different scratch buffers are independent. */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_x448_peerset_lookup_batch_dev(uint8_t *out, goldilocks_error_t *status, uint32_t *peer_index /*or NULL*/,
                                                                                const goldilocks_b200_x448_peerset *set, const uint8_t *base, const uint8_t *scalar,
                                                                                size_t n, void *scratch, void *stream);
/* scratch of a device-resident decaf peer-set call: the sort keys, the order and the sort's temporary storage, about 16 bytes
 * per element.  The call writes only there and into scaled / status, so calls in flight on different streams with different
 * scratch buffers are independent.  Returns 0 without a usable GPU. */
GOLDILOCKS_B200_API size_t goldilocks_b200_decaf_peerset_scratch_bytes(size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_direct_scalarmul_peerset_batch_dev(uint8_t *scaled, goldilocks_error_t *status, const goldilocks_b200_decaf_peerset *set,
                                                                                         const uint32_t *peer_index, const goldilocks_448_scalar_s *scalar,
                                                                                         goldilocks_bool_t short_circuit, size_t n, void *scratch, void *stream);
/* scratch of a device-resident point-set call: the sort keys, the order and the sort's temporary storage, about 16 bytes per
 * element.  The call writes only there and into out, so calls in flight on different streams with different scratch buffers are
 * independent.  Returns 0 without a usable GPU. */
GOLDILOCKS_B200_API size_t goldilocks_b200_pointset_scratch_bytes(size_t n);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_base_double_scalarmul_non_secret_pointset_batch_dev(goldilocks_448_point_s *out, const goldilocks_b200_pointset *set,
                                                                                                          const uint32_t *point_index, const goldilocks_448_scalar_s *scalar1,
                                                                                                          const goldilocks_448_scalar_s *scalar2, size_t n, void *scratch, void *stream);
/* scratch of the device-resident key-set calls below, for n signatures and msg_bytes (= msg_off[n]) bytes of messages: the
 * looked-up indices and their order, scalars, the sign-check records, the misses packed, and goldilocks_b200_verify_scratch_bytes(n)
 * for them.  Returns 0 without a usable GPU. */
GOLDILOCKS_B200_API size_t goldilocks_b200_keyset_scratch_bytes(size_t n, size_t msg_bytes);
/* device-pointer form of goldilocks_ed448_verify_keyset_lookup_batch; scratch >= goldilocks_b200_keyset_scratch_bytes(n, msg_off[n]).
 * The call synchronises `stream` ONCE, after the lookup (it needs the number of misses on the host), then queues the rest and
 * returns: the statuses are written when `stream` reaches that point.  It writes only into scratch, status and key_index. */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_ed448_verify_keyset_lookup_batch_dev(goldilocks_error_t *status, uint32_t *key_index /*or NULL*/, const goldilocks_b200_keyset *keyset,
                                                                                       const uint8_t *signature, const uint8_t *pubkey, const uint8_t *msg, const size_t *msg_off,
                                                                                       uint8_t prehashed, const uint8_t *context /*device or NULL*/, uint8_t context_len, size_t n,
                                                                                       void *scratch, void *stream);
/* device-pointer form of goldilocks_ed448_verify_keyset_batch (indices already known); asynchronous on `stream`, scratch as above */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_ed448_verify_keyset_batch_dev(goldilocks_error_t *status, const goldilocks_b200_keyset *keyset, const uint32_t *key_index,
                                                                                const uint8_t *signature, const uint8_t *msg, const size_t *msg_off, uint8_t prehashed,
                                                                                const uint8_t *context /*device or NULL*/, uint8_t context_len, size_t n, void *scratch, void *stream);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_precomputed_scalarmul_batch_dev(goldilocks_448_point_s *out, const goldilocks_448_scalar_s *scalar, size_t n, void *stream);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_gf_mul_batch_dev(uint8_t *out, const uint8_t *a, const uint8_t *b, size_t n, void *stream);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_add_batch_dev(goldilocks_448_point_s *out, const goldilocks_448_point_s *a, const goldilocks_448_point_s *b, size_t n, void *stream);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_double_batch_dev(goldilocks_448_point_s *out, const goldilocks_448_point_s *a, size_t n, void *stream);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_decode_batch_dev(goldilocks_448_point_s *pts, goldilocks_error_t *status, const uint8_t *ser, goldilocks_bool_t allow_identity, size_t n, void *stream);
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_448_point_encode_batch_dev(uint8_t *ser, const goldilocks_448_point_s *pts, size_t n, void *stream);

/* ======================================================================================
 * 4. Library control / introspection
 * ====================================================================================== */
/* Initialise the library on the current CUDA device (builds the fixed-base tables on the device).
 * Called lazily by every entry point; thread-safe.  Returns FAILURE when no usable GPU exists. */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_b200_init(void);
GOLDILOCKS_B200_API const char *goldilocks_b200_last_error(void);
/* Device sets: ONE host-pointer batch spread over several GPUs (SURVEY 8(e); the reference has no counterpart -- its
 * per-element functions eddsa.c:253-306, goldilocks.c:1006-1076, 98-176 are what each range runs).  After
 * goldilocks_b200_set_devices(devs, count) every `*_batch` entry point with HOST pointers cuts [0, n) into contiguous
 * ranges, one run of ranges per listed device, each executed on a worker thread bound to that device with its own
 * stream and arena; the calling thread blocks until all ranges are back.  No collective and no peer traffic.  Heavy
 * operations (verify, sign, X448, scalar multiplications) get one range per device; the light, PCIe-bound field / point /
 * codec operations are pipelined in ~24 MB chunks over three contexts per device so copy-in, kernel and copy-out overlap
 * (a set of ONE device therefore still pipelines them).  Results are identical to the unsharded call (elements are
 * independent); verification groups keys per range.  count = 0 restores the default: the caller's current device only.
 * The environment variable GOLDILOCKS_B200_DEVICES ("all" or "0,1,2,3") sets the same thing at first use.  `_dev` entry
 * points and key sets always run on the current device.  A device may be listed more than once (its ranges then queue
 * on the same contexts: useful to exercise the partition on a single GPU).  Host buffers should be pinned (cudaHostAlloc/cudaHostRegister)
 * for full PCIe speed; pageable buffers work. */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_b200_set_devices(const int *devices, int count);
GOLDILOCKS_B200_API int goldilocks_b200_get_devices(int *devices, int max); /* returns the size of the set (0 = default) */
/* The partition such a call would use over `ndev` devices (pure arithmetic, needs no GPU): piece k covers [lo[k], hi[k]) on
 * device_slot[k] (index into the set) and context lane[k]; returns the number of pieces (writes at most `max`). */
GOLDILOCKS_B200_API size_t goldilocks_b200_shard_plan(size_t *lo, size_t *hi, int *device_slot, int *lane, size_t max, size_t n, int ndev, size_t bytes_per_elem, int pipelined);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
GOLDILOCKS_B200_API uint64_t goldilocks_b200_launch_count(void);
/* Per-launch CUDA-event timing for bench.py's roofline leg.  profile(1) clears the log and starts
 * bracketing every kernel launch with two events on its stream; profile(0) stops.  profile_read()
 * waits for the recorded events and writes up to `max` entries: names[64*k..] = lane functor name of
 * launch k (e.g. "LaneEdVerifyFinish"), ms[k] = its device time.  Returns the number written. */
GOLDILOCKS_B200_API void goldilocks_b200_profile(int enable);
GOLDILOCKS_B200_API size_t goldilocks_b200_profile_read(char *names, float *ms, size_t max);
/* the same log as a timeline: begin and end of launch k in ms after the begin of the first logged launch (kernels of one
 * call may run on two streams: goldilocks_ed448_verify_rlc_batch) */
GOLDILOCKS_B200_API size_t goldilocks_b200_profile_timeline(char *names, float *start_ms, float *end_ms, size_t max);
/* Test entry point (no counterpart in the reference's API: goldilocks.c:271-380 keeps these static).  One mixed addition or conversion
 * per element, all four coordinates returned: op 0 pniels_to_pt(pt_to_pniels(q)); 1 / 2 p +/- pniels(q) and 3 / 4 p +/- comb[which % 80]
 * through the by-value code of the lane kernels; 5 niels_to_pt(comb[which % 80]); 6 / 7 and 8 / 9 the same additions through the
 * slot-machine code of the scalar-multiplication kernels.  comb = the base-point comb table (goldilocks_b200_export_comb_table). */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_b200_debug_niels_batch(goldilocks_448_point_s *out, const goldilocks_448_point_s *p, const goldilocks_448_point_s *q, const uint32_t *which, uint32_t op, size_t n);
/* Copies the device-built fixed-base comb table (80 niels x 3 gf, canonical radix-2^56 limbs =
 * 15360 bytes, the layout of the reference's goldilocks_448_precomputed_base) to `out`. */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_b200_export_comb_table(uint8_t out[15360]);
/* Same for the 32-entry wNAF base table (reference goldilocks_448_precomputed_wnaf_as_fe, 6144 bytes). */
GOLDILOCKS_B200_API goldilocks_error_t goldilocks_b200_export_wnaf_table(uint8_t out[6144]);

#ifdef __cplusplus
}
#endif
#endif /* GOLDILOCKS_B200_H */
