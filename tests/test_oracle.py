"""Pins the oracle (oracle/liboracle.so, our CPU restatement): against every golden vector the
reference's own tests hold for the path, and -- where the unmodified reference was compiled
(oracle/_ref, build container) -- against the reference itself on random and edge inputs."""
import os

import parity
import util


def test_oracle_rfc8032_vectors(oracle, vectors):
    parity.check_eddsa_vectors(oracle, vectors)


def test_oracle_rfc7748_vectors(oracle, vectors):
    parity.check_x448_vectors(oracle, vectors, iters=1000)


def test_oracle_decaf_elligator_vectors(oracle, vectors):
    parity.check_decaf_vectors(oracle, vectors)


def test_oracle_shake_vs_hashlib(oracle):
    parity.check_shake(oracle)


def test_reference_build_reproduces_vectors(ref, vectors):
    """the compiled reference itself (sanity of the oracle/_ref recipe)"""
    parity.check_eddsa_vectors(ref, vectors)
    parity.check_decaf_vectors(ref, vectors)
    parity.check_x448_vectors(ref, vectors, iters=1000)


def test_oracle_vs_reference(oracle):
    """the reference's Ed448 / X448 outputs stored as golden data always; everything else against the reference build
    where it exists"""
    parity.check_openssl_golden(oracle, util.openssl_golden())
    ref = util.ref_lib()
    if ref is None:
        return
    t = os.cpu_count() or 1
    util.set_threads(oracle, t)
    util.set_threads(ref, t)
    parity.check_tables(oracle, ref)
    parity.check_field(oracle, ref, 4096)
    parity.check_field_isr(oracle, ref, 128)
    parity.check_points(oracle, ref, 512)
    parity.check_codec(oracle, ref, 128)
    parity.check_elligator_inverse(oracle, ref, 96)
    parity.check_scalars(oracle, ref, 1024)
    parity.check_comb(oracle, ref, 128)
    parity.check_scalarmul(oracle, ref, 48)
    parity.check_x448(oracle, ref, 96)
    parity.check_eddsa_random(oracle, ref, 128)


def test_reference_arch_backends_agree(ref):
    """arch_x86_64 (the CPU baseline) and arch_ref64 / arch_32 builds of the reference give identical bytes"""
    for arch in ("ref64", "32"):
        other = util.ref_lib(arch)
        if other is None:
            continue
        parity.check_field(other, ref, 1024)
        parity.check_x448(other, ref, 32)
        if arch == "ref64":          # arch_32 has a different in-memory point/table layout (16 x u32 limbs)
            parity.check_points(other, ref, 128)
            parity.check_tables(other, ref)
