"""Seeded INPUTS of the committed golden fixtures (tests/golden/*.npz hold only the outputs; scripts/make_golden.py
wrote them).  Everything here is plain numpy with fixed seeds, so the inputs are identical wherever the tests run."""
import numpy as np

from conftest import parity_fixture


def encoder_problems():
    """name -> (x [n x d], codebooks ks=256, codebooks ks=16, coarse [kc x d], assign [n], m)"""
    out = {}
    # the reference's own fixture (PQEncodeParity_AoS_C_vs_Swift_Tests.swift:5-31), u8 and u4 codebooks by the same formula
    x, cb8, coarse, assign = parity_fixture(16, 32, 8, 256, 4)
    _, cb4, _, _ = parity_fixture(16, 32, 8, 16, 4)
    out["parity"] = (x, cb8, cb4, coarse, assign, 8)
    rng = np.random.default_rng(20261018)
    n, d, m, kc = 257, 48, 6, 5
    x = rng.standard_normal((n, d)).astype(np.float32)
    cb8 = rng.standard_normal(m * 256 * (d // m)).astype(np.float32)
    cb4 = rng.standard_normal(m * 16 * (d // m)).astype(np.float32)
    coarse = (rng.standard_normal((kc, d)) * 0.5).astype(np.float32)
    assign = rng.integers(0, kc, n).astype(np.int32)
    out["random"] = (x, cb8, cb4, coarse, assign, m)
    return out


ENCODER_VARIANTS = ["u8", "u8_nodot", "u8_csq", "res", "res_csq", "res_nodot", "u4", "res_u4"]


def encoder_variant_problem(variant):
    """seeded random problem of tests/test_oracle_pins.py::test_oracle_encoder_equals_reference_encoder:
    (x, codebooks, coarse, assign, m, ks); the codebooks have ks = 16 for the u4 variants"""
    rng = np.random.default_rng(7)
    n, d, m, kc = 300, 48, 6, 5
    ks = 16 if variant.endswith("u4") else 256
    x = rng.standard_normal((n, d)).astype(np.float32)
    cb = rng.standard_normal((m * ks * (d // m))).astype(np.float32)
    coarse = rng.standard_normal((kc, d)).astype(np.float32) * np.float32(0.5)
    assign = rng.integers(0, kc, n).astype(np.int32)
    return x, cb, coarse, assign, m, ks


def long_subvector_residual_problem():
    """ResidualKernelTests.swift:126-200 (n = 2000, d = 1024, m = 8, ks = 256, kc = 100, uniform [-1, 1)):
    (x, coarse, assign, codebooks, m, ks)"""
    rng = np.random.default_rng(1)
    n, d, m, ks, kc = 2000, 1024, 8, 256, 100
    x = rng.uniform(-1, 1, (n, d)).astype(np.float32)
    cent = rng.uniform(-1, 1, (kc, d)).astype(np.float32)
    asg = rng.integers(0, kc, n).astype(np.int32)
    cb = rng.uniform(-1, 1, (m * ks, d // m)).astype(np.float32)
    return x, cent, asg, cb, m, ks


# output layouts of pq_encode.c:260-276 on parity_fixture(n=70): (name, layout, soa_block_B, interleave_g)
LAYOUTS = [("soa_b64", 1, 64, 0), ("soa_b16", 1, 16, 0), ("interleaved_g8", 2, 0, 8), ("interleaved_g4", 2, 0, 4)]


def search_problem():
    """small SIFT-shaped IVF-PQ problem: non-negative integer-valued components (many exact ties)"""
    rng = np.random.default_rng(96)
    n, nq, d, m, kc = 3000, 24, 32, 8, 24
    centres = np.floor(np.abs(rng.standard_normal((40, d))) * 40).clip(0, 218)
    which = rng.integers(0, 40, n + nq)
    x = np.floor(np.abs(centres[which] + 12.0 * rng.standard_normal((n + nq, d)))).clip(0, 218).astype(np.float32)
    coarse = x[rng.choice(n, kc, replace=False)].copy()
    cb = (rng.standard_normal((m, 256, d // m)) * 14.0).astype(np.float32)
    return dict(xb=np.ascontiguousarray(x[:n]), q=np.ascontiguousarray(x[n:]), coarse=coarse, cb=cb, m=m, kc=kc, nprobe=5, k=10)
