"""Generates the committed fixtures under tests/golden/ (run in the build container, where /root/reference exists):

    python scripts/make_golden.py

cpq_encode_reference.npz   outputs of the REFERENCE's own C encoder (Sources/CPQEncode/pq_encode.c, compiled unmodified
                           into oracle/_ref/libcpq_ref.so by `make -C oracle ref`) on the sin/cos fixture of
                           Tests/VectorIndexTests/PQEncodeParity_AoS_C_vs_Swift_Tests.swift:5-31 and on a seeded random
                           problem, every entry point.  Real reference outputs: the oracle and the CUDA library must
                           reproduce them bit for bit.
cpq_encode_reference_fixtures.npz
                           outputs of the same compiled reference encoder on the inputs of the oracle pins and the GPU layout
                           test (tests/golden_inputs.py): every entry point on a seeded random problem, plain and fused
                           residual codes at d / m = 128, and the with-CSQ codes and the SoA-blocked and interleaved layouts
                           of the n = 70 parity fixture.  The committed file was written where the reference source was not
                           at hand, from the oracle's codes (the layouts: pq_encode.c's index formulas applied to them).
                           The same oracle and CUDA code had passed the tests that now read these arrays while those tests
                           still called the compiled reference: they asserted these codes and buffers bit-equal to its
                           outputs.  Run where oracle/_ref is built, this script rewrites them from the reference itself.
oracle_search_small.npz    a small IVF-PQ problem (SIFT-shaped values with many ties) with the ORACLE's outputs of every
                           stage of the search path: list assignment, residual PQ codes, probe lists, residual LUTs, ADC
                           distances, flat top-k and the IVF-PQ top-k.  No reference test pins LUT / ADC arithmetic (SURVEY.md
                           8c), so these vectors only freeze the restatement; the GPU tests compare against them so that a
                           parity claim does not depend on rebuilding the oracle.
Inputs are regenerated from seeds by the tests (tests/golden_inputs.py); only outputs are stored."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import oracle  # noqa: E402
import golden_inputs as gi  # noqa: E402
from conftest import parity_fixture  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
os.makedirs(OUT, exist_ok=True)


def encoder_golden():
    if oracle.ref_lib() is None:
        oracle.build(ref=True)
    assert oracle.ref_lib() is not None, "oracle/_ref/libcpq_ref.so is needed (make -C oracle ref)"
    out = {}
    for name, (x, cb8, cb4, coarse, assign, m) in gi.encoder_problems().items():
        d = x.shape[1]
        csq = oracle.pq_centroid_sq(cb8, m, 256, d // m, swift=True)
        nodot = oracle.PQEncodeOpts(0, False, False, 8, 0, 0, 0)
        out[f"{name}.u8"] = oracle.ref_encode("cpq_encode_u8_f32", x, cb8, m, 256)
        out[f"{name}.u8_nodot"] = oracle.ref_encode("cpq_encode_u8_f32", x, cb8, m, 256, opts=nodot)
        out[f"{name}.u8_csq"] = oracle.ref_encode("cpq_encode_u8_f32_with_csq", x, cb8, m, 256, centroid_sq=csq)
        out[f"{name}.res"] = oracle.ref_encode("cpq_encode_residual_u8_f32", x, cb8, m, 256, coarse=coarse, assign_=assign)
        out[f"{name}.res_nodot"] = oracle.ref_encode("cpq_encode_residual_u8_f32", x, cb8, m, 256, coarse=coarse,
                                                     assign_=assign, opts=nodot)
        out[f"{name}.res_csq"] = oracle.ref_encode("cpq_encode_residual_u8_f32_with_csq", x, cb8, m, 256, centroid_sq=csq,
                                                   coarse=coarse, assign_=assign)
        out[f"{name}.u4"] = oracle.ref_encode("cpq_encode_u4_f32", x, cb4, m, 16, packed_u4=True)
        out[f"{name}.res_u4"] = oracle.ref_encode("cpq_encode_residual_u4_f32", x, cb4, m, 16, coarse=coarse, assign_=assign,
                                                  packed_u4=True)
        out[f"{name}.csq"] = csq
    np.savez_compressed(os.path.join(OUT, "cpq_encode_reference.npz"), **out)
    print("cpq_encode_reference.npz:", {k: v.shape for k, v in out.items()})


def reference_fixtures_golden():
    assert oracle.ref_lib() is not None, "oracle/_ref/libcpq_ref.so is needed (make -C oracle ref)"
    out = {}
    nodot = oracle.PQEncodeOpts(0, False, False, 8, 0, 0, 0)
    for v in gi.ENCODER_VARIANTS:
        x, cb, coarse, assign, m, ks = gi.encoder_variant_problem(v)
        res = dict(coarse=coarse, assign_=assign)
        csq = oracle.pq_centroid_sq(cb, m, ks, x.shape[1] // m, swift=True)
        out[f"variant.{v}"] = {
            "u8": lambda: oracle.ref_encode("cpq_encode_u8_f32", x, cb, m, ks),
            "u8_nodot": lambda: oracle.ref_encode("cpq_encode_u8_f32", x, cb, m, ks, opts=nodot),
            "u8_csq": lambda: oracle.ref_encode("cpq_encode_u8_f32_with_csq", x, cb, m, ks, centroid_sq=csq),
            "res": lambda: oracle.ref_encode("cpq_encode_residual_u8_f32", x, cb, m, ks, **res),
            "res_nodot": lambda: oracle.ref_encode("cpq_encode_residual_u8_f32", x, cb, m, ks, opts=nodot, **res),
            "res_csq": lambda: oracle.ref_encode("cpq_encode_residual_u8_f32_with_csq", x, cb, m, ks, centroid_sq=csq, **res),
            "u4": lambda: oracle.ref_encode("cpq_encode_u4_f32", x, cb, m, ks, packed_u4=True),
            "res_u4": lambda: oracle.ref_encode("cpq_encode_residual_u4_f32", x, cb, m, ks, packed_u4=True, **res),
        }[v]()
    x, cent, asg, cb, m, ks = gi.long_subvector_residual_problem()
    out["long_residual.plain"] = oracle.ref_encode("cpq_encode_u8_f32", (x - cent[asg]).astype(np.float32), cb, m, ks)
    out["long_residual.fused"] = oracle.ref_encode("cpq_encode_residual_u8_f32", x, cb, m, ks, coarse=cent, assign_=asg)
    x, cb, _, _ = parity_fixture(n=70)
    n, d, m = x.shape[0], x.shape[1], 8
    out["parity70.u8_csq"] = oracle.ref_encode("cpq_encode_u8_f32_with_csq", x, cb, m, 256,
                                               centroid_sq=oracle.pq_centroid_sq(cb, m, 256, d // m, swift=False))
    L = oracle.ref_lib()
    L.cpq_encode_u8_f32.restype = None
    for name, layout, B, g in gi.LAYOUTS:
        Bq, gq = (B or 64), (g or 8)
        buf = np.zeros(m * ((n + Bq - 1) // Bq) * Bq if layout == 1 else ((n + gq - 1) // gq) * m * gq, dtype=np.uint8)
        L.cpq_encode_u8_f32(x.ctypes.data_as(oracle.f32p), C.c_int64(n), C.c_int(d), C.c_int(m), C.c_int(256),
                            cb.ctypes.data_as(oracle.f32p), buf.ctypes.data_as(oracle.u8p),
                            C.byref(oracle.PQEncodeOpts(layout, True, False, 8, 0, B, g)))
        out[f"layout.{name}"] = buf
    np.savez_compressed(os.path.join(OUT, "cpq_encode_reference_fixtures.npz"), **out)
    print("cpq_encode_reference_fixtures.npz:", {k: v.shape for k, v in out.items()})


def search_golden():
    P = gi.search_problem()
    xb, q, coarse, cb, m, kc, nprobe, k = P["xb"], P["q"], P["coarse"], P["cb"], P["m"], P["kc"], P["nprobe"], P["k"]
    d = xb.shape[1]
    out = {}
    norms = oracle.pq_centroid_sq(cb.reshape(-1), m, 256, d // m, swift=True).reshape(m, 256)
    out["cb_norms"] = norms
    asg, adist = oracle.assign(xb, coarse)
    out["assign"], out["assign_dist"] = asg, adist
    codes = oracle.pq_encode_u8(xb, cb, m, 256, centroid_sq=norms.reshape(-1), coarse=coarse, assign_=asg)
    out["codes"] = codes
    cn = oracle.centroid_norms(coarse)
    pid, psc = oracle.probe_select_batch(q, coarse, nprobe, 0, cn)
    out["probe_ids"], out["probe_scores"] = pid, psc
    # per (query, first probe) residual LUT and the ADC distances of that list (reference defaults)
    off, order = oracle.build_lists(asg, kc)
    luts, adcs = [], []
    for r in range(8):
        l = int(pid[r, 0])
        lut = oracle.pq_lut_residual_l2(q[r], coarse[l], cb, m, 256, cnorms=norms)
        rows = order[off[l]:off[l + 1]]
        luts.append(lut)
        adcs.append(oracle.adc_scan_u8(codes[rows], lut, m, 256) if rows.size else np.zeros(0, np.float32))
    out["lut_first_probe"] = np.stack(luts)
    out["adc_first_probe"] = np.concatenate(adcs)
    out["adc_first_probe_len"] = np.array([a.size for a in adcs], dtype=np.int64)
    fd, fi, _ = oracle.flat_search(q, xb, k, 0)
    out["flat_dist"], out["flat_ids"] = fd, fi
    cd, ci, _ = oracle.flat_search(q, xb, k, 2)                        # cosine (Cosine.run two-pass), distance 1 - sim
    out["cosine_dist"], out["cosine_ids"] = cd, ci
    ids = np.arange(xb.shape[0], dtype=np.int64)
    od, oi, op = oracle.ivfpq_search(q, coarse, cb, norms, off, codes[order], ids[order], m, 256, nprobe, k, 0)
    out["ivfpq_dist"], out["ivfpq_ids"] = od, oi
    assert np.array_equal(op, pid)
    # cosine rows of the coarse quantiser and the IVF-Flat index (CentroidBatchScore.swift:70-84; IVFIndex.swift:376-435,
    # 905-927; DistanceUtils.swift:22-38), one centroid degenerate
    cz = coarse.copy()
    cz[5] = 0.0
    out["cbs_cosine"] = oracle.centroid_batch_score(q, cz, 2)
    out["probe_ids_cosine"] = oracle.probe_select_batch(q, cz, nprobe, 2)[0]
    casg = oracle.assign_metric(xb, cz, 2)
    out["assign_cosine"] = casg
    coff, corder = oracle.build_lists(casg, kc)
    out["ivfflat_cosine_dist"], out["ivfflat_cosine_ids"] = oracle.ivfflat_search(q, cz, coff, xb[corder], ids[corder], nprobe, k, 2)
    np.savez_compressed(os.path.join(OUT, "oracle_search_small.npz"), **out)
    print("oracle_search_small.npz:", {k_: v.shape for k_, v in out.items()})


if __name__ == "__main__":
    encoder_golden()
    reference_fixtures_golden()
    search_golden()
