"""Probability-domain (MMI) table generation (SURVEY 8f row f3, BASELINE config 4's tables).  Golden vectors
(tests/golden/mmi_golden.npz) were produced by the REFERENCE's own generator code, QDensityEvolution_MMI.py on top of its
numpy MMI quantizer (make_mmi_golden.py states the two pinned conventions).  CPU: the fixture is well formed and its tables
drive the oracle decoders (layout check: levels = n, Qc x Qc root tables).  GPU: lutgen.mmi_quantize_batch /
MMILUTGenerator vs golden bit for bit, and the CUDA decoders on those tables (float64 symbols, like
mainQuantizedDecoder_ProbabilityDomain.py:174-179) vs the compiled reference."""
import os

import numpy as np
import pytest

from oracle import polar_oracle as po
from quantized_decoder_polar_codes_b200 import simulation as sim
import common

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mmi_golden.npz")
RUNS = [("n16q4", 16, 4, 4), ("n32q8c6", 32, 8, 6), ("n64q16", 64, 16, 16)]


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def tables_of(gold, tag, N):
    f = [gold[tag + "/f_root"][None]] + [t[None] for t in gold[tag + "/lut_f"]]
    g = [gold[tag + "/g_root"][None]] + [t[None] for t in gold[tag + "/lut_g"]]
    assert len(f) == N - 1 and len(g) == N - 1
    return f, g, gold[tag + "/llrs"]


def mmi_case(gold, tag, N, qc, kind, K, L=4, A=None, B=48, seed=3):
    """constructor arguments + channel symbols (float64, as the probability-domain driver passes them)"""
    rng = np.random.default_rng(seed)
    fm, mm = sim.frozen_mask(N, K)
    f, g, llrs = tables_of(gold, tag, N)
    kw = dict(N=N, K=K, frozen_bits=fm, message_bits=mm)
    if kind in common.LIST_KINDS:
        kw["L"] = L
    if kind in common.CA_KINDS:
        kw["A"] = A
    if kind == "CASCLLUTDecoder":
        kw.update(crc_n=24, crc_p=list(sim.CRC24_LOC))
    if "Fast" in kind:
        kw["node_type"] = sim.identify_nodes(N, fm)
    nf, ng = ("LUT_Fs", "LUT_Gs") if kind == "FastSCLUTDecoder" else ("LUT_f", "LUT_g")
    kw[nf], kw[ng], kw["virtual_channel_llr"] = f, g, llrs
    x = rng.integers(0, qc, (B, N)).astype(np.float64)
    return kw, x


def test_fixture_is_well_formed(gold):
    for tag, N, qd, qc in RUNS:
        n = int(np.log2(N))
        assert gold[tag + "/llrs"].shape == (n, N, qd)                    # levels = n (QDensityEvolution_MMI.py:38)
        assert gold[tag + "/f_root"].shape == (qc, qc) and gold[tag + "/g_root"].shape == (2, qc, qc)
        assert gold[tag + "/lut_f"].shape == (N - 2, qd, qd) and gold[tag + "/lut_g"].shape == (N - 2, 2, qd, qd)
        for k in ("/f_root", "/g_root", "/lut_f", "/lut_g"):
            t = gold[tag + k]
            assert t.min() >= 0 and t.max() < qd
    for i in range(int(gold["nq"])):
        Q, Az = gold[f"q{i}/Q"], gold[f"q{i}/Az"]
        assert (Q.sum(axis=0) == 1).all() and (np.diff(Az) >= 1).all()     # every input symbol in exactly one cluster
        assert np.allclose(gold[f"q{i}/pzx"].sum(axis=1), 1.0)


@pytest.mark.parametrize("kind,K", [("SCLUTDecoder", 30), ("SCLLUTDecoder", 32), ("FastSCLUTDecoder", 30), ("CAFastSCLLUTDecoder", 40)])
def test_oracle_decodes_with_mmi_tables(gold, refmod, kind, K):
    """probability-domain layout through the C restatement vs the compiled reference (CPU only)"""
    for tag, N, qd, qc in RUNS[1:]:
        if K >= N:
            continue
        kw, x = mmi_case(gold, tag, N, qc, kind, min(K, N - 4), A=min(K, N - 4) - 8 if kind in common.CA_KINDS else None, B=24)
        want = common.ref_decode(refmod, kind, kw, x)
        got = po.OracleDecoder(kind, **kw).decode(x.astype(np.int32))
        assert (got == want).all(), (kind, tag)


# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_cuda_mmi_quantizer_matches_golden(gold):
    from quantized_decoder_polar_codes_b200.lutgen import mmi_quantize_batch
    for i in range(int(gold["nq"])):
        K = int(gold[f"q{i}/K"])
        Q, pzx, Az, perm = mmi_quantize_batch(gold[f"q{i}/joint"][None], K)
        assert (perm[0] == gold[f"q{i}/perm"]).all(), i
        assert (Az[0] == gold[f"q{i}/Az"]).all(), i
        assert (Q[0] == gold[f"q{i}/Q"]).all(), i
        assert (pzx[0] == gold[f"q{i}/pzx"]).all(), i


@pytest.mark.gpu
@pytest.mark.parametrize("tag,N,qd,qc", RUNS)
def test_cuda_mmi_generator_matches_reference_generator(gold, tag, N, qd, qc):
    from quantized_decoder_polar_codes_b200.lutgen import MMILUTGenerator
    lut_f, lut_g, llrs, probs = MMILUTGenerator(N, qd).run(gold[tag + "/pzx"].copy())
    assert (lut_f[0] == gold[tag + "/f_root"]).all() and (lut_g[0] == gold[tag + "/g_root"]).all()
    assert (np.stack(lut_f[1:]) == gold[tag + "/lut_f"]).all()
    assert (np.stack(lut_g[1:]) == gold[tag + "/lut_g"]).all()
    assert (llrs == gold[tag + "/llrs"]).all()
    assert (probs == gold[tag + "/probs"]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("kind,K,L", [("SCLUTDecoder", 30, 1), ("SCLLUTDecoder", 32, 8), ("FastSCLUTDecoder", 30, 1),
                                      ("FastSCLLUTDecoder", 30, 4), ("CASCLLUTDecoder", 44, 8), ("CAFastSCLLUTDecoder", 40, 8)])
def test_cuda_decoders_on_mmi_tables_vs_reference(gold, kind, K, L):
    """config-4 class and friends on probability-domain tables: levels = n indexing, Qc != Qd root tables, float64 symbols.
    The checker is the compiled reference where it has been built.  Without it the checker is the oracle, and the test then
    shows only that the CUDA decoders and the C restatement read this layout alike: no decoded words of the reference on
    MMI tables are stored, so whether both read it as the reference does rests on test_oracle_decodes_with_mmi_tables,
    which needs the reference."""
    import quantized_decoder_polar_codes_b200 as q
    ref = po.load_reference()
    for tag, N, qd, qc in RUNS[1:]:
        k = min(K, N - 4)
        kw, x = mmi_case(gold, tag, N, qc, kind, k, L=L, A=k - 24 if kind == "CASCLLUTDecoder" else (k - 8 if kind in common.CA_KINDS else None), B=96)
        if kind == "CASCLLUTDecoder" and k - 24 < 1:
            continue
        want = common.ref_decode(ref, kind, kw, x) if ref is not None else po.OracleDecoder(kind, **kw).decode(x)
        dec = getattr(q, kind)(**kw)
        got = dec.decode(x)                      # float64 (B, N), forcecast like the reference's py::array_t<int>
        assert (got == want).all(), (kind, tag, dec.kernel)
