"""Plug-in proof (BASELINE north star: "the main*Decoder_*.py simulation drivers and the pickled lookup tables plug in
unchanged"; SURVEY App. C).

CPU, where the reference tree exists: the UNMODIFIED mainQuantizedDecoder_LLRDomain.py runs under
quantized_decoder_polar_codes_b200.run_driver (compat shims: numpy, torchtracer, matplotlib, frame cap) from pickles in the
generator's layout, with the compiled reference's decoders behind the PolarDecoder import path -- and the restated loop of
tests/driver_loop.py, same seed, ends with the same error counters.  That pins the restated loop to the script.
GPU: the restated loop from the same pickles with THIS package behind every import the script makes (PolarDecoder.Decoder.*,
PolarBDEnc.Encoder.*, quantizers.quantizer.LLROptLSQuantizer) against the compiled reference's decoders (the oracle's where
the reference is not built): every decoded word and therefore BER/BLER identical."""
import os
import sys
import types

import numpy as np
import pytest

import driver_loop
import real_lut
from quantized_decoder_polar_codes_b200 import compat, simulation as sim

REF = "/root/reference"
have_ref = os.path.isfile(os.path.join(REF, "mainQuantizedDecoder_LLRDomain.py"))
N, QD, QC, QCU, DESIGN = 128, 16, 16, 128, 3.0


class NumpyPolarEnc:
    """PolarBDEnc.Encoder.PolarEnc on numpy (CPU tests only; the package's own is the GPU encoder)"""
    def __init__(self, N, K, frozenbits, msgbits):
        self.fm = np.ones(N, np.int32)
        self.fm[np.asarray(msgbits)] = 0

    def encode(self, msg):
        return sim.polar_encode(np.asarray(msg, np.uint8), self.fm)[0]


class NumpyCRCEnc:
    def __init__(self, crc_n, crc_p):
        self.n, self.p = crc_n, crc_p

    def encode(self, msg):
        return sim.crc_attach(np.asarray(msg, np.uint8), self.n, tuple(self.p))[0]


def pw_sets(N, K):
    fm, mm = sim.frozen_mask(N, K)
    return np.flatnonzero(fm), np.flatnonzero(mm), fm, mm


def node_types(N, K, frozenbits, msgbits):
    fm = np.zeros(N, np.int32)
    fm[frozenbits] = 1
    return sim.identify_nodes(N, fm)


@pytest.fixture(scope="module")
def workdir(tmp_path_factory):
    z = real_lut.load()
    d = tmp_path_factory.mktemp("driver")
    driver_loop.write_llr_domain_pickles(str(d), N, QC, QD, DESIGN, z["lut_f"], z["lut_g"], z["llr_quanta"])
    return str(d)


def _ref_numpy_quantizer():
    """quantizers.quantizer.LLROptLSQuantizer.LLRQuantizer on the reference's numpy restatement (CPU test only)"""
    sys.path.insert(0, REF)
    from QuantizeDensityEvolution import MinDistortionQuantizer as mdq

    class LLRQuantizer:
        def find_OptLS_quantizer(self, density, quanta, M, K):
            d, q, lut = mdq.find_OptLS_quantizer(np.asarray(density, np.float64).ravel(), np.asarray(quanta, np.float64).ravel(), K)
            return d[None], q[None], lut[None], 0.0
    return LLRQuantizer


@pytest.mark.skipif(not have_ref, reason="reference sources not present")
@pytest.mark.parametrize("decoder_type,is_crc", [("SCL-LUT", "no"), ("FastSC-LUT", "no"), ("CASCL-LUT", "yes")])
def test_unmodified_driver_runs_under_the_compat_layer(workdir, refmod, decoder_type, is_crc, monkeypatch):
    from quantized_decoder_polar_codes_b200 import run_driver
    LLRQuantizer = _ref_numpy_quantizer()
    # the script's imports: decoders = compiled reference, encoder = numpy, quantizer = the reference's numpy DP
    mods = {"PolarDecoder": types.ModuleType("PolarDecoder"), "PolarDecoder.Decoder": types.ModuleType("PolarDecoder.Decoder"),
            "PolarBDEnc": types.ModuleType("PolarBDEnc"), "PolarBDEnc.Encoder": types.ModuleType("PolarBDEnc.Encoder"),
            "quantizers": types.ModuleType("quantizers"), "quantizers.quantizer": types.ModuleType("quantizers.quantizer")}
    for k in ["SCLUTDecoder", "SCLLUTDecoder", "FastSCLUTDecoder", "FastSCLLUTDecoder", "CASCLLUTDecoder"]:
        m = types.ModuleType("PolarDecoder.Decoder." + k)
        setattr(m, k, getattr(refmod, k))
        mods["PolarDecoder.Decoder." + k] = m
    for k, cls in (("PolarEnc", NumpyPolarEnc), ("CRCEnc", NumpyCRCEnc)):
        m = types.ModuleType("PolarBDEnc.Encoder." + k)
        setattr(m, k, cls)
        mods["PolarBDEnc.Encoder." + k] = m
    m = types.ModuleType("quantizers.quantizer.LLROptLSQuantizer")
    m.LLRQuantizer = LLRQuantizer
    mods["quantizers.quantizer.LLROptLSQuantizer"] = m
    for k, v in mods.items():
        monkeypatch.setitem(sys.modules, k, v)
    monkeypatch.chdir(workdir)
    if not os.path.exists("reliable sequence.txt"):
        os.symlink(os.path.join(REF, "reliable sequence.txt"), "reliable sequence.txt")
    frames, seed, A = 25, 7, 32
    argv = ["--N", str(N), "--A", str(A), "--L", "8", "--DecoderType", decoder_type, "--isCRC", is_crc, "--QChannelUniform", str(QCU),
            "--QDecoder", str(QD), "--QChannel", str(QC), "--DesignSNRdB", str(DESIGN)]
    import tqdm
    real_tqdm = tqdm.tqdm
    try:
        g = run_driver.run(os.path.join(REF, "mainQuantizedDecoder_LLRDomain.py"), argv, max_frames=frames, seed=seed,
                           decoders=False, encoder=False, quantizers=False)
    finally:
        tqdm.tqdm = real_tqdm
    assert g["Nblocks"] == frames and g["DecoderType"] == decoder_type
    # the restated loop on the same seed ends the last Eb/N0 point (5 dB) with the same counters
    sys.path.insert(0, REF)
    from utils import channel_llr_density_table
    stats, _ = driver_loop.run(workdir, N, A, 8, decoder_type, is_crc == "yes", QCU, QD, QC, DESIGN, frames, seed, [0, 1, 2, 3, 4, 5],
                               {k: getattr(refmod, k) for k in ["SCLUTDecoder", "SCLLUTDecoder", "FastSCLUTDecoder", "FastSCLLUTDecoder", "CASCLLUTDecoder"]},
                               NumpyPolarEnc, NumpyCRCEnc, LLRQuantizer, pw_sets, node_types, channel_llr_density_table)
    assert stats[-1] == (int(g["Nbiterrs"]), int(g["Nblkerrs"]), int(g["Nblocks"]))
    assert sum(s[2] for s in stats) == int(g["total_blocks"])


def test_compat_numpy_shims():
    compat.install(decoders=False, encoder=False, quantizers=False)
    assert np.int is int
    ragged = np.array([np.zeros((2, 3)), np.zeros((1, 3))])
    assert ragged.dtype == object and ragged[1].shape == (1, 3)
    import io
    assert np.loadtxt(io.StringIO("3\n1\n2\n"), delimiter="\n").tolist() == [3, 1, 2]
    import torchtracer  # noqa: F401  (stub or real)
    import matplotlib.pyplot  # noqa: F401


# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("decoder_type,is_crc", [("SC-LUT", False), ("SCL-LUT", False), ("FastSC-LUT", False), ("FastSCL-LUT", False), ("CASCL-LUT", True)])
def test_driver_loop_on_this_package_equals_the_reference(workdir, decoder_type, is_crc):
    """what the script would do with this package installed: same pickles, same seed, every import served by the package.
    The other side is the compiled reference's decoders where it has been built.  Without it they are oracle decoders whose
    positional arguments are named by test_abi.REF_SIGNATURES, the reference's constructor signatures as transcribed from its
    sources; only test_reference_signatures_agree_with_compiled_reference, which needs the reference, checks that
    transcription.  On the LLR-domain tables used here the oracle's decoded words are pinned to the reference's by
    tests/golden/real_lut_n128.npz."""
    from oracle import polar_oracle as po
    from quantized_decoder_polar_codes_b200 import lutgen
    from test_abi import REF_SIGNATURES
    compat.install()
    import importlib
    ours = {k: getattr(importlib.import_module("PolarDecoder.Decoder." + k), k)
            for k in ["SCLUTDecoder", "SCLLUTDecoder", "FastSCLUTDecoder", "FastSCLLUTDecoder", "CASCLLUTDecoder"]}
    PolarEnc = importlib.import_module("PolarBDEnc.Encoder.PolarEnc").PolarEnc
    CRCEnc = importlib.import_module("PolarBDEnc.Encoder.CRCEnc").CRCEnc
    LLRQuantizer = importlib.import_module("quantizers.quantizer.LLROptLSQuantizer").LLRQuantizer
    refmod = po.load_reference()
    if refmod is not None:
        ref = {k: getattr(refmod, k) for k in ours}
    else:
        ref = {k: (lambda *a, k=k: po.OracleDecoder(k, **dict(zip(REF_SIGNATURES[k], a)))) for k in ours}
    frames, seed, A = 60, 11, 32
    args = (workdir, N, A, 8, decoder_type, is_crc, QCU, QD, QC, DESIGN, frames, seed, [0, 2, 4])
    s1, w1 = driver_loop.run(*args, ours, PolarEnc, CRCEnc, LLRQuantizer, pw_sets, node_types, lutgen.channel_llr_density_table)
    s2, w2 = driver_loop.run(*args, ref, NumpyPolarEnc, NumpyCRCEnc, LLRQuantizer, pw_sets, node_types, lutgen.channel_llr_density_table)
    assert s1 == s2                      # BER / BLER counters per Eb/N0 point
    for a, b in zip(w1, w2):
        assert (a == b).all()            # every decoded word
