"""Shared case generator for the parity tests: seeded constructor arguments + inputs for every decoder class.

`make_case(...)` returns (ctor_kwargs, x) with numpy tables; `ref_kwargs(...)` turns them into the plain
nested lists the compiled reference (oracle/_ref) needs.  Random tables with tiny LLR alphabets force
path-metric and |LLR| ties on almost every frame (SURVEY.md App. B1), which is what separates a merely
correct decoder from a bit-exact one.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from quantized_decoder_polar_codes_b200 import simulation as sim  # noqa: E402

ALL_KINDS = [
    "SCDecoder", "FastSCDecoder", "SCLDecoder", "FastSCLDecoder", "CASCLDecoder",
    "SCLUTDecoder", "FastSCLUTDecoder", "SCLLUTDecoder", "FastSCLLUTDecoder", "CASCLLUTDecoder",
    "CAFastSCLLUTDecoder", "SCUniformQuantizedDecoder", "SCLUniformQuantizedDecoder",
    "SCLloydQuantizedDecoder", "SCLLloydQuantizedDecoder",
]
LIST_KINDS = {"SCLDecoder", "FastSCLDecoder", "CASCLDecoder", "SCLLUTDecoder", "FastSCLLUTDecoder",
              "CASCLLUTDecoder", "CAFastSCLLUTDecoder", "SCLUniformQuantizedDecoder", "SCLLloydQuantizedDecoder"}
CA_KINDS = {"CASCLDecoder", "CASCLLUTDecoder", "CAFastSCLLUTDecoder"}
TIE_ALPHABET = (-2.0, -1.0, -0.5, 0.0, 0.5, 1.0, 2.0)


def make_case(kind, N, K, L=8, A=None, B=64, Q=16, Qc=None, seed=0, tables="random", alphabet=TIE_ALPHABET,
              per_position=False, share=True, v=16, construction="nr", ebn0_db=2.0, llr_levels=None, frozen=None):
    """Returns (kwargs, x, truth) -- truth is the transmitted info word when the inputs come from a real
    encode+AWGN chain (tables == "minsum" or the float family with channel=True), else None.
    `frozen` (int mask, 1 = frozen, K zeros) replaces the frozen set of `construction`."""
    rng = np.random.default_rng(seed)
    if frozen is None:
        fm, mm = sim.frozen_mask(N, K, construction)
    else:
        fm = np.asarray(frozen, np.int32)
        assert fm.shape == (N,) and int((fm == 0).sum()) == K
        mm = (1 - fm).astype(np.int32)
    kw = dict(N=N, K=K, frozen_bits=fm, message_bits=mm)
    if kind in LIST_KINDS:
        kw["L"] = L
    if kind in CA_KINDS:
        kw["A"] = K - 24 if A is None else A
    if kind in ("CASCLDecoder", "CASCLLUTDecoder"):
        kw.update(crc_n=24, crc_p=list(sim.CRC24_LOC))
    if "Fast" in kind:
        kw["node_type"] = sim.identify_nodes(N, fm)
    truth = None
    if "LUT" in kind:
        if tables == "minsum":
            f, g, llr = sim.minsum_lut_tables(N, Q, Qc, delta=1.0, per_position=per_position, levels=llr_levels)
            msg = rng.integers(0, 2, (B, kw.get("A", K)), dtype=np.uint8)
            word = sim.crc_attach(msg) if kind in CA_KINDS else msg
            cw = sim.polar_encode(word, fm)
            sigma = sim.awgn_sigma(ebn0_db, kw.get("A", K) / N)
            x = sim.quantize_uniform(sim.awgn_llr(cw, sigma, rng), Qc or Q, 1.0).astype(np.int32)
            truth = msg if kind in CA_KINDS else word
        else:
            f, g, llr = sim.random_lut_tables(N, Q, Qc, rng=rng, llr_alphabet=alphabet, per_position=per_position,
                                              share=share, levels=llr_levels)
            x = rng.integers(0, Qc or Q, (B, N)).astype(np.int32)
        name_f, name_g = ("LUT_Fs", "LUT_Gs") if kind == "FastSCLUTDecoder" else ("LUT_f", "LUT_g")
        kw[name_f], kw[name_g], kw["virtual_channel_llr"] = f, g, llr
    else:
        if tables == "channel":
            msg = rng.integers(0, 2, (B, kw.get("A", K)), dtype=np.uint8)
            word = sim.crc_attach(msg) if kind in CA_KINDS else msg
            cw = sim.polar_encode(word, fm)
            sigma = sim.awgn_sigma(ebn0_db, kw.get("A", K) / N)
            x = sim.awgn_llr(cw, sigma, rng)
            truth = msg if kind in CA_KINDS else word
        else:
            x = np.round(rng.standard_normal((B, N)) * 4) / 2  # coarse grid: ties and exact zeros
        if "Uniform" in kind:
            kw.update(decoder_r_f=rng.uniform(0.3, 1.0, N - 1), decoder_r_g=rng.uniform(0.3, 1.0, N - 1), v=v)
        if "Lloyd" in kind:
            def mk():
                b = np.sort(rng.uniform(-8, 8, (N - 1, v + 1)), axis=1)
                b[:, 0], b[:, -1] = -1e300, 1e300
                return b, np.sort(rng.uniform(-8, 8, (N - 1, v)), axis=1)
            bf, rf = mk()
            bg, rg = mk()
            kw.update(boundaries_f=bf, boundaries_g=bg, reconstruction_f=rf, reconstruction_g=rg, v=v)
    return kw, x, truth


def ref_kwargs(kw):
    """numpy -> nested lists, with per-position LUT replication where the compact form was used."""
    out = {}
    N = kw["N"]
    for k, val in kw.items():
        if k in ("LUT_f", "LUT_g", "LUT_Fs", "LUT_Gs"):
            lst = []
            for p, t in enumerate(val):
                t = np.asarray(t)
                d = int(np.floor(np.log2(p + 1)))
                npos = N >> (d + 1)
                if t.shape[0] == 1 and npos > 1:
                    t = np.broadcast_to(t, (npos,) + t.shape[1:])
                lst.append(t.tolist())
            out[k] = lst
        elif isinstance(val, np.ndarray):
            out[k] = val.tolist()
        else:
            out[k] = val
    return out


def ref_decode(refmod, kind, kw, x):
    dec = getattr(refmod, kind)(**ref_kwargs(kw))
    xx = x.astype(np.int32) if "LUT" in kind else x.astype(np.float64)
    return np.stack([np.asarray(dec.decode(xx[i])) for i in range(xx.shape[0])])
