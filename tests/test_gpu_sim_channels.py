"""Channel front ends of the on-device frame generator (pd_sim_set_channel, Simulator.set_channel): the probability-domain
driver's cut of y at the MMI channel quantizer's edges and the continuous-domain driver's QUniform, checked element by
element against numpy on the same draw; the LLR-domain modes unchanged by switching; BLER of device-generated frames against
host-generated ones for C4 and a uniformly quantized list decoder; lutgen.llr_channel_quantizer against the reference's own
channel designs; argument validation; and (without a GPU) the layout of pd_sim_channel against capi.SimChannel."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import common
import real_lut
from quantized_decoder_polar_codes_b200 import simulation as sim

DATA = os.path.join(common.ROOT, "quantized_decoder_polar_codes_b200", "data")


# The drivers' rules in numpy, as tests/test_gpu_sweep.py states them (mmi_channel_frames, c5_case, channel_frames).
def y_rule(y, edges, Q):
    """mainQuantizedDecoder_ProbabilityDomain.py:153-177: y cut at edges = interval_x[channel_lut]"""
    idx = np.searchsorted(edges, y, side="left") - 1
    return np.where(y <= edges[0], 0, np.where(y >= edges[-1], Q - 1, idx)).astype(np.uint8)


def q_uniform(llr, r, v):
    """QUniform, mainQuantizedDecoder_ContinuousDomain.py:29-32"""
    M = (v // 2 - 0.5) * r
    return np.where(np.abs(llr) > M, np.sign(llr) * (M - 0.5 * r), (np.floor(llr / r) + 0.5) * r)


def llr_rule(llr, edges, lut, Q):
    """mainQuantizedDecoder_LLRDomain.py:167-176"""
    idx = np.clip(np.searchsorted(edges[:-1], llr, side="left") - 1, 0, lut.size - 1)
    return np.where(llr <= edges[0], 0, np.where(llr >= edges[-1], Q - 1, lut[idx])).astype(np.uint8)


@pytest.fixture(scope="module")
def q():
    import quantized_decoder_polar_codes_b200 as q
    return q


def _sim(q, N, K, A, crc, channel=None):
    from quantized_decoder_polar_codes_b200.simulate import Simulator
    fm, mm = sim.frozen_mask(N, K)
    dec = q.SCDecoder(N=N, K=K, frozen_bits=fm, message_bits=mm)
    return Simulator(dec, fm, A=A, crc=crc, channel_quantizer=channel)


def _gen(s, sigma, frames, seed, first_frame=0):
    msg, out = s.generate(sigma, frames, seed=seed, first_frame=first_frame)
    return msg.cpu().numpy(), out.cpu().numpy()


def _mmi_edges(eb=2):
    return np.load(os.path.join(DATA, "mmi_n1024_q16_3dB.npz"))[f"chan_A512_eb{eb}/edges"]


@pytest.mark.gpu
def test_y_quantizer_exact_on_every_element(q):
    """sigma = 0.5: llr = 8 y exactly, so the LLR output of the same draw gives y = llr / 8 exactly."""
    from quantized_decoder_polar_codes_b200.simulate import YQuantizer
    s = _sim(q, 1024, 536, 512, True)
    msg0, llr = _gen(s, 0.5, 4000, seed=11, first_frame=7)
    y = llr / 8
    assert np.array_equal(y * 8, llr)
    edges = _mmi_edges()
    s.set_channel(YQuantizer(edges, 16))
    msg1, sym = _gen(s, 0.5, 4000, seed=11, first_frame=7)
    assert sym.dtype == np.uint8
    assert np.array_equal(msg0, msg1)
    want = y_rule(y, edges, 16)
    assert np.array_equal(sym, want)
    assert set(np.unique(want)) == set(range(16))
    # edges taken from this draw's y values: y == edge happens, interior ties go to the lower cell ('left')
    tie_edges = np.sort(np.random.default_rng(3).choice(np.unique(y), 17, replace=False))
    assert np.isin(y, tie_edges[1:-1]).sum() >= 15
    s.set_channel(YQuantizer(tie_edges, 16))
    msg2, sym = _gen(s, 0.5, 4000, seed=11, first_frame=7)
    assert np.array_equal(msg0, msg2)
    assert np.array_equal(sym, y_rule(y, tie_edges, 16))


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [1.0, 1e-3])
def test_uniform_llr_exact_on_every_element(q, scale):
    """QUniform bit for bit (the library builds with -fmad=false and IEEE fp64 division), at the driver's root step for a
    2 dB point and at a step a thousand times smaller."""
    from quantized_decoder_polar_codes_b200.simulate import UniformLLR
    sigma = sim.awgn_sigma(2.0, 0.5)
    r = sim.uniform_quantizer_steps(2, 16, sigma)[0][0] * scale     # the root step depends on sigma only, not on N
    s = _sim(q, 1024, 512, 512, False)
    msg0, llr = _gen(s, sigma, 4000, seed=12)
    s.set_channel(UniformLLR(r, 16))
    msg1, x = _gen(s, sigma, 4000, seed=12)
    assert x.dtype == np.float64
    assert np.array_equal(msg0, msg1)
    assert np.array_equal(x, q_uniform(llr, r, 16))
    M = 7.5 * r
    assert (llr > M).sum() > 0 and (llr < -M).sum() > 0 and (np.abs(llr) <= M).sum() > 0


@pytest.mark.gpu
def test_llr_domain_modes_unchanged_by_switching(q):
    from quantized_decoder_polar_codes_b200.simulate import LLRQuantizer, UniformLLR, YQuantizer
    z = np.load(os.path.join(DATA, "mindistortion_n1024_q16_3dB.npz"))
    edges, lut = z["chan_A512_eb2/edges"], z["chan_A512_eb2/lut"]
    sigma = sim.awgn_sigma(2.0, 0.5)
    created = _sim(q, 1024, 536, 512, True, (edges, lut, 16))
    switched = _sim(q, 1024, 536, 512, True)
    _, llr = _gen(switched, sigma, 3000, seed=13, first_frame=5)
    switched.set_channel(LLRQuantizer(edges, lut, 16))
    ma, a = _gen(created, sigma, 3000, seed=13, first_frame=5)
    mb, b = _gen(switched, sigma, 3000, seed=13, first_frame=5)
    assert a.dtype == b.dtype == np.uint8
    assert np.array_equal(ma, mb) and np.array_equal(a, b)
    assert np.array_equal(a, llr_rule(llr, edges, lut, 16))
    # away and back
    r = sim.uniform_quantizer_steps(2, 16, sigma)[0][0]
    for ch in (YQuantizer(_mmi_edges(), 16), UniformLLR(r, 16), None, LLRQuantizer(edges, lut, 16)):
        switched.set_channel(ch)
        _, out = _gen(switched, sigma, 3000, seed=13, first_frame=5)
        if ch is None:
            assert np.array_equal(out, llr)
    assert np.array_equal(out, a)
    # the same frames however the run is split, in each new mode
    for ch in (YQuantizer(_mmi_edges(), 16), UniformLLR(r, 16)):
        switched.set_channel(ch)
        _, whole = _gen(switched, sigma, 3000, seed=13, first_frame=5)
        _, p1 = _gen(switched, sigma, 1000, seed=13, first_frame=5)
        _, p2 = _gen(switched, sigma, 2000, seed=13, first_frame=1005)
        assert np.array_equal(whole, np.concatenate([p1, p2]))


def _band_agree(res, host_bler, host_frames):
    band = 5 * np.sqrt(max(res["bler"], 1e-3) * (1 - res["bler"]) / host_frames)
    assert abs(res["bler"] - host_bler) < band, (res["bler"], host_bler)


@pytest.mark.gpu
def test_c4_end_to_end_bler(q):
    """C4: CAFastSCLLUTDecoder N=1024 A=512 K=536 L=8 on the MMI tables, frames cut from y on the device vs the numpy rule on
    the host."""
    from quantized_decoder_polar_codes_b200.simulate import Simulator, YQuantizer
    N, A, K, eb = 1024, 512, 536, 2.0
    z = np.load(os.path.join(DATA, "mmi_n1024_q16_3dB.npz"))
    fm, mm = sim.frozen_mask(N, K)
    dec = q.CAFastSCLLUTDecoder(N=N, K=K, A=A, L=8, frozen_bits=fm, message_bits=mm, node_type=sim.identify_nodes(N, fm),
                                LUT_f=[z["lut_f"][p].astype(np.int32)[None] for p in range(N - 1)],
                                LUT_g=[z["lut_g"][p].astype(np.int32)[None] for p in range(N - 1)], virtual_channel_llr=z["llrs"])
    edges = z["chan_A512_eb2/edges"]
    s = Simulator(dec, fm, A=A, crc=True, channel_quantizer=YQuantizer(edges, 16))
    res = s.run(eb, 200000, batch=50000, seed=1)
    assert res["frames"] == 200000 and res["block_errors"] > 0 and res["ber"] < res["bler"]
    rng = np.random.default_rng(21)
    hf = 20000
    msg = rng.integers(0, 2, (hf, A), dtype=np.uint8)
    cw = sim.polar_encode(sim.crc_attach(msg), fm)
    y = (1.0 - 2.0 * cw) + rng.normal(0.0, sim.awgn_sigma(eb, A / N), cw.shape)
    got = dec.decode(y_rule(y, edges, 16).astype(np.float64))
    _band_agree(res, (got != msg).any(axis=1).mean(), hf)
    assert s.run(eb, 200000, batch=50000, seed=1) == res
    early = s.run(0.0, 200000, batch=20000, seed=1, max_block_errors=1000)
    assert early["frames"] < 200000 and early["block_errors"] > 1000


def _uniform_decoder(q, N, K, L, eb, v=16):
    sigma = sim.awgn_sigma(eb, K / N)
    fm, mm = sim.frozen_mask_ga(N, K, sigma)
    r_f, r_g = sim.uniform_quantizer_steps(N, v, sigma)
    dec = q.SCLUniformQuantizedDecoder(N=N, K=K, L=L, frozen_bits=fm, message_bits=mm, decoder_r_f=r_f, decoder_r_g=r_g, v=v)
    return dec, fm, sigma, r_f[0]


@pytest.mark.gpu
def test_uniform_decoder_end_to_end_bler(q):
    """the continuous-domain driver's loop: SCLUniformQuantizedDecoder N=256 K=128 L=8, GA construction, steps at the point's
    sigma, QUniform with the root step on the device vs numpy on the host"""
    from quantized_decoder_polar_codes_b200.simulate import Simulator, UniformLLR
    N, K, eb = 256, 128, 2.0
    dec, fm, sigma, r = _uniform_decoder(q, N, K, 8, eb)
    s = Simulator(dec, fm, A=K, channel_quantizer=UniformLLR(r, 16))
    res = s.run(eb, 200000, batch=50000, seed=2)
    assert res["frames"] == 200000 and res["block_errors"] > 0 and res["ber"] < res["bler"]
    rng = np.random.default_rng(22)
    hf = 20000
    msg = rng.integers(0, 2, (hf, K), dtype=np.uint8)
    got = dec.decode(q_uniform(sim.awgn_llr(sim.polar_encode(msg, fm), sigma, rng), r, 16))
    _band_agree(res, (got != msg).any(axis=1).mean(), hf)
    assert s.run(eb, 200000, batch=50000, seed=2) == res
    early = s.run(-1.0, 200000, batch=20000, seed=2, max_block_errors=1000)
    assert early["frames"] < 200000 and early["block_errors"] > 1000


@pytest.mark.gpu
def test_uniform_decoder_c5_shape(q):
    """N=2048 L=32 (C5): run() counts exactly the errors of decoding the frames generate() gives for the same seed."""
    from quantized_decoder_polar_codes_b200.simulate import Simulator, UniformLLR
    N, K, eb = 2048, 1024, 2.0
    dec, fm, sigma, r = _uniform_decoder(q, N, K, 32, eb)
    s = Simulator(dec, fm, A=K, channel_quantizer=UniformLLR(r, 16))
    res = s.run(eb, 512, batch=256, seed=3)
    msg, x = _gen(s, sigma, 512, seed=3)
    assert x.dtype == np.float64 and x.shape == (512, N)
    got = dec.decode(x)
    assert res["frames"] == 512
    assert res["bit_errors"] == int((got != msg).sum()) and res["block_errors"] == int((got != msg).any(axis=1).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("source,N,A,eb", [("n1024", 1024, 512, e) for e in (1, 2, 3, 4)] + [("n128", 128, 32, e) for e in (1, 2, 3)])
def test_llr_channel_quantizer_matches_reference_designs(source, N, A, eb):
    """the stored channel quantizers were made by the reference's own code (tests/golden/make_real_luts.py and
    make_real_lut_n1024.py)"""
    from quantized_decoder_polar_codes_b200 import lutgen
    if source == "n1024":
        z = np.load(os.path.join(DATA, "mindistortion_n1024_q16_3dB.npz"))
        want_edges, want_lut = z[f"chan_A{A}_eb{eb}/edges"], z[f"chan_A{A}_eb{eb}/lut"]
    else:
        z = real_lut.load()
        want_edges, want_lut = z[f"A{A}_eb{eb}/chan_edges"], z[f"A{A}_eb{eb}/chan_lut"]
    edges, lut = lutgen.llr_channel_quantizer(sim.awgn_sigma(eb, A / N))
    assert edges.dtype == want_edges.dtype and edges.tobytes() == want_edges.tobytes()
    assert lut.dtype == want_lut.dtype and lut.tobytes() == want_lut.tobytes()


@pytest.mark.gpu
def test_set_channel_validation(q):
    from quantized_decoder_polar_codes_b200.simulate import LLRQuantizer, UniformLLR, YQuantizer
    s = _sim(q, 128, 64, 64, False)
    e17 = np.linspace(-2.0, 2.0, 17)
    lut = np.arange(16, dtype=np.uint8)
    bad = [
        (None, "unknown channel mode"),
        (YQuantizer(None, 16), "NULL"),
        (LLRQuantizer(None, lut, 16), "NULL"),
        (LLRQuantizer(e17, None, 16), "NULL"),
        (YQuantizer(e17[:1], 0), "at least 2"),
        (LLRQuantizer(e17[:1], lut[:0], 16), "at least 2"),
        (YQuantizer(e17[::-1], 16), "ascending"),
        (LLRQuantizer(np.where(np.arange(17) == 5, np.nan, e17), lut, 16), "ascending"),
        (YQuantizer(e17, 15), "q_channel \\+ 1"),
        (YQuantizer(np.linspace(-2, 2, 258), 257), "q_channel"),
        (LLRQuantizer(e17, lut, 0), "q_channel"),
        (LLRQuantizer(e17, lut, 300), "q_channel"),
        (LLRQuantizer(e17, lut, 8), "chan_lut"),
        (UniformLLR(0.0, 16), "r="),
        (UniformLLR(-1.0, 16), "r="),
        (UniformLLR(float("inf"), 16), "r="),
        (UniformLLR(float("nan"), 16), "r="),
        (UniformLLR(0.5, 1), "v="),
    ]
    from quantized_decoder_polar_codes_b200 import capi
    for ch, msg in bad:
        if ch is None:      # a mode number no front end has: through the C ABI directly
            raw = capi.SimChannel()
            raw.mode = 7
            with pytest.raises(ValueError, match=msg):
                capi.check(s.lib.pd_sim_set_channel(s._h, C.byref(raw)))
            continue
        with pytest.raises(ValueError, match=msg):
            s.set_channel(ch)
    with pytest.raises(TypeError):
        s.set_channel((e17, lut, 16))
    # a refused call leaves the front end as it was
    assert s.channel is None
    _, out = _gen(s, 0.7, 10, seed=1)
    assert out.dtype == np.float64


def test_sim_channel_layout_matches_header(tmp_path):
    """pd_sim_channel as a C99 compiler lays it out == capi.SimChannel (ctypes)"""
    from quantized_decoder_polar_codes_b200 import capi
    names = [f for f, _ in capi.SimChannel._fields_]
    assert names == ["mode", "edges", "n_edges", "chan_lut", "q_channel", "r", "v"]
    src = tmp_path / "layout.c"
    src.write_text("#include <stdio.h>\n#include <stddef.h>\n#include \"polar_b200.h\"\nint main(void) {\n"
                   "    printf(\"size %zu\\n\", sizeof(pd_sim_channel));\n" +
                   "".join(f"    printf(\"{n} %zu\\n\", offsetof(pd_sim_channel, {n}));\n" for n in names) +
                   "    printf(\"modes %d %d %d %d\\n\", PD_SIM_LLR, PD_SIM_LLR_QUANT, PD_SIM_Y_QUANT, PD_SIM_LLR_UNIFORM);\n"
                   "    return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(common.ROOT, "include"),
                           str(src), "-o", str(exe)])
    got = dict(line.split(" ", 1) for line in subprocess.check_output([str(exe)]).decode().splitlines())
    assert int(got["size"]) == C.sizeof(capi.SimChannel)
    for n in names:
        assert int(got[n]) == getattr(capi.SimChannel, n).offset, n
    assert [int(v) for v in got["modes"].split()] == [capi.PD_SIM_LLR, capi.PD_SIM_LLR_QUANT, capi.PD_SIM_Y_QUANT,
                                                       capi.PD_SIM_LLR_UNIFORM]
