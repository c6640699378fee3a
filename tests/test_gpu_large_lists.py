"""List sizes 64, 128 and 256 on the GPU (the path_cta kernel, one CTA per frame, one thread per path): bit-exact parity
with the oracle for all nine list classes, the host pipeline and multi-device dealing, the debug taps, the on-device
simulator, and the largest shape (N = 4096, L = 256)."""
import numpy as np
import pytest

import common
from oracle import polar_oracle as po

pytestmark = pytest.mark.gpu

LS = (64, 128, 256)
NS = (32, 64, 128, 256)
KINDS = sorted(common.LIST_KINDS)


@pytest.fixture(scope="module")
def q():
    import quantized_decoder_polar_codes_b200 as q
    return q


def _shape(kind, N):
    """(K, A) of a half-rate code; the CA kinds carry 24 CRC bits, so at N = 32 their message is 4 bits."""
    if kind in common.CA_KINDS:
        K = N // 2 + 24 if N >= 64 else 28
        return K, K - 24
    return N // 2, None


def _check(q, kind, kw, x):
    dec = getattr(q, kind)(**kw)
    assert dec.kernel == "path_cta"
    got = dec.decode(x)
    want = po.OracleDecoder(kind, **kw).decode(x)
    bad = int((got != want).any(axis=1).sum())
    assert bad == 0, f"{bad}/{x.shape[0]} frames differ from the oracle"


# every class x list size x input kind, the code length cycling through NS so that each (class, N) pair appears
_CASES = [(kind, L, tables, NS[(i + j + 2 * t) % len(NS)])
          for i, kind in enumerate(KINDS) for j, L in enumerate(LS) for t, tables in enumerate(("random", "working"))]


@pytest.mark.parametrize("kind,L,tables,N", _CASES, ids=[f"{k}-L{L}-{t}-N{N}" for k, L, t, N in _CASES])
def test_matches_oracle(q, kind, L, tables, N):
    """random: tie-heavy tables / coarse-grid LLRs (common.make_case), which send most forks to the exact sort;
    working: encode + AWGN frames (min-sum LUT tables or fp64 LLRs), which run the parallel rank."""
    K, A = _shape(kind, N)
    t = "random" if tables == "random" else ("minsum" if "LUT" in kind else "channel")
    B = 300 if N * L <= 64 * 128 else 120
    kw, x, _ = common.make_case(kind, N, K, L=L, A=A, B=B, seed=N + L, tables=t, ebn0_db=1.0)
    _check(q, kind, kw, x)


@pytest.mark.parametrize("kind", KINDS)
def test_matches_oracle_at_n1024(q, kind):
    L = LS[KINDS.index(kind) % len(LS)]
    K = 536 if kind in common.CA_KINDS else 512
    t = "minsum" if "LUT" in kind else "channel"
    kw, x, _ = common.make_case(kind, 1024, K, L=L, B=3, seed=11, tables=t, ebn0_db=1.0)
    _check(q, kind, kw, x)


@pytest.mark.parametrize("kind", ["SCLLUTDecoder", "SCLDecoder", "FastSCLLUTDecoder", "SCLUniformQuantizedDecoder"])
@pytest.mark.parametrize("L", [64, 256])
def test_more_paths_than_codewords(q, kind, L):
    """L > 2^K: the list never fills, dead paths (PM = pm_init) tie with each other up to the last bit."""
    kw, x, _ = common.make_case(kind, 32, 5, L=L, B=200, seed=L)
    _check(q, kind, kw, x)


def test_host_paths_and_devices_agree_with_the_device_path(q, monkeypatch):
    import torch
    from quantized_decoder_polar_codes_b200 import capi
    kind, N, L = "SCLLUTDecoder", 128, 64
    kw, x, _ = common.make_case(kind, N, 64, L=L, B=700, seed=5)
    dec = q.SCLLUTDecoder(**kw)
    assert dec.kernel == "path_cta"
    want = po.OracleDecoder(kind, **kw).decode(x)
    xin = torch.from_numpy(x.astype(np.uint8)).cuda()
    out = torch.empty((x.shape[0], 64), dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    capi.decode_device(dec, xin.data_ptr(), capi.PD_U8, x.shape[0], out.data_ptr(), stream)
    capi.sync_check(dec, stream)
    dev = out.cpu().numpy()
    assert (dev == want).all()
    assert capi.wave_frames(dec, capi.PD_U8) >= 148
    for xx in (x.astype(np.uint8), x.astype(np.int32), x.astype(np.float64)):
        assert (dec.decode(xx) == dev).all()
    monkeypatch.setenv("POLAR_B200_CHUNK_FRAMES", "97")     # many pipeline chunks, dealt over two units
    dec.set_devices([0, 0])
    assert (dec.decode(x.astype(np.int32)) == dev).all()
    assert (dec.decode(x.astype(np.uint8)) == dev).all()


def test_out_of_range_symbol_raises(q):
    import torch
    from quantized_decoder_polar_codes_b200 import capi
    kw, x, _ = common.make_case("CASCLLUTDecoder", 64, 40, L=128, A=16, B=8, seed=3)
    dec = q.CASCLLUTDecoder(**kw)
    bad = x.copy()
    bad[2, 5] = 16
    with pytest.raises(ValueError, match="outside the root lookup table"):
        dec.decode(bad)
    xin = torch.from_numpy(bad.astype(np.uint8)).cuda()
    out = torch.empty((8, 16), dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    capi.decode_device(dec, xin.data_ptr(), capi.PD_U8, 8, out.data_ptr(), stream)
    with pytest.raises(ValueError, match="outside the root lookup table"):
        capi.sync_check(dec, stream)
    assert (dec.decode(x) == po.OracleDecoder("CASCLLUTDecoder", **kw).decode(x)).all()   # still usable


@pytest.mark.parametrize("L", LS)
def test_debug_taps_match_the_oracle(q, L):
    import torch
    from quantized_decoder_polar_codes_b200 import capi
    kw, x, _ = common.make_case("SCLDecoder", 128, 64, L=L, B=100, seed=9, tables="channel", ebn0_db=1.0)
    want, pm_want, win_want = po.OracleDecoder("SCLDecoder", **kw).decode(x, return_pm=True)
    dec = q.SCLDecoder(**kw)
    xin = torch.from_numpy(x.astype(np.float64)).cuda()
    out = torch.empty((x.shape[0], 64), dtype=torch.uint8, device="cuda")
    pm = torch.zeros((x.shape[0], L), dtype=torch.float64, device="cuda")
    win = torch.zeros(x.shape[0], dtype=torch.int32, device="cuda")
    capi.check(capi.lib().pd_set_debug_outputs(dec._handle, pm.data_ptr(), win.data_ptr()))
    stream = torch.cuda.current_stream().cuda_stream
    capi.decode_device(dec, xin.data_ptr(), capi.PD_F64, x.shape[0], out.data_ptr(), stream)
    capi.sync_check(dec, stream)
    capi.check(capi.lib().pd_set_debug_outputs(dec._handle, None, None))
    assert (out.cpu().numpy() == want).all()
    assert (pm.cpu().numpy() == pm_want).all()
    assert (win.cpu().numpy() == win_want).all()


def test_simulator_counts_the_oracles_errors(q):
    import torch
    from quantized_decoder_polar_codes_b200 import simulation as sim
    from quantized_decoder_polar_codes_b200.simulate import Simulator
    N, K, A, L = 128, 64, 40, 128
    kw, _, _ = common.make_case("CASCLDecoder", N, K, L=L, A=A, B=1)
    dec = q.CASCLDecoder(**kw)
    s = Simulator(dec, kw["frozen_bits"], A=A, crc=True)
    ebn0, frames, batch, seed = 1.0, 600, 250, 4
    res = s.run(ebn0, frames, batch=batch, seed=seed)
    sigma = sim.awgn_sigma(ebn0, A / N)
    oracle = po.OracleDecoder("CASCLDecoder", **kw)
    be = ble = 0
    for f0 in range(0, frames, batch):
        msg, llr = s.generate(sigma, min(batch, frames - f0), seed=seed, first_frame=f0)
        torch.cuda.synchronize()
        err = oracle.decode(llr.cpu().numpy()) != msg.cpu().numpy()
        be += int(err.sum())
        ble += int(err.any(axis=1).sum())
    assert ble > 0
    assert (res["frames"], res["bit_errors"], res["block_errors"]) == (frames, be, ble)


def test_largest_shape(q):
    """SCLDecoder N = 4096, L = 256: 158.5 KB of shared memory per CTA (the partial sums alone 128 KB) and 8 MB of
    workspace per CTA, so the grid is capped below one CTA per SM by the 1 GiB workspace budget."""
    import torch
    from quantized_decoder_polar_codes_b200 import capi
    kw, x, _ = common.make_case("SCLDecoder", 4096, 2048, L=256, B=2 * 148 + 40, seed=21, tables="channel", ebn0_db=1.5,
                                construction="pw")
    dec = q.SCLDecoder(**kw)
    assert dec.kernel == "path_cta"
    wave = capi.wave_frames(dec, capi.PD_F64)
    assert 0 < wave < x.shape[0] // 2
    got = dec.decode(x)
    assert (got[:1] == po.OracleDecoder("SCLDecoder", **kw).decode(x[:1])).all()
    xin = torch.from_numpy(x).cuda()
    out = torch.empty((x.shape[0], 2048), dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    capi.decode_device(dec, xin.data_ptr(), capi.PD_F64, x.shape[0], out.data_ptr(), stream)   # overlapping one-wave pieces
    capi.sync_check(dec, stream)
    assert (out.cpu().numpy() == got).all()
    parts = np.concatenate([dec.decode(x[a:b]) for a, b in ((0, 2), (2, 150), (150, x.shape[0]))])
    assert (parts == got).all()
