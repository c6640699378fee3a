"""The Fast-SSC walks of scl_lut_warp on the B200, on the codes of tests/fast_walk.py that reach every special-node shape
of the project's constructions (N = 32..1024): FastSCLUTDecoder, FastSCLLUTDecoder and CAFastSCLLUTDecoder at L = 2, 4, 8,
on AWGN frames with min-sum tables and on a tie alphabet.
  * scl_lut_warp, through pd_decode_device with the debug taps, on a batch of more than two waves (these kernels then
    launch one-wave pieces on two streams): bits, path metrics and winners of a few hundred unique frames equal the
    oracle's, and every tiled copy of them equals the first (the taps of every piece but the first used to be lost);
  * the generic and path_warp kernels, which interpret the same node types, decode the same codes to the oracle's bits."""
import numpy as np
import pytest

import common
import fast_walk as fw
from oracle import polar_oracle as po

pytestmark = pytest.mark.gpu

CASES = fw.decode_cases(1024)
UNIQUE = 256


@pytest.fixture(scope="module")
def q():
    import quantized_decoder_polar_codes_b200 as q
    return q


@pytest.mark.parametrize("name,kind,code,ckw", CASES, ids=[c[0] for c in CASES])
def test_every_kernel_matches_the_oracle(q, name, kind, code, ckw, monkeypatch):
    import torch
    from quantized_decoder_polar_codes_b200 import capi
    L = ckw.get("L", 1)
    kw, x, _ = common.make_case(kind, B=UNIQUE, frozen=fw.frozen_of(code), **ckw)
    want, pm_want, win_want = po.OracleDecoder(kind, **kw).decode(x, return_pm=True)
    dec = getattr(q, kind)(**kw)
    assert dec.kernel == "scl_lut_warp"
    wave = capi.wave_frames(dec, capi.PD_U8)
    assert wave > 0
    B = 2 * wave + UNIQUE // 2 + 1
    reps = -(-B // UNIQUE)
    d_in = torch.from_numpy(np.tile(x.astype(np.uint8), (reps, 1))[:B].copy()).cuda()
    d_out = torch.empty((B, want.shape[1]), dtype=torch.uint8, device="cuda")
    pm = torch.full((B, L), -1.0, dtype=torch.float64, device="cuda")
    win = torch.full((B,), -1, dtype=torch.int32, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    capi.check(capi.lib().pd_set_debug_outputs(dec._handle, pm.data_ptr(), win.data_ptr()))
    try:
        capi.decode_device(dec, d_in.data_ptr(), capi.PD_U8, B, d_out.data_ptr(), s)
        capi.sync_check(dec, s)
    finally:
        capi.check(capi.lib().pd_set_debug_outputs(dec._handle, None, None))
    got, pmg, wing = d_out.cpu().numpy(), pm.cpu().numpy(), win.cpu().numpy()
    assert np.array_equal(got[:UNIQUE], want)
    assert np.array_equal(pmg[:UNIQUE], pm_want)
    assert np.array_equal(wing[:UNIQUE], win_want)
    for a, first in ((got, want), (pmg, pm_want), (wing, win_want)):
        for r in range(1, reps):
            part = a[r * UNIQUE:(r + 1) * UNIQUE]
            assert np.array_equal(part, first[:part.shape[0]]), (r, B)
    # the schedule interpreters, on the unique frames
    for force, kernel in (("1", "generic"), ("2", "path_warp")):
        monkeypatch.setenv("POLAR_B200_FORCE_GENERIC", force)
        other = getattr(q, kind)(**kw)
        assert other.kernel == kernel
        assert np.array_equal(other.decode(x), want), kernel
