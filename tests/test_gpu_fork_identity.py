"""The identity exit of the scl_lut_warp fork on the GPU: a decoder with the exit (default) and one without it
(POLAR_B200_KDEBUG=2, read when the decoder is built) give byte-equal bits, path metrics and winners over more than two
waves of the persistent kernel, at the north-star shape (SCL-LUT N=1024 L=8) and at C3's (N=128 L=8); a sample of the
frames also equals the oracle."""
import os

import numpy as np
import pytest

import common
from oracle import polar_oracle as po

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def q():
    import quantized_decoder_polar_codes_b200 as q
    return q


def _build(q, kw, dbg):
    old = os.environ.get("POLAR_B200_KDEBUG")
    os.environ["POLAR_B200_KDEBUG"] = dbg
    try:
        return q.SCLLUTDecoder(**kw)
    finally:
        if old is None:
            del os.environ["POLAR_B200_KDEBUG"]
        else:
            os.environ["POLAR_B200_KDEBUG"] = old


def _run(dec, x, K, L):
    import torch
    from quantized_decoder_polar_codes_b200 import capi
    B = x.shape[0]
    xin = torch.from_numpy(x.astype(np.uint8)).cuda()
    out = torch.empty((B, K), dtype=torch.uint8, device="cuda")
    pm = torch.zeros((B, L), dtype=torch.float64, device="cuda")
    win = torch.zeros(B, dtype=torch.int32, device="cuda")
    capi.check(capi.lib().pd_set_debug_outputs(dec._handle, pm.data_ptr(), win.data_ptr()))
    stream = torch.cuda.current_stream().cuda_stream
    capi.decode_device(dec, xin.data_ptr(), capi.PD_U8, B, out.data_ptr(), stream)
    capi.sync_check(dec, stream)
    capi.check(capi.lib().pd_set_debug_outputs(dec._handle, None, None))
    return out.cpu().numpy(), pm.cpu().numpy(), win.cpu().numpy()


@pytest.mark.parametrize("N,K", [(1024, 512), (128, 32)], ids=["ns", "c3"])
def test_identity_exit_changes_nothing(q, N, K):
    from quantized_decoder_polar_codes_b200 import capi
    L = 8
    kw, _, _ = common.make_case("SCLLUTDecoder", N=N, K=K, L=L, B=1, tables="minsum", ebn0_db=2.0, seed=11)
    dec, ref = _build(q, kw, "0"), _build(q, kw, "2")
    assert dec.kernel == ref.kernel == "scl_lut_warp"
    wave = capi.wave_frames(dec, capi.PD_U8)
    assert wave > 0
    kw, x, _ = common.make_case("SCLLUTDecoder", N=N, K=K, L=L, B=2 * wave + wave // 2 + 7, tables="minsum", ebn0_db=2.0,
                                seed=11)
    got, want = _run(dec, x, K, L), _run(ref, x, K, L)
    for a, b in zip(got, want):
        assert a.tobytes() == b.tobytes()
    s = np.linspace(0, x.shape[0] - 1, 64).astype(np.int64)
    bits, pm, win = po.OracleDecoder("SCLLUTDecoder", **kw).decode(x[s], return_pm=True)
    assert np.array_equal(got[0][s], bits) and np.array_equal(got[1][s], pm) and np.array_equal(got[2][s], win)
