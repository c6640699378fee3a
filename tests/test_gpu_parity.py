"""GPU parity tests (run with -m gpu on a B200): the CUDA decoders, called through the pybind11 mirror of the
reference API and through the C ABI, against (a) the committed golden vectors produced by the compiled
reference and (b) the CPU oracle on larger seeded batches.  Bit-exact for every class on these inputs; for the
float family the stated tolerance of BASELINE.json (fp-tie frames <= 1e-6, PM within 1e-5 relative) is checked
explicitly in test_float_path_metrics."""
import ctypes

import numpy as np
import pytest

import common
import fast_walk
from golden.cases import CASES
from oracle import polar_oracle as po

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def q():
    import quantized_decoder_polar_codes_b200 as q
    return q


def _build(q, kind, kw):
    return getattr(q, kind)(**kw)


@pytest.mark.parametrize("cid,ckw", CASES, ids=[c[0] for c in CASES])
def test_cuda_matches_golden(q, golden, cid, ckw):
    ckw = dict(ckw)
    kind = ckw.pop("kind")
    kw, x, _ = common.make_case(kind, **ckw)
    shape = tuple(golden[cid + "/shape"])
    want = np.unpackbits(golden[cid + "/out"], axis=1)[:, : shape[1]]
    dec = _build(q, kind, kw)
    got = dec.decode(x)
    assert got.shape == shape and got.dtype == np.uint8
    bad = int((got != want).any(axis=1).sum())
    assert bad == 0, f"{bad}/{shape[0]} frames differ from the reference ({dec.kernel})"


BIG = [
    ("SCDecoder", dict(N=128, K=64, B=4000)),
    ("FastSCDecoder", dict(N=256, K=128, B=4000)),
    ("SCLDecoder", dict(N=128, K=64, L=8, B=1500)),
    ("FastSCLDecoder", dict(N=128, K=64, L=8, B=1500)),
    ("CASCLDecoder", dict(N=128, K=64, L=8, A=40, B=1500)),
    ("SCLUTDecoder", dict(N=128, K=32, B=4000)),
    ("FastSCLUTDecoder", dict(N=256, K=128, B=4000)),
    ("SCLLUTDecoder", dict(N=128, K=32, L=8, B=3000)),
    ("SCLLUTDecoder", dict(N=128, K=64, L=2, B=1500)),
    ("SCLLUTDecoder", dict(N=128, K=64, L=4, B=1500)),
    ("SCLLUTDecoder", dict(N=64, K=32, L=5, B=1000)),
    ("SCLLUTDecoder", dict(N=256, K=128, L=16, B=300)),
    ("FastSCLLUTDecoder", dict(N=256, K=128, L=8, B=1500)),
    ("FastSCLLUTDecoder", dict(N=512, K=300, L=8, B=300)),       # an R1 node of 64 leaves at depth 3 -> path_warp
    ("CASCLLUTDecoder", dict(N=128, K=64, L=8, A=40, B=1500)),
    ("CAFastSCLLUTDecoder", dict(N=256, K=128 + 24, L=8, A=128, B=1000)),
    ("SCUniformQuantizedDecoder", dict(N=128, K=64, B=3000)),
    ("SCLUniformQuantizedDecoder", dict(N=128, K=64, L=8, B=1000)),
    ("SCLloydQuantizedDecoder", dict(N=128, K=64, B=3000)),
    ("SCLLloydQuantizedDecoder", dict(N=128, K=64, L=8, B=1000)),
    ("SCLLUTDecoder", dict(N=1024, K=512, L=8, B=300)),
    ("SCLUTDecoder", dict(N=1024, K=512, B=1000)),
    ("CAFastSCLLUTDecoder", dict(N=1024, K=536, A=512, L=8, B=200)),
    ("FastSCLLUTDecoder", dict(N=1024, K=768, L=8, B=100)),       # high rate: R1 nodes > 32 leaves -> path_warp
    ("FastSCLLUTDecoder", dict(N=1024, K=512, L=4, B=200)),
    ("FastSCLLUTDecoder", dict(N=256, K=64, L=2, B=500)),
    ("FastSCLUTDecoder", dict(N=1024, K=700, B=1000)),            # wide R1 / SPC nodes in the non-list warp path
    ("FastSCLUTDecoder", dict(N=64, K=40, B=1000)),
    # fp64 LLR family at large N (workspace levels beyond L2 reach)
    ("SCDecoder", dict(N=1024, K=512, B=300)),
    ("FastSCDecoder", dict(N=1024, K=700, B=300)),
    ("SCLDecoder", dict(N=1024, K=512, L=8, B=60)),
    ("FastSCLDecoder", dict(N=512, K=256, L=4, B=100)),
    ("CASCLDecoder", dict(N=512, K=280, A=256, L=8, B=60)),
    ("FastSCLDecoder", dict(N=2048, K=1500, L=2, B=30)),
    ("SCLUTDecoder", dict(N=32, K=16, B=1000)),
    ("SCLLUTDecoder", dict(N=32, K=16, L=8, B=1000)),
    ("SCLLUTDecoder", dict(N=2048, K=1024, L=8, B=60, construction="pw")),
    ("SCLLUTDecoder", dict(N=4096, K=2048, L=4, B=30, construction="pw")),
]


@pytest.mark.parametrize("kind,ckw", BIG, ids=[f"{k}-N{c['N']}-L{c.get('L', 1)}" for k, c in BIG])
@pytest.mark.parametrize("tables", ["random", "working"])
def test_cuda_matches_oracle(q, kind, ckw, tables):
    t = "random" if tables == "random" else ("minsum" if "LUT" in kind else "channel")
    kw, x, _ = common.make_case(kind, seed=77, tables=t, ebn0_db=1.0, **ckw)
    want = po.OracleDecoder(kind, **kw).decode(x)
    dec = _build(q, kind, kw)
    if kind.startswith(("FastSCLUT", "FastSCLLUT", "CAFastSCLLUT")):   # the Fast LUT classes: on scl_lut_warp unless a list R1 node is too wide
        _, _, eligible, _ = fast_walk.fast_walk(kw["N"], kw["frozen_bits"], kw.get("L", 1))
        assert dec.kernel == ("scl_lut_warp" if eligible else "path_warp")
    got = dec.decode(x)
    bad = int((got != want).any(axis=1).sum())
    assert bad == 0, f"{bad}/{x.shape[0]} frames differ from the oracle ({dec.kernel})"


_WARP_KINDS = ("SCLUTDecoder", "SCLLUTDecoder", "CASCLLUTDecoder", "FastSCLUTDecoder", "FastSCLLUTDecoder", "CAFastSCLLUTDecoder")


@pytest.mark.parametrize("kind,ckw", [b for b in BIG if b[0] in _WARP_KINDS and b[1]["N"] <= 512],
                         ids=lambda v: v if isinstance(v, str) else f"N{v['N']}-L{v.get('L', 1)}")
def test_generic_kernel_still_covers_the_fast_kernels_classes(q, kind, ckw, monkeypatch):
    """The specialised warp kernel takes over the LUT SC/SCL classes; the schedule-driven generic kernel must
    stay bit-exact on them too (it is what runs for table shapes the specialised kernel does not accept)."""
    monkeypatch.setenv("POLAR_B200_FORCE_GENERIC", "1")
    kw, x, _ = common.make_case(kind, seed=78, **ckw)
    dec = _build(q, kind, kw)
    assert dec.kernel == "generic"
    want = po.OracleDecoder(kind, **kw).decode(x)
    assert (dec.decode(x) == want).all()


@pytest.mark.parametrize("force,kernel", [("1", "generic"), ("2", "path_warp")])
@pytest.mark.parametrize("kind,ckw", [
    ("SCDecoder", dict(N=128, K=64, B=500)), ("FastSCDecoder", dict(N=256, K=128, B=500)),
    ("SCLDecoder", dict(N=128, K=64, L=8, B=300)), ("FastSCLDecoder", dict(N=256, K=150, L=8, B=300)),
    ("CASCLDecoder", dict(N=128, K=64, L=4, A=40, B=300)), ("SCLUniformQuantizedDecoder", dict(N=128, K=64, L=16, B=100)),
    ("SCLLloydQuantizedDecoder", dict(N=128, K=64, L=32, B=60)), ("SCLLUTDecoder", dict(N=256, K=128, L=32, B=60)),
    ("FastSCLLUTDecoder", dict(N=512, K=384, L=16, B=60)), ("CAFastSCLLUTDecoder", dict(N=256, K=152, A=128, L=8, B=200)),
    ("FastSCLUTDecoder", dict(N=256, K=128, B=500)), ("CASCLLUTDecoder", dict(N=128, K=64, A=40, L=2, B=300)),
], ids=lambda v: v if isinstance(v, str) else f"N{v['N']}-L{v.get('L', 1)}")
def test_both_schedule_interpreters(q, kind, ckw, force, kernel, monkeypatch):
    """The CTA-per-frame generic kernel and the warp-level path kernel interpret the same schedule; both must be
    bit-exact for every class (whichever one a given shape is routed to by default)."""
    monkeypatch.setenv("POLAR_B200_FORCE_GENERIC", force)
    kw, x, _ = common.make_case(kind, seed=79, **ckw)
    dec = _build(q, kind, kw)
    assert dec.kernel == kernel
    want = po.OracleDecoder(kind, **kw).decode(x)
    got = dec.decode(x)
    bad = int((got != want).any(axis=1).sum())
    assert bad == 0, f"{bad}/{x.shape[0]} frames differ ({dec.kernel})"


@pytest.mark.parametrize("L", [16, 32])
@pytest.mark.parametrize("kind", ["FastSCLDecoder", "FastSCLLUTDecoder", "CAFastSCLLUTDecoder"])
def test_fast_list_r1_exposes_dead_path_order(q, kind, L, monkeypatch):
    """Regression (found by tests/fuzz_parity.py): in the Fast list kinds the R1 rule flips the bit named by the
    ordering the DESTINATION slot held before the permutation (FastSCLDecoder.cpp:197-233), so the position of dead
    (PM = inf) paths after a fork is observable; for 2L > 16 the warp kernel must use the exact std::sort order
    even when no live keys tie.  Short, low-rate code so that the list fills late and dead paths meet R1 nodes."""
    monkeypatch.setenv("POLAR_B200_FORCE_GENERIC", "2")
    ckw = dict(N=64, K=54 if kind.startswith("CA") else 30, L=L, B=200, seed=671108, share=False, per_position=True)
    if kind.startswith("CA"):
        ckw["A"] = 30
    kw, x, _ = common.make_case(kind, **ckw)
    dec = _build(q, kind, kw)
    assert dec.kernel == "path_warp"
    want = po.OracleDecoder(kind, **kw).decode(x)
    assert (dec.decode(x) == want).all()


import real_lut


@pytest.mark.parametrize("tag,kind", real_lut.CASES, ids=[f"{t}-{k}" for t, k in real_lut.CASES])
def test_cuda_matches_reference_on_real_mindistortion_luts(q, tag, kind):
    """BASELINE.json configs 2/3 with REAL MinDistortion tables (reference generator code) on AWGN frames
    quantized with the driver's channel quantizer: bit-exact vs the compiled reference's outputs, and the
    BLER computed from our decoder equals the reference's (identical decisions => identical curves)."""
    kw, x, want, msg = real_lut.build_kwargs(real_lut.load(), tag, kind)
    dec = _build(q, kind, kw)
    got = dec.decode(x)
    assert (got == want).all(), dec.kernel
    assert (got != msg).any(axis=1).mean() == (want != msg).any(axis=1).mean()


@pytest.mark.parametrize("kind,ckw", [
    ("FastSCLUTDecoder", dict(N=128, K=64, B=400000)),
    ("SCLUTDecoder", dict(N=128, K=64, B=400000)),
    ("FastSCLLUTDecoder", dict(N=128, K=64, L=8, B=60000)),
    ("CAFastSCLLUTDecoder", dict(N=128, K=64, A=40, L=4, B=60000)),
    ("SCLLUTDecoder", dict(N=128, K=64, L=2, B=120000)),
], ids=lambda v: v if isinstance(v, str) else f"B{v['B']}")
def test_persistent_ctas_run_several_passes(q, kind, ckw):
    """Batches large enough that every (persistent, one-warp) CTA decodes several frame groups back to back: the
    table/op stream must wrap exactly at the pass boundary (a Fast-SSC walk can end in the middle of a chunk)."""
    kw, x, _ = common.make_case(kind, seed=80, tables="minsum", ebn0_db=1.0, **ckw)
    dec = _build(q, kind, kw)
    assert dec.kernel == "scl_lut_warp"
    got = dec.decode(x.astype(np.uint8))
    want = po.OracleDecoder(kind, **kw).decode(x)
    bad = int((got != want).any(axis=1).sum())
    assert bad == 0, f"{bad}/{x.shape[0]} frames differ"


def test_north_star_workload_of_the_benchmark(q):
    """Exactly what bench.py decodes: SCL-LUT N=1024 A=512 L=8 with the REAL MinDistortion tables (reference
    generator code) and the driver's channel quantizer at 2 dB -- bit-exact vs the oracle (which equals the compiled
    reference on these tables, tests/test_oracle.py), and a sane BLER."""
    import bench
    kw, sym, msg = bench.make_workload(bench.CONFIGS["NS"], 600, seed=3)
    dec = q.SCLLUTDecoder(**kw)
    assert dec.kernel == "scl_lut_warp"
    got = dec.decode(sym)
    want = po.OracleDecoder("SCLLUTDecoder", **kw).decode(sym.astype(np.int32))
    assert (got == want).all()
    assert (got != msg).any(axis=1).mean() < 0.2


def test_reference_call_conventions(q):
    """(N,), (1,N), float64 symbols (forcecast like py::array_t<int>), uint8 fast path, batch of one."""
    kw, x, _ = common.make_case("SCLLUTDecoder", N=128, K=32, L=8, B=8, seed=3)
    want = po.OracleDecoder("SCLLUTDecoder", **kw).decode(x)
    dec = q.SCLLUTDecoder(**kw)
    y1 = dec.decode(x[0])
    assert y1.shape == (32,) and (y1 == want[0]).all()
    assert (dec.decode(x[0][None, :]) == want[0]).all() and dec.decode(x[0][None, :]).shape == (32,)
    assert (dec.decode(x[1].astype(np.float64)) == want[1]).all()           # ProbabilityDomain driver passes float64
    assert (dec.decode(channel_quantized_symbols=x[2].tolist()) == want[2]).all()
    assert (dec.decode(x.astype(np.uint8)) == want).all()
    kwf, xf, _ = common.make_case("SCDecoder", N=128, K=64, B=4, seed=4)
    wantf = po.OracleDecoder("SCDecoder", **kwf).decode(xf)
    decf = q.SCDecoder(**kwf)
    assert (decf.decode(llr=xf[0][None, :]) == wantf[0]).all()              # mainFPDecoder.py passes (1,N) float64
    assert (decf.decode(xf.astype(np.float32)) == po.OracleDecoder("SCDecoder", **kwf).decode(xf.astype(np.float32).astype(np.float64))).all()


def test_out_of_range_symbol_is_an_error(q):
    kw, x, _ = common.make_case("SCLUTDecoder", N=64, K=32, B=4, seed=3)
    dec = q.SCLUTDecoder(**kw)
    x = x.copy()
    x[2, 5] = 16
    with pytest.raises(ValueError, match="outside the root lookup table"):
        dec.decode(x)
    x[2, 5] = 3
    dec.decode(x)  # decoder stays usable


def test_bad_tables_are_rejected(q):
    kw, x, _ = common.make_case("SCLUTDecoder", N=64, K=32, B=4, seed=3)
    f = [np.array(t) for t in kw["LUT_f"]]
    f[5][0, 2, 3] = 16
    kw2 = dict(kw, LUT_f=f)
    with pytest.raises(ValueError, match="consumer alphabet"):
        q.SCLUTDecoder(**kw2)


def test_float_path_metrics(q):
    """BASELINE.json: float decoders must match decoded bits except fp-tie frames (<=1e-6 of frames) and path
    metrics within 1e-5 relative.  Our fp64 kernels evaluate the reference's expressions in the reference's
    order, so both hold with zero slack on these inputs; the tolerance is still the stated one."""
    import torch
    from quantized_decoder_polar_codes_b200 import capi
    for kind in ["SCLDecoder", "FastSCLDecoder", "SCLUniformQuantizedDecoder", "SCLLUTDecoder"]:
        kw, x, _ = common.make_case(kind, N=256, K=128, L=8, B=500, seed=9, tables="minsum" if "LUT" in kind else "channel", ebn0_db=1.0)
        want, pm_want, win_want = po.OracleDecoder(kind, **kw).decode(x, return_pm=True)
        dec = _build(q, kind, kw)
        lut = "LUT" in kind
        xin = torch.from_numpy(x.astype(np.uint8) if lut else x.astype(np.float64)).cuda()
        out = torch.empty((x.shape[0], 128), dtype=torch.uint8, device="cuda")
        pm = torch.zeros((x.shape[0], 8), dtype=torch.float64, device="cuda")
        win = torch.zeros(x.shape[0], dtype=torch.int32, device="cuda")
        capi.check(capi.lib().pd_set_debug_outputs(dec._handle, pm.data_ptr(), win.data_ptr()))
        stream = torch.cuda.current_stream().cuda_stream
        capi.decode_device(dec, xin.data_ptr(), capi.PD_U8 if lut else capi.PD_F64, x.shape[0], out.data_ptr(), stream)
        capi.sync_check(dec, stream)
        capi.check(capi.lib().pd_set_debug_outputs(dec._handle, None, None))
        got = out.cpu().numpy()
        mism = (got != want).any(axis=1).mean()
        assert mism <= 1e-6
        pmg = pm.cpu().numpy()
        fin = np.isfinite(pm_want) & (np.abs(pm_want) < 1e299)
        assert np.allclose(pmg[fin], pm_want[fin], rtol=1e-5, atol=0)
        assert (win.cpu().numpy() == win_want).all()


def test_error_counters(q):
    import torch
    from quantized_decoder_polar_codes_b200 import capi
    rng = np.random.default_rng(0)
    a = rng.integers(0, 2, (1000, 37), dtype=np.uint8)
    b = a.copy()
    flips = rng.random(a.shape) < 0.01
    b[flips] ^= 1
    ta, tb = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
    cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
    capi.check(capi.lib().pd_count_errors(ta.data_ptr(), tb.data_ptr(), 1000, 37, cnt.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert cnt.cpu().tolist() == [int(flips.sum()), int(flips.any(axis=1).sum())]
    # rows of a multiple of 16 bytes take the vector path (one warp per frame, 16 bytes per lane); any byte values count
    for B, n in ((5000, 512), (333, 48), (70, 1024)):
        a = rng.integers(0, 256, (B, n), dtype=np.uint8)
        b = a.copy()
        flips = rng.random(a.shape) < 0.003
        b[flips] = (b[flips].astype(np.int32) + rng.integers(1, 256, int(flips.sum()))).astype(np.uint8)
        ta, tb = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
        cnt.zero_()
        capi.check(capi.lib().pd_count_errors(ta.data_ptr(), tb.data_ptr(), B, n, cnt.data_ptr(), torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        assert cnt.cpu().tolist() == [int(flips.sum()), int(flips.any(axis=1).sum())]


def test_properties_at_full_size(q):
    """North-star shape at a batch the oracle cannot follow: size-independent properties.
    (1) decoding is per-frame independent: any sub-batch / permutation gives the same rows;
    (2) high-SNR frames decode to the transmitted word (encode -> channel -> decode round trip);
    (3) SCL with L=1 equals SC wherever no LLR is exactly zero-tied (here: identical decisions on clean frames)."""
    kw, x, truth = common.make_case("SCLLUTDecoder", N=1024, K=512, L=8, B=20000, seed=123, tables="minsum", ebn0_db=3.5)
    dec = q.SCLLUTDecoder(**kw)
    xb = x.astype(np.uint8)
    y = dec.decode(xb)
    assert y.shape == (20000, 512)
    perm = np.random.default_rng(1).permutation(20000)
    assert (dec.decode(xb[perm]) == y[perm]).all()
    assert (dec.decode(xb[:777]) == y[:777]).all()
    bler = (y != truth).any(axis=1).mean()
    assert bler < 0.05, bler
    sub = np.arange(0, 20000, 400)
    want = po.OracleDecoder("SCLLUTDecoder", **kw).decode(x[sub])
    assert (y[sub] == want).all()


def test_routing_note_says_why_a_lut_decoder_left_the_nibble_kernel(q, capfd):
    """VERDICT r1 item 10: falling off scl_lut_warp costs 3-100x and used to be silent."""
    kw, x, _ = common.make_case("SCLLUTDecoder", N=128, K=64, L=8, B=32, seed=3)
    dec = q.SCLLUTDecoder(**kw)
    assert dec.kernel == "scl_lut_warp" and dec.kernel_note == ""
    kw16, x16, _ = common.make_case("SCLLUTDecoder", N=128, K=64, L=16, B=32, seed=3)
    capfd.readouterr()
    dec16 = q.SCLLUTDecoder(**kw16)
    assert dec16.kernel != "scl_lut_warp" and "list size" in dec16.kernel_note
    assert "list size" in capfd.readouterr().err or True      # (printed once per process and reason; an earlier test may have had it)
    assert (dec16.decode(x16) == po.OracleDecoder("SCLLUTDecoder", **kw16).decode(x16)).all()
    kwf, xf, _ = common.make_case("SCLDecoder", N=128, K=64, L=8, B=8, seed=3, tables="channel")
    assert q.SCLDecoder(**kwf).kernel_note == ""               # not a LUT class: nothing to note


@pytest.mark.parametrize("kind,force", [("SCLLUTDecoder", 0), ("SCLDecoder", 0), ("SCLLUTDecoder", 1), ("SCLDecoder", 1)])
def test_large_decoder_survives_a_smaller_one_created_later(monkeypatch, kind, force):
    """cudaFuncAttributeMaxDynamicSharedMemorySize is per kernel function, shared by every decoder of the family (ADVICE r1):
    an N=128 decoder created after an N=1024 one must not shrink the cap under the live larger decoder."""
    import quantized_decoder_polar_codes_b200 as q
    if force:
        monkeypatch.setenv("POLAR_B200_FORCE_GENERIC", "1")
    tab = dict(tables="minsum") if "LUT" in kind else dict(tables="channel")
    kw_big, x_big, _ = common.make_case(kind, N=1024, K=512, L=4, B=16, seed=5, **tab)
    kw_small, x_small, _ = common.make_case(kind, N=128, K=64, L=4, B=16, seed=6, **tab)
    big = getattr(q, kind)(**kw_big)
    first = big.decode(x_big)
    small = getattr(q, kind)(**kw_small)
    small.decode(x_small)
    again = big.decode(x_big)          # used to fail with "invalid argument" once the cap had shrunk
    assert (first == again).all()
    assert (first == po.OracleDecoder(kind, **kw_big).decode(x_big)).all()


@pytest.mark.parametrize("kind,N,K,L,B", [("SCLUTDecoder", 256, 128, 1, 1 << 19), ("SCLUTDecoder", 1024, 512, 1, 113664 + 32),
                                           ("FastSCLUTDecoder", 1024, 512, 1, 1 << 17), ("SCLLUTDecoder", 512, 256, 4, 1 << 17)])
def test_full_residency_batches(q, kind, N, K, L, B):
    """Batches that fill every SM with its full complement of CTAs (and a few passes more): resident CTAs at the
    occupancy limit, warps taking several frame groups each, and the decoded copies of the same frames agreeing from the
    first pass to the last -- shapes that no small-batch test reaches."""
    import torch
    from quantized_decoder_polar_codes_b200 import capi
    kw, x, _ = common.make_case(kind, N=N, K=K, L=L, B=2048, seed=9, tables="minsum", ebn0_db=3.0)
    want = po.OracleDecoder(kind, **kw).decode(x[:256].astype(np.int32))
    reps = -(-B // 2048)
    xs = np.tile(x.astype(np.uint8), (reps, 1))[:B]
    dec = getattr(q, kind)(**kw)
    d_in = torch.from_numpy(xs).cuda()
    d_out = torch.empty((B, want.shape[1]), dtype=torch.uint8, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    for _ in range(2):
        capi.decode_device(dec, d_in.data_ptr(), capi.PD_U8, B, d_out.data_ptr(), s)
    capi.sync_check(dec, s)
    got = d_out.cpu().numpy()
    assert (got[:256] == want).all()
    last = (B // 2048 - 1) * 2048                      # the last full copy of the 2048 unique frames
    assert (got[last:last + 256] == want).all()
    assert (got[:2048] == got[last:last + 2048]).all()


@pytest.mark.parametrize("dtype", ["int32", "uint8", "float64", "int64"])
def test_host_call_staging_paths(q, monkeypatch, dtype):
    """decode((B,N)) from pageable numpy memory in the dtypes the drivers use: int32 symbols are narrowed to bytes on the host
    (thread pool -> pinned staging -> H2D), results come back in a pinned array; many small chunks to turn the pipeline over."""
    monkeypatch.setenv("POLAR_B200_CHUNK_FRAMES", "3000")
    kw, x, _ = common.make_case("SCLLUTDecoder", N=256, K=128, L=4, B=20000, seed=12)
    dec = q.SCLLUTDecoder(**kw)
    got = dec.decode(x.astype(dtype))
    want = po.OracleDecoder("SCLLUTDecoder", **kw).decode(x.astype(np.int32))
    assert got.shape == want.shape and (got == want).all()
    bad = x.astype(np.int32).copy()
    bad[12345 % bad.shape[0], 7] = 300                  # does not fit a byte: must be reported, not truncated to 44
    with pytest.raises(ValueError):
        dec.decode(bad)
    assert (dec.decode(x.astype(dtype)) == want).all()  # and the decoder stays usable
    if dtype == "float64":                               # float64-typed symbols are truncated on the host like the reference's cast
        assert (dec.decode(x[:3].astype(np.float64)) == want[:3]).all()       # tiny call: mapped staging area
        assert (dec.decode(x.astype(np.float64) + 0.75) == want).all()
        badf = x.astype(np.float64)
        badf[5, 9] = np.nan
        with pytest.raises(ValueError):
            dec.decode(badf)
        badf[5, 9] = -2.0
        with pytest.raises(ValueError):
            dec.decode(badf[4:8])


def test_set_devices_shards_one_call(q, monkeypatch):
    """pd_set_devices: one decode() call dealt to several pipelines (here: three on the one visible GPU; the same code path
    deals to several GPUs) returns what a single device returns; [] restores the single-device path."""
    import torch
    monkeypatch.setenv("POLAR_B200_CHUNK_FRAMES", "2500")
    kw, x, _ = common.make_case("CASCLLUTDecoder", N=256, K=152, A=128, L=8, B=16000, seed=13)
    dec = q.CASCLLUTDecoder(**kw)
    want = dec.decode(x)
    ids = [0, 0, 0] if torch.cuda.device_count() < 2 else [0, 1, 0, 1]
    dec.set_devices(ids)
    assert dec.device_count == len(ids)
    assert (dec.decode(x) == want).all()
    dec.set_devices([])
    assert dec.device_count == 1 and (dec.decode(x) == want).all()
    assert (want[:64] == po.OracleDecoder("CASCLLUTDecoder", **kw).decode(x[:64])).all()
