"""List sizes 64, 128 and 256 (the path_cta kernel) without a GPU: which list sizes the constructors accept, and the kernel
source under the host emulator (tools/emu) against the oracle.  The GPU parity proof is tests/test_gpu_large_lists.py."""
import os
import subprocess
import sys

import pytest

import common

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tools", "emu")


def _kw(kind, N, K, L, **extra):
    kw, _, _ = common.make_case(kind, N, K, L=L, B=1, **extra)
    return kw


@pytest.mark.parametrize("kind,N,K,L", [
    ("SCLDecoder", 64, 32, 48),                  # not a power of two
    ("SCLLUTDecoder", 64, 32, 512),              # above 256
    ("SCLDecoder", 16, 8, 64),                   # N < 32: partial sums are 32-bit words per path
    ("CASCLLUTDecoder", 128, 88, 96),
    ("SCLUniformQuantizedDecoder", 64, 32, 33),
    ("FastSCLDecoder", 64, 32, 0),
])
def test_unsupported_list_sizes_raise_value_error(kind, N, K, L):
    import quantized_decoder_polar_codes_b200 as q
    with pytest.raises(ValueError, match="L="):
        getattr(q, kind)(**_kw(kind, N, K, L))


def test_blind_detection_cascl_keeps_l_at_most_32():
    import quantized_decoder_polar_codes_b200 as q
    fm, mm = common.sim.frozen_mask(64, 40)
    with pytest.raises(ValueError, match="L="):
        q.BDCASCLDecoder(N=64, K=40, A=16, L=64, frozen_bits=fm, message_bits=mm, crc_n=24, crc_p=list(common.sim.CRC24_LOC))


@pytest.mark.parametrize("L", [64, 128, 256])
@pytest.mark.parametrize("kind", sorted(common.LIST_KINDS))
def test_large_list_sizes_pass_validation(kind, L):
    """Accepted list sizes get past every argument check: without a GPU the constructor then fails on the device probe
    (PD_ECUDA), not with ValueError; with one it builds a path_cta decoder."""
    import quantized_decoder_polar_codes_b200 as q
    K = 40 if kind in common.CA_KINDS else 16
    kw = _kw(kind, 64, K, L, **({"A": 16} if kind in common.CA_KINDS else {}))
    try:
        dec = getattr(q, kind)(**kw)
    except ValueError as e:
        pytest.fail(f"L={L} rejected: {e}")
    except RuntimeError as e:
        assert "no CUDA device" in str(e)
    else:
        assert dec.kernel == "path_cta"


@pytest.fixture(scope="module")
def emu_built():
    r = subprocess.run(["bash", os.path.join(EMU, "build.sh")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def test_path_cta_matches_the_oracle_under_the_emulator(emu_built):
    """SCL-LUT, CA-SCL-LUT, Fast-SCL-LUT, CA-Fast-SCL-LUT, float SCL / Fast-SCL / CA-SCL, uniform and Lloyd SCL at
    N in {32, 64, 128} and L in {64, 128, 256}, tie-heavy random tables and channel frames (tools/emu/check.py CTA_CASES)."""
    r = subprocess.run([sys.executable, os.path.join(EMU, "check.py"), "path_cta"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout[-3000:] + r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if "kernel=" in ln]
    assert len(lines) >= 15 and all("kernel=path_cta" in ln and "mismatching=   0" in ln for ln in lines)
