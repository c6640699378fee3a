#!/usr/bin/env python
"""Bit-exactness of the decode kernels under the host emulator (tools/emu/build) against the CPU oracle.
Development tooling: lets kernel changes be checked on the GPU-less build box.  Usage: check.py [case-filter]
(a filter starting with "path_cta" selects the path_cta cases, which the default run leaves out)"""
import importlib.util
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
# the package's __init__ loads the real (CUDA) extension, whose pybind types would clash with the emulated module's:
# register a bare package so that only the pure-numpy helper `simulation` is imported from it
import types  # noqa: E402
_pkg = types.ModuleType("quantized_decoder_polar_codes_b200")
_pkg.__path__ = [os.path.join(ROOT, "quantized_decoder_polar_codes_b200")]
sys.modules["quantized_decoder_polar_codes_b200"] = _pkg
import common  # noqa: E402
from oracle import polar_oracle as po  # noqa: E402


def load_emu():
    import sysconfig
    path = os.path.join(HERE, "build", "_libPolarDecoder" + sysconfig.get_config_var("EXT_SUFFIX"))
    spec = importlib.util.spec_from_file_location("_libPolarDecoder", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


CASES = [
    ("ns_small", "SCLLUTDecoder", dict(N=128, K=64, L=8, B=24)),
    ("ns_1024", "SCLLUTDecoder", dict(N=1024, K=512, L=8, B=20, tables="minsum", ebn0_db=2.0)),
    ("ns_1024_rand", "SCLLUTDecoder", dict(N=1024, K=512, L=8, B=12)),
    ("sclut_256", "SCLUTDecoder", dict(N=256, K=100, B=70)),
    ("scl_l4", "SCLLUTDecoder", dict(N=256, K=128, L=4, B=40)),
    ("scl_l2", "SCLLUTDecoder", dict(N=64, K=30, L=2, B=40)),
    ("ca_512", "CASCLLUTDecoder", dict(N=512, K=280, A=256, L=8, B=16)),
    ("fastsclut", "FastSCLUTDecoder", dict(N=512, K=256, B=70)),
    ("fastscl", "FastSCLLUTDecoder", dict(N=512, K=256, L=8, B=16)),
    ("cafast", "CAFastSCLLUTDecoder", dict(N=1024, K=536, A=512, L=8, B=8)),
    ("cafast_q", "CAFastSCLLUTDecoder", dict(N=256, K=152, A=128, L=4, B=24, Q=12, Qc=9)),
    ("multi_pass", "SCLLUTDecoder", dict(N=128, K=64, L=8, B=1001)),
    ("staged_io", "SCLLUTDecoder", dict(N=128, K=64, L=4, B=9000)),
    ("staged_f64sym", "SCLLUTDecoder", dict(N=128, K=64, L=4, B=5000, xdtype="float64")),
    ("multidev", "SCLLUTDecoder", dict(N=128, K=64, L=4, B=9000)),
    ("multidev_f64", "SCLDecoder", dict(N=128, K=64, L=4, B=3000, tables="channel")),
    ("multi_pass_l1", "SCLUTDecoder", dict(N=64, K=30, B=3000)),
    ("sclut_1024", "SCLUTDecoder", dict(N=1024, K=512, B=200, tables="minsum")),
    ("cascl_1024", "CASCLLUTDecoder", dict(N=1024, K=536, A=512, L=8, B=16, tables="minsum")),
    ("cafast_1024m", "CAFastSCLLUTDecoder", dict(N=1024, K=536, A=512, L=8, B=16, tables="minsum")),
    ("fastsc_1024", "FastSCLUTDecoder", dict(N=1024, K=512, B=100, tables="minsum")),
    ("float_scl", "SCLDecoder", dict(N=128, K=64, L=8, B=16, tables="channel")),
    ("uniform_l32", "SCLUniformQuantizedDecoder", dict(N=128, K=64, L=32, B=8)),
    # N=32: the depth top-1 node of SUB16 is at depth 1, right below the root
    ("sclut_32", "SCLUTDecoder", dict(N=32, K=16, B=200)),
    ("scl_32", "SCLLUTDecoder", dict(N=32, K=16, L=8, B=40)),
]

# path_cta (L = 64, 128, 256): one fiber per path makes these slow under the emulator, so they run only when asked for
# (`check.py path_cta`, or a filter starting with it), never in the default run.
CTA_CASES = [
    ("path_cta_sclut_32", "SCLLUTDecoder", dict(N=32, K=16, L=64, B=48)),
    ("path_cta_sclut_32_dead", "SCLLUTDecoder", dict(N=32, K=5, L=64, B=48)),      # L > 2^K: dead-path ties to the end
    ("path_cta_sclut_64", "SCLLUTDecoder", dict(N=64, K=32, L=256, B=24)),
    ("path_cta_sclut_128m", "SCLLUTDecoder", dict(N=128, K=64, L=64, B=4, tables="minsum", ebn0_db=1.0)),
    ("path_cta_ca_128", "CASCLLUTDecoder", dict(N=128, K=88, A=64, L=64, B=32)),
    ("path_cta_ca_64", "CASCLLUTDecoder", dict(N=64, K=40, A=16, L=256, B=16)),
    ("path_cta_fast_64", "FastSCLLUTDecoder", dict(N=64, K=30, L=64, B=32)),
    ("path_cta_fast_128", "FastSCLLUTDecoder", dict(N=128, K=64, L=256, B=16)),
    ("path_cta_float_32", "SCLDecoder", dict(N=32, K=16, L=256, B=3, tables="channel")),
    ("path_cta_float_128", "SCLDecoder", dict(N=128, K=64, L=64, B=4, tables="channel")),
    ("path_cta_float_rand", "SCLDecoder", dict(N=64, K=32, L=64, B=32)),
    ("path_cta_uniform_64", "SCLUniformQuantizedDecoder", dict(N=64, K=32, L=64, B=32)),
    ("path_cta_lloyd_64", "SCLLloydQuantizedDecoder", dict(N=64, K=32, L=128, B=16)),
    ("path_cta_fastf_64", "FastSCLDecoder", dict(N=64, K=30, L=128, B=16)),
    ("path_cta_cafast_64", "CAFastSCLLUTDecoder", dict(N=64, K=54, A=30, L=64, B=16)),
    ("path_cta_cascl_64", "CASCLDecoder", dict(N=64, K=40, A=16, L=128, B=16, tables="channel")),
    ("path_cta_uniform_128", "SCLUniformQuantizedDecoder", dict(N=128, K=64, L=256, B=16)),
]


def main():
    flt = sys.argv[1] if len(sys.argv) > 1 else ""
    emu = load_emu()
    bad_total = 0
    for name, kind, ckw in (CTA_CASES if flt.startswith("path_cta") else CASES):
        if flt and flt not in name:
            continue
        ckw = dict(ckw)
        xdtype = ckw.pop("xdtype", None)
        kw, x, _ = common.make_case(kind, seed=77, **ckw)
        t0 = time.time()
        dec = getattr(emu, kind)(**kw)
        if name.startswith("multidev"):
            dec.set_devices([0, 0, 0])
        got = dec.decode(x if xdtype is None else x.astype(xdtype) + 0.5)   # (float64-typed symbols are truncated)
        t1 = time.time()
        want = po.OracleDecoder(kind, **kw).decode(x)
        bad = int((got != want).any(axis=1).sum())
        bad_total += bad
        print(f"{name:14s} {kind:26s} kernel={dec.kernel:13s} frames={x.shape[0]:4d} mismatching={bad:4d}  emu {t1 - t0:6.1f} s", flush=True)
    print("OK" if bad_total == 0 else f"FAILED: {bad_total} mismatching frames")
    return 1 if bad_total else 0


if __name__ == "__main__":
    sys.exit(main())
