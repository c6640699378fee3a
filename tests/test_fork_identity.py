"""The identity exit of the scl_lut_warp fork (pb_scl_lut.cuh): when the keeps are sorted and every flip key is >= the
largest keep on all lanes of the warp, the fork returns at once and the paths stay where they are.  Checked through the
host emulator (tools/emu) against the oracle:
  * bits, debug path metrics and winners equal the oracle's, on AWGN channel inputs and on tie-heavy tables (LLR rows
    of 0.0 / -0.0 / +-1, so that flip keys equal to the largest keep occur);
  * the number of exits the kernel takes is the number of (warp, leaf) forks at which the oracle finds every frame of
    the warp unchanged and the kernel knows the keeps are sorted (tools/fork_stats.py), and it is > 0 on channel inputs;
  * POLAR_B200_KDEBUG=2 turns the exit off: no exit, the same outputs."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tools", "emu")
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import common  # noqa: E402

TIES = (-1.0, -0.0, 0.0, 1.0)


def _case(kind, N, L, inputs):
    K = N // 2
    ckw = dict(N=N, K=K, L=L, B=2 * (32 // L) + 1, seed=N + L)   # two full warps and one frame of a third
    if kind == "CASCLLUTDecoder":
        ckw["A"] = K - 24
    if inputs == "awgn":
        ckw.update(tables="minsum", ebn0_db=2.0)
    else:
        ckw.update(alphabet=TIES)
    return ckw


CASES = [("%s_n%d_l%d_%s" % (kind[:-10], N, L, inputs), kind, _case(kind, N, L, inputs))
         for kind in ("SCLLUTDecoder", "CASCLLUTDecoder") for N in (128, 256, 1024) for L in (2, 4, 8)
         for inputs in ("awgn", "ties")]

_PROBE = r"""
import ctypes, os, sys
import numpy as np
sys.path.insert(0, os.path.join(%(root)r, "tools", "emu"))
import check, common
emu = check.load_emu()
lib = ctypes.CDLL(os.path.join(%(root)r, "tools", "emu", "build", "libpolar_b200.so"))
seen, taken = ctypes.c_ulonglong(), ctypes.c_ulonglong()
res = {}
for name, kind, ckw in %(cases)r:
    kw, x, _ = common.make_case(kind, **ckw)
    d = getattr(emu, kind)(**kw)
    assert d.kernel == "scl_lut_warp", (name, d.kernel)
    pm = np.zeros((x.shape[0], kw["L"]), np.float64)
    win = np.zeros(x.shape[0], np.int32)
    assert lib.pd_set_debug_outputs(ctypes.c_void_p(d._handle), ctypes.c_void_p(pm.ctypes.data), ctypes.c_void_p(win.ctypes.data)) == 0
    lib.pb_emu_fork_counts(ctypes.byref(seen), ctypes.byref(taken), 1)
    bits = d.decode(x)
    lib.pb_emu_fork_counts(ctypes.byref(seen), ctypes.byref(taken), 1)
    lib.pd_set_debug_outputs(ctypes.c_void_p(d._handle), None, None)
    res[name + "/bits"], res[name + "/pm"], res[name + "/win"] = bits, pm, win
    res[name + "/counts"] = np.array([seen.value, taken.value], np.int64)
np.savez(sys.argv[1], **res)
"""


def _fork_stats():
    spec = importlib.util.spec_from_file_location("_fork_stats", os.path.join(ROOT, "tools", "fork_stats.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    r = subprocess.run(["bash", os.path.join(EMU, "build.sh")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    out = {}
    for dbg in ("0", "2"):
        path = str(tmp_path_factory.mktemp("fork") / ("kdebug%s.npz" % dbg))
        env = dict(os.environ, POLAR_B200_KDEBUG=dbg)
        r = subprocess.run([sys.executable, "-c", _PROBE % dict(root=ROOT, cases=CASES), path],
                           capture_output=True, text=True, timeout=1800, cwd=EMU, env=env)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        out[dbg] = dict(np.load(path))
    return out


@pytest.fixture(scope="module")
def oracle():
    return _fork_stats()


@pytest.mark.parametrize("name,kind,ckw", CASES, ids=[c[0] for c in CASES])
def test_identity_exit_matches_the_oracle(runs, oracle, name, kind, ckw):
    kw, x, _ = common.make_case(kind, **ckw)
    want, pm_want, win_want = oracle.hooked_oracle().OracleDecoder(kind, **kw).decode(x, return_pm=True)
    bits, classes = oracle.fork_classes(kind, kw, x)
    assert np.array_equal(bits, want)
    expect = oracle.warp_identity(classes, kw["frozen_bits"], kw["L"])
    n_warps = -(-x.shape[0] // (32 // kw["L"]))
    n_info = int((np.asarray(kw["frozen_bits"]) == 0).sum())
    for dbg in ("0", "2"):
        r = runs[dbg]
        assert np.array_equal(r[name + "/bits"], want), dbg
        assert np.array_equal(r[name + "/pm"], pm_want), dbg
        assert np.array_equal(r[name + "/win"], win_want), dbg
        seen, taken = (int(v) for v in r[name + "/counts"])
        assert seen == n_warps * n_info, dbg
        assert taken == (expect if dbg == "0" else 0), (dbg, taken, expect)
    if name.endswith("awgn"):
        assert expect > 0
