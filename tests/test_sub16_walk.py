"""The op list scl_lut_warp compiles for a decoder, read through the host emulator (tools/emu, like
test_emulated_kernels.py): a plain walk decodes every depth top-1 node with its two 8-leaf subtrees as ONE op (SUB16),
so no upper f / g / combine op is left at that depth; a Fast-SSC walk keeps the separate SUB8 subtrees."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tools", "emu")

FOP_UF, FOP_UG, FOP_UC, FOP_SUB8, FOP_SUB16 = 0, 1, 2, 3, 14

# decoders built inside a child process: the emulated pybind module must not meet the real package's types
_PROBE = r"""
import ctypes, json, os, sys
sys.path.insert(0, os.path.join(%(root)r, "tools", "emu"))
import check, common
emu = check.load_emu()
lib = ctypes.CDLL(os.path.join(%(root)r, "tools", "emu", "build", "libpolar_b200.so"))
out = {}
for name, kind, kw in %(cases)r:
    k, _, _ = common.make_case(kind, seed=77, **kw)
    d = getattr(emu, kind)(**k)
    hist = (ctypes.c_int * (16 * 32))()
    n_ops, n_chunks = ctypes.c_int(), ctypes.c_int()
    rc = lib.pb_emu_fast_plan(ctypes.c_void_p(d._handle), hist, ctypes.byref(n_ops), ctypes.byref(n_chunks))
    out[name] = dict(rc=rc, N=kw["N"], hist=[list(hist[t * 32:(t + 1) * 32]) for t in range(16)], n_ops=n_ops.value, n_chunks=n_chunks.value)
print(json.dumps(out))
"""

CASES = [
    ("ns", "SCLLUTDecoder", dict(N=1024, K=512, L=8, B=2)),
    ("sc_32", "SCLUTDecoder", dict(N=32, K=16, B=2)),
    ("cafast", "CAFastSCLLUTDecoder", dict(N=1024, K=536, A=512, L=8, B=2)),
]


@pytest.fixture(scope="module")
def plans():
    r = subprocess.run(["bash", os.path.join(EMU, "build.sh")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    r = subprocess.run([sys.executable, "-c", _PROBE % dict(root=ROOT, cases=CASES)], capture_output=True, text=True,
                       timeout=600, cwd=EMU)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    for name, p in out.items():
        assert p["rc"] == 0, name + " is not on scl_lut_warp"
    return out


def _top(p):
    return p["N"].bit_length() - 1 - 3   # depth of the 8-leaf subtree roots, n - 3


@pytest.mark.parametrize("name", ["ns", "sc_32"])
def test_plain_walk_has_no_upper_op_at_depth_top_minus_1(plans, name):
    p = plans[name]
    t = _top(p)
    for ty in (FOP_UF, FOP_UG, FOP_UC):
        assert p["hist"][ty][t - 1] == 0
    assert sum(p["hist"][FOP_SUB8]) == 0
    assert p["hist"][FOP_SUB16][t - 1] == 1 << (t - 1) and sum(p["hist"][FOP_SUB16]) == 1 << (t - 1)


def test_north_star_plan_size(plans):
    p = plans["ns"]
    # before SUB16 the walk had 127 UF + 127 UG + 127 UC + 128 SUB8 = 509 ops in 1180 chunks
    assert p["n_ops"] == 253
    assert p["n_chunks"] <= 1180


def test_fast_ssc_walk_keeps_sub8(plans):
    p = plans["cafast"]
    assert sum(p["hist"][FOP_SUB8]) > 0
    assert sum(p["hist"][FOP_SUB16]) == 0
