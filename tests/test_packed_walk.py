"""What plan_fast_lut hands the plain scl_lut_warp kernels, read through the host emulator (tools/emu, like
test_sub16_walk.py):
  * the table stream is followed by copies of its first kRingChunks - 1 chunks, so that the plain kernels' prefetch runs
    through the end of a pass without a wrap test;
  * every upper f / g / combine entry of a plain walk carries the constants the kernel used to derive from the depth and
    the node: level offsets and memory spaces, the node's first leaf, the leftmost-chain and re-point flags."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tools", "emu")

FOP_UF, FOP_UG, FOP_UC, FOP_SUB16 = 0, 1, 2, 14
K_RING_CHUNKS = 4
OFF_MASK, IN_WS, LEFTMOST, OWN_LEFT, LEAF_SHIFT = 0x7FFF, 0x8000, 0x10000, 0x10000, 17
K_MAX_LOG = 12

_PROBE = r"""
import ctypes, json, os, sys
sys.path.insert(0, os.path.join(%(root)r, "tools", "emu"))
import check, common
emu = check.load_emu()
lib = ctypes.CDLL(os.path.join(%(root)r, "tools", "emu", "build", "libpolar_b200.so"))
out = {}
for name, kind, kw in %(cases)r:
    k, _, _ = common.make_case(kind, seed=5, **kw)
    d = getattr(emu, kind)(**k)
    ops = (ctypes.c_uint32 * (2 * 4096))()
    voff = (ctypes.c_int * (%(kmaxlog)d + 2))()
    gl = ctypes.c_int()
    cap = 1 << 21
    stream = (ctypes.c_uint32 * cap)()
    words = ctypes.c_longlong()
    n_ops, n_chunks = ctypes.c_int(), ctypes.c_int()
    hist = (ctypes.c_int * (16 * 32))()
    rc = lib.pb_emu_fast_plan(ctypes.c_void_p(d._handle), hist, ctypes.byref(n_ops), ctypes.byref(n_chunks))
    nops = lib.pb_emu_fast_plan_detail(ctypes.c_void_p(d._handle), ops, 4096, voff, ctypes.byref(gl), stream,
                                       ctypes.c_longlong(cap), ctypes.byref(words))
    w = min(words.value, cap)
    out[name] = dict(rc=rc, N=kw["N"], n_ops=nops, n_chunks=n_chunks.value, ops=list(ops[:2 * max(nops, 0)]),
                     voff=list(voff), gl=gl.value, words=words.value, head=list(stream[:128 * (%(ring)d - 1)]),
                     tail=list(stream[w - 128 * (%(ring)d - 1):w]), first_line=[stream[4 * l] for l in range(32)])
print(json.dumps(out))
"""

CASES = [("n%d_l%d" % (1 << n, L), "SCLUTDecoder" if L == 1 else "SCLLUTDecoder", dict(N=1 << n, K=1 << (n - 1), L=L, B=1))
         for n in range(5, 13) for L in (1, 2, 4, 8)]


@pytest.fixture(scope="module")
def plans():
    r = subprocess.run(["bash", os.path.join(EMU, "build.sh")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    r = subprocess.run([sys.executable, "-c", _PROBE % dict(root=ROOT, cases=CASES, kmaxlog=K_MAX_LOG, ring=K_RING_CHUNKS)],
                       capture_output=True, text=True, timeout=900, cwd=EMU)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    out = json.loads(r.stdout.strip().splitlines()[-1])
    for name, p in out.items():
        assert p["rc"] == 0 and p["n_ops"] > 0, name + " is not on scl_lut_warp"
    return out


def _plain_walk(N):
    """(type, depth, node) of a plain walk in order: the recursion of plan_fast_lut without special nodes."""
    top = N.bit_length() - 1 - 3
    ops = []

    def walk(depth, node):
        if depth == top - 1:
            ops.append((FOP_SUB16, depth, node))
            return
        ops.append((FOP_UF, depth, node))
        walk(depth + 1, 2 * node)
        ops.append((FOP_UG, depth, node))
        walk(depth + 1, 2 * node + 1)
        ops.append((FOP_UC, depth, node))

    walk(0, 0)
    return ops


@pytest.mark.parametrize("name", [c[0] for c in CASES])
def test_stream_head_is_copied_after_its_end(plans, name):
    p = plans[name]
    assert p["words"] == (p["n_chunks"] + K_RING_CHUNKS - 1) * 128
    assert p["tail"] == p["head"]


@pytest.mark.parametrize("name", [c[0] for c in CASES])
def test_upper_op_entries_carry_their_operands(plans, name):
    p = plans[name]
    N, voff, gl = p["N"], p["voff"], p["gl"]
    want = _plain_walk(N)
    assert p["n_ops"] == len(want)
    for i, (ty, dd, node) in enumerate(want):
        x, y = p["ops"][2 * i], p["ops"][2 * i + 1]
        assert x & 0xFF == ty and (x >> 8) & 0xFF == dd, (i, hex(x))
        leaf0 = 2 * node * (N >> (dd + 1))
        if ty == FOP_SUB16:
            assert y == node
        elif ty == FOP_UC:
            assert y == (OWN_LEFT if dd >= 1 and node % 2 == 0 else 0) | (leaf0 << LEAF_SHIFT), (i, hex(y))
        else:
            hi = x >> 16
            assert hi & OFF_MASK == voff[dd] * 32 and bool(hi & IN_WS) == (dd <= gl), (i, hex(x))
            assert y & OFF_MASK == voff[dd + 1] * 32 and bool(y & IN_WS) == (dd + 1 <= gl), (i, hex(y))
            assert bool(y & LEFTMOST) == (ty == FOP_UF and node == 0), (i, hex(y))
            assert y >> LEAF_SHIFT == leaf0, (i, hex(y))
    # the stream's first line is the first op line: the same entries the kernel reads
    n16 = min(16, len(want))
    assert p["first_line"][:2 * n16] == p["ops"][:2 * n16]
