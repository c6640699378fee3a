"""All-frozen 8-leaf subtrees in the plain scl_lut_warp walks (pb_scl_lut.cuh), through the host emulator (tools/emu):
  * plan: arg bit h of every SUB16 entry says whether the 8 leaves of its half h are all frozen, and the stream has the
    length that follows from those marks (an all-frozen half takes 22 lines at L > 1 and none at L = 1, instead of 32);
  * decoding: such halves run a feed-forward step (L > 1) or nothing at all (L = 1).  Bits, debug path metrics and
    winners equal the oracle's bit for bit -- the metrics pin the order of the fp64 sums -- and the number of identity
    exits of the fork is still the one tools/fork_stats.py predicts.
Frozen sets: simulation.frozen_mask (the NR sequence; PW above N = 1024) at K/N = 1/8, 1/4, 1/2 and 3/4, where the
rate-0 subtrees vary most."""
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

FOP_UF, FOP_UG, FOP_UC, FOP_SUB16 = 0, 1, 2, 14
RATES = ((1, 8), (1, 4), (1, 2), (3, 4))
TIES = (-1.0, -0.0, 0.0, 1.0)


def _kind(L):
    return "SCLUTDecoder" if L == 1 else "SCLLUTDecoder"


PLAN_CASES = [("n%d_l%d_k%d" % (1 << n, L, (1 << n) * a // b), _kind(L), dict(N=1 << n, K=(1 << n) * a // b, L=L, B=1))
              for n in range(5, 13) for L in (1, 2, 4, 8) for a, b in RATES]

_PLAN_PROBE = r"""
import ctypes, json, os, sys
sys.path.insert(0, os.path.join(%(root)r, "tools", "emu"))
import check, common
emu = check.load_emu()
lib = ctypes.CDLL(os.path.join(%(root)r, "tools", "emu", "build", "libpolar_b200.so"))
out = {}
for name, kind, kw in %(cases)r:
    k, _, _ = common.make_case(kind, seed=3, **kw)
    d = getattr(emu, kind)(**k)
    ops = (ctypes.c_uint32 * (2 * 4096))()
    voff = (ctypes.c_int * 16)()
    gl, words = ctypes.c_int(), ctypes.c_longlong()
    stream = (ctypes.c_uint32 * 1)()
    hist = (ctypes.c_int * (16 * 32))()
    n_ops, n_chunks = ctypes.c_int(), ctypes.c_int()
    rc = lib.pb_emu_fast_plan(ctypes.c_void_p(d._handle), hist, ctypes.byref(n_ops), ctypes.byref(n_chunks))
    nops = lib.pb_emu_fast_plan_detail(ctypes.c_void_p(d._handle), ops, 4096, voff, ctypes.byref(gl), stream,
                                       ctypes.c_longlong(0), ctypes.byref(words))
    out[name] = dict(rc=rc, n_ops=nops, n_chunks=n_chunks.value, ops=list(ops[:2 * max(nops, 0)]))
print(json.dumps(out))
"""


def _build_emu():
    r = subprocess.run(["bash", os.path.join(EMU, "build.sh")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def _rate0_halves(frozen):
    """-> bool per 8-leaf subtree: all of its leaves frozen"""
    return (np.asarray(frozen).reshape(-1, 8) == 1).all(axis=1)


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


def _predicted_chunks(N, L, frozen):
    """The stream's length in chunks of 4 lines: an op line per 16 ops, f for UF, g0 g1 for UG; per SUB16 half h the
    node's 1 + h lines at the end of a chunk, then 32 lines, or 22 for an all-frozen half at L > 1 (none at all, the
    node's lines included, at L = 1); the whole padded to kRingChunks = 4 chunks."""
    r0 = _rate0_halves(frozen)
    lines = 0
    for i, (ty, _, node) in enumerate(_plain_walk(N)):
        lines += (i % 16 == 0) + {FOP_UF: 1, FOP_UG: 2, FOP_UC: 0}.get(ty, 0)
        if ty != FOP_SUB16:
            continue
        for h in (0, 1):
            z = bool(r0[2 * node + h])
            if L == 1 and z:
                continue
            lines += (3 - h - lines) % 4 + 1 + h + (22 if z else 32)
    lines += -lines % 16
    return lines // 4


@pytest.fixture(scope="module")
def plans():
    _build_emu()
    r = subprocess.run([sys.executable, "-c", _PLAN_PROBE % dict(root=ROOT, cases=PLAN_CASES)],
                       capture_output=True, text=True, timeout=1800, cwd=EMU)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("name,kind,ckw", PLAN_CASES, ids=[c[0] for c in PLAN_CASES])
def test_sub16_marks_and_stream_length(plans, name, kind, ckw):
    p = plans[name]
    assert p["rc"] == 0 and p["n_ops"] > 0, name + " is not on scl_lut_warp"
    N, L = ckw["N"], ckw["L"]
    frozen = common.make_case(kind, seed=3, **ckw)[0]["frozen_bits"]
    r0 = _rate0_halves(frozen)
    want = _plain_walk(N)
    assert p["n_ops"] == len(want)
    for i, (ty, dd, node) in enumerate(want):
        x = p["ops"][2 * i]
        assert x & 0xFFFF == ty | dd << 8, (i, hex(x))
        if ty == FOP_SUB16:
            assert x >> 16 == int(r0[2 * node]) | int(r0[2 * node + 1]) << 1, (i, hex(x))
    assert p["n_chunks"] == _predicted_chunks(N, L, frozen)


def _decode_case(kind, N, L, a, b, inputs):
    K = N * a // b
    ckw = dict(N=N, K=K, B=(2 * (32 // L) + 1) if L > 1 else 40, seed=N + L + K)
    if L > 1:
        ckw["L"] = L
    if kind == "CASCLLUTDecoder":
        ckw["A"] = K - 24
    if inputs == "awgn":
        ckw.update(tables="minsum", ebn0_db=2.0)
    else:
        ckw.update(alphabet=TIES)
    return ckw


# CA-SCL only where the 24-bit CRC leaves at least 8 message bits
DECODE_CASES = [("%s_n%d_l%d_k%d_%s" % (kind[:-10], N, L, N * a // b, inputs), kind, _decode_case(kind, N, L, a, b, inputs))
                for kind, Ls in (("SCLUTDecoder", (1,)), ("SCLLUTDecoder", (2, 4, 8)), ("CASCLLUTDecoder", (2, 4, 8)))
                for L in Ls for N in (32, 64, 128, 256, 512, 1024) for a, b in RATES for inputs in ("awgn", "ties")
                if kind != "CASCLLUTDecoder" or N * a // b >= 32]

_DECODE_PROBE = r"""
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
    L = kw.get("L", 1)
    pm = np.zeros((x.shape[0], L), np.float64)
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


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    _build_emu()
    path = str(tmp_path_factory.mktemp("rate0") / "runs.npz")
    r = subprocess.run([sys.executable, "-c", _DECODE_PROBE % dict(root=ROOT, cases=DECODE_CASES), path],
                       capture_output=True, text=True, timeout=3600, cwd=EMU)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return dict(np.load(path))


@pytest.fixture(scope="module")
def fork_stats():
    spec = importlib.util.spec_from_file_location("_fork_stats", os.path.join(ROOT, "tools", "fork_stats.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


@pytest.mark.parametrize("name,kind,ckw", DECODE_CASES, ids=[c[0] for c in DECODE_CASES])
def test_decodes_like_the_oracle(runs, fork_stats, name, kind, ckw):
    kw, x, _ = common.make_case(kind, **ckw)
    bits = runs[name + "/bits"]
    if kind == "SCLUTDecoder":
        assert np.array_equal(bits, fork_stats.hooked_oracle().OracleDecoder(kind, **kw).decode(x))
        return
    want, pm_want, win_want = fork_stats.hooked_oracle().OracleDecoder(kind, **kw).decode(x, return_pm=True)
    assert np.array_equal(bits, want)
    assert np.array_equal(runs[name + "/pm"], pm_want)
    assert np.array_equal(runs[name + "/win"], win_want)
    _, classes = fork_stats.fork_classes(kind, kw, x)
    seen, taken = (int(v) for v in runs[name + "/counts"])
    L = kw["L"]
    assert seen == -(-x.shape[0] // (32 // L)) * int((np.asarray(kw["frozen_bits"]) == 0).sum())
    assert taken == fork_stats.warp_identity(classes, kw["frozen_bits"], L)
