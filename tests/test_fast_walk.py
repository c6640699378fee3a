"""The Fast-SSC walks of scl_lut_warp (FastSCLUTDecoder, FastSCLLUTDecoder, CAFastSCLLUTDecoder), through the host
emulator (tools/emu), on codes that between them reach every special-node shape the project's constructions produce
(tests/fast_walk.py):
  * coverage: the NR / PW / GA sweep still reaches every cell of a committed list, and the picked codes cover it;
  * plan: the op list plan_fast_lut compiles (SP type, SUB8 or SBEGIN..SEND, SF2/SG2/SC2 half) equals the Python
    restatement, and the decoder is on scl_lut_warp exactly when the restatement says it may be;
  * decoding: bits, debug path metrics and winners equal the oracle's bit for bit on AWGN frames with min-sum tables and
    on a tie alphabet.  The metrics pin the order of the R0 / REP penalty sums and the R1 rounds (flip-index rule,
    dead paths, rounds = leaves when a node has fewer than L - 1), which move the metrics long before a decoded bit."""
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
import fast_walk as fw  # noqa: E402
from oracle import polar_oracle as po  # noqa: E402

# Every cell the constructions reach (fast_walk.cell_universe lists the conceivable ones).  A change to identify_nodes
# or to a construction that loses one of these fails test_picked_codes_cover_every_reachable_cell.
_UP = "upper"
REACHED = {
    "L1": [(t, s, _UP, side) for t in ("R0", "REP") for s in (16, 32, 64) for side in "LR"]
    + [(t, s, _UP, "L") for t in ("R0", "REP") for s in (128, 256, 512)]
    + [(t, s, p, side) for t in ("R0", "REP") for s, p in ((2, "top+2"), (4, "top+1"), (8, "top")) for side in "LR"]
    + [("R1", 2, "top+2", "L"), ("R1", 2, "top+2", "R"), ("R1", 4, "top+1", "R"), ("R1", 8, "top", "R")]
    + [("R1", s, _UP, "R") for s in (16, 32, 64, 128, 256, 512)]
    + [("SPC", 4, "top+1", side) for side in "LR"] + [("SPC", 8, "top", side) for side in "LR"]
    + [("SPC", s, _UP, side) for s in (16, 32, 64) for side in "LR"]
    + [("SPC", s, _UP, "R") for s in (128, 256, 512)],
    "list": [(t, s, _UP, side) for t in ("R0", "REP") for s in (16, 32, 64) for side in "LR"]
    + [(t, s, _UP, "L") for t in ("R0", "REP") for s in (128, 256, 512)]
    + [(t, s, p, side) for t in ("R0", "REP") for s, p in ((2, "top+2"), (4, "top+1"), (8, "top")) for side in "LR"]
    + [("R1", 2, "top+2", "L"), ("R1", 2, "top+2", "R"), ("R1", 4, "top+1", "R"), ("R1", 8, "top", "R"),
       ("R1", 16, _UP, "R"), ("R1", 32, _UP, "R"),       # <= 16 leaves: selection by extraction; 17..32: sort_r1_packed
       ("R1", "leaves < L-1"), ("R1", "list not full")],
}


def test_picked_codes_cover_every_reachable_cell():
    r = fw.reach()
    for cls in ("L1", "list"):
        every = set().union(*r[cls].values())
        assert len(REACHED[cls]) == len(set(REACHED[cls]))
        lost = set(REACHED[cls]) - every
        assert not lost, "%s: no construction reaches %s any more" % (cls, sorted(lost, key=str))
        assert every <= fw.cell_universe(cls)
        picked = fw.picked(cls)
        by = {}
        for c in picked:
            for cell in r[cls][c]:
                by.setdefault(cell, fw.name(c))
        assert set(by) == every
        print("\n%s: picked %s" % (cls, " ".join(fw.name(c) for c in picked)))
        for cell in sorted(fw.cell_universe(cls), key=lambda c: (c[0], str(c[1]).zfill(4), c[-1])):
            print("  %-36s %s" % (cell, by.get(cell, "not reached by any construction")))


# ---- the compiled walk -------------------------------------------------------------------------------------------
def _plan_cases():
    codes = sorted(set(fw.picked("L1")) | set(fw.picked("list")), key=lambda c: (c[1], c))
    out = [(fw.name(c) + "-l%d" % L, c, L) for c in codes for L in (1, 2, 4, 8)]
    # BIG's and tools/emu/check.py's N=512 list cases: an R1 node of 64 leaves at depth 3 takes them off the kernel
    out += [("nr-512-300-l8", ("nr", 512, 300), 8), ("nr-512-256-l8", ("nr", 512, 256), 8)]
    return out


_PLAN_PROBE = r"""
import ctypes, json, os, sys
sys.path.insert(0, os.path.join(%(root)r, "tools", "emu"))
import check, common, fast_walk
emu = check.load_emu()
lib = ctypes.CDLL(os.path.join(%(root)r, "tools", "emu", "build", "libpolar_b200.so"))
out = {}
for name, code, L in %(cases)r:
    kind = fast_walk.kind_of(L)
    kw, _, _ = common.make_case(kind, N=code[1], K=code[2], L=L, B=1, seed=3, frozen=fast_walk.frozen_of(code))
    try:
        d = getattr(emu, kind)(**kw)
    except Exception as e:
        out[name] = dict(refused=str(e))
        continue
    ops = (ctypes.c_uint32 * (2 * 8192))()
    voff = (ctypes.c_int * 16)()
    gl, words = ctypes.c_int(), ctypes.c_longlong()
    stream = (ctypes.c_uint32 * 1)()
    nops = lib.pb_emu_fast_plan_detail(ctypes.c_void_p(d._handle), ops, 8192, voff, ctypes.byref(gl), stream,
                                       ctypes.c_longlong(0), ctypes.byref(words))
    out[name] = dict(kernel=d.kernel, n_ops=nops, ops=list(ops[:2 * max(nops, 0)]))
print(json.dumps(out))
"""


def _build_emu():
    r = subprocess.run(["bash", os.path.join(EMU, "build.sh")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def _probe(src, *args, timeout):
    r = subprocess.run([sys.executable, "-c", src] + list(args), capture_output=True, text=True, timeout=timeout, cwd=EMU)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return r.stdout


PLAN_CASES = _plan_cases()


@pytest.fixture(scope="module")
def plans():
    _build_emu()
    out = _probe(_PLAN_PROBE % dict(root=ROOT, cases=PLAN_CASES), timeout=1800)
    return json.loads(out.strip().splitlines()[-1])


@pytest.mark.parametrize("name,code,L", PLAN_CASES, ids=[c[0] for c in PLAN_CASES])
def test_plan_matches_the_restatement(plans, name, code, L):
    p = plans[name]
    ops, _, eligible, root_special = fw.fast_walk(code[1], fw.frozen_of(code), L)
    if root_special:
        assert "root itself is a special node" in p.get("refused", ""), p
        return
    assert "refused" not in p, p["refused"]
    assert (p["kernel"] == "scl_lut_warp") == eligible, (p["kernel"], eligible)
    if not eligible:
        assert p["n_ops"] == -1
        return
    assert p["n_ops"] == len(ops)
    for i, (ty, dd, arg, node) in enumerate(ops):
        x, y = p["ops"][2 * i], p["ops"][2 * i + 1]
        assert (x & 0xff, (x >> 8) & 0xff, (x >> 16) & 0xff, y) == (ty, dd, arg, node), (i, hex(x), y)


# ---- decoding ----------------------------------------------------------------------------------------------------
DECODE_CASES = fw.decode_cases(256)

_DECODE_PROBE = r"""
import ctypes, os, sys
import numpy as np
sys.path.insert(0, os.path.join(%(root)r, "tools", "emu"))
import check, common, fast_walk
emu = check.load_emu()
lib = ctypes.CDLL(os.path.join(%(root)r, "tools", "emu", "build", "libpolar_b200.so"))
res = {}
for name, kind, code, ckw in %(cases)r:
    L = ckw.get("L", 1)
    kw, x, _ = common.make_case(kind, B=2 * (32 // L) + 1, frozen=fast_walk.frozen_of(code), **ckw)
    d = getattr(emu, kind)(**kw)
    assert d.kernel == "scl_lut_warp", (name, d.kernel)
    pm = np.zeros((x.shape[0], L), np.float64)
    win = np.zeros(x.shape[0], np.int32)
    assert lib.pd_set_debug_outputs(ctypes.c_void_p(d._handle), ctypes.c_void_p(pm.ctypes.data), ctypes.c_void_p(win.ctypes.data)) == 0
    res[name + "/bits"] = d.decode(x)
    lib.pd_set_debug_outputs(ctypes.c_void_p(d._handle), None, None)
    res[name + "/pm"], res[name + "/win"] = pm, win
np.savez(sys.argv[1], **res)
"""


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    _build_emu()
    path = str(tmp_path_factory.mktemp("fast_walk") / "runs.npz")
    _probe(_DECODE_PROBE % dict(root=ROOT, cases=DECODE_CASES), path, timeout=3600)
    return dict(np.load(path))


@pytest.mark.parametrize("name,kind,code,ckw", DECODE_CASES, ids=[c[0] for c in DECODE_CASES])
def test_decodes_like_the_oracle(runs, name, kind, code, ckw):
    L = ckw.get("L", 1)
    kw, x, _ = common.make_case(kind, B=2 * (32 // L) + 1, frozen=fw.frozen_of(code), **ckw)
    want, pm_want, win_want = po.OracleDecoder(kind, **kw).decode(x, return_pm=True)
    assert np.array_equal(runs[name + "/bits"], want)
    assert np.array_equal(runs[name + "/pm"], pm_want)
    assert np.array_equal(runs[name + "/win"], win_want)
