"""The Fast-SSC walk of scl_lut_warp (plan_fast_lut in pb_scl_lut.cuh, max_special >= 0) restated in Python, and the set of
codes from the project's own constructions that between them reach every special-node shape the walk can meet.  Shared
by tests/test_fast_walk.py (planner and emulator) and tests/test_gpu_fast_walk.py (B200).

A cell is one special-node shape: (type, leaves, position, side) with position "upper" (a level above the walk's
8-leaf subtrees, depth < top), "top", "top+1" or "top+2" (inside one), and side L / R (left or right child).  List
decoders add two R1 cells: ("R1", "leaves < L-1") -- the node has fewer elements than the L - 1 rounds the reference
would otherwise run -- and ("R1", "list not full") -- fewer than log2(L) information bits precede the node, so dead
paths (PM = inf) take part in its forks."""
import functools

import numpy as np

import common

sim = common.sim

(FOP_UF, FOP_UG, FOP_UC, FOP_SUB8, FOP_SBEGIN, FOP_SF3, FOP_SG3, FOP_SF2, FOP_SG2, FOP_SPAIR, FOP_SC2, FOP_SC3,
 FOP_SEND, FOP_SP) = range(14)
TYPES = ("R0", "R1", "REP", "SPC")
GA_SIGMAS = (0.5, 0.8, 1.1)


def kind_of(L, ca=False):
    return "FastSCLUTDecoder" if L == 1 else ("CAFastSCLLUTDecoder" if ca else "FastSCLLUTDecoder")


def fast_walk(N, frozen, L):
    """-> (ops, cells, eligible, root_special) of the Fast walk of a code at list size L (1 = FastSCLUTDecoder):
    ops = [(type, depth, arg, node)] in the order plan_fast_lut emits them; eligible = the decoder stays on scl_lut_warp
    (a list R1 node wider than 32 leaves sends it to path_warp); root_special = the decoder refuses the code (the root
    is itself a special node)."""
    n = N.bit_length() - 1
    top = n - 3
    node_type = sim.identify_nodes(N, frozen)
    max_special = 3 if L == 1 else 2          # the list decoders expand SPC nodes
    info_before = np.concatenate([[0], np.cumsum(1 - np.asarray(frozen))])

    def special(d, node):
        if d >= n:
            return -1
        t = int(node_type[(1 << d) + node - 1])
        return t if 0 <= t <= max_special else -1

    def plain(d, node):
        return d >= n or (special(d, node) < 0 and plain(d + 1, 2 * node) and plain(d + 1, 2 * node + 1))

    ops, cells = [], set()
    eligible = True

    def walk(d, node):
        nonlocal eligible
        t = special(d, node)
        if t >= 0:
            temp = N >> d
            ops.append((FOP_SP, d, t, node))
            cells.add((TYPES[t], temp, "upper" if d < top else "top" if d == top else "top+%d" % (d - top), "LR"[node & 1]))
            if L > 1 and t == 1:
                eligible &= temp <= 32
                if temp < L - 1:
                    cells.add(("R1", "leaves < L-1"))
                if 2 ** int(info_before[node * temp]) < L:
                    cells.add(("R1", "list not full"))
            return
        if d < top:
            ops.append((FOP_UF, d, 0, node)); walk(d + 1, 2 * node)
            ops.append((FOP_UG, d, 0, node)); walk(d + 1, 2 * node + 1)
            ops.append((FOP_UC, d, 0, node))
        elif d == top:
            if plain(d, node):
                ops.append((FOP_SUB8, d, 0, node))
                return
            ops.extend([(FOP_SBEGIN, d, 0, node), (FOP_SF3, d, 0, node)]); walk(d + 1, 2 * node)
            ops.append((FOP_SG3, d, 0, node)); walk(d + 1, 2 * node + 1)
            ops.extend([(FOP_SC3, d, 0, node), (FOP_SEND, d, 0, node)])
        elif d == top + 1:                  # arg: which half of the 8-leaf subtree
            ops.append((FOP_SF2, d, node & 1, node)); walk(d + 1, 2 * node)
            ops.append((FOP_SG2, d, node & 1, node)); walk(d + 1, 2 * node + 1)
            ops.append((FOP_SC2, d, node & 1, node))
        else:
            ops.append((FOP_SPAIR, d, 0, node))

    walk(0, 0)
    return ops, cells, eligible, special(0, 0) >= 0


def frozen_of(code):
    """code = (construction, N, K), construction "nr", "pw" or "ga<sigma>" -> frozen mask"""
    c, N, K = code
    if c.startswith("ga"):
        return sim.frozen_mask_ga(N, K, float(c[2:]))[0]
    return sim.frozen_mask(N, K, c)[0]


def all_codes():
    """NR and PW at N = 32..1024 for every K; GA at GA_SIGMAS for every K up to N = 64 and every (N/32)-th K above (the
    GA recursion costs 60 ms a code at N = 1024)"""
    for N in (32, 64, 128, 256, 512, 1024):
        for K in range(1, N):
            yield ("nr", N, K)
            yield ("pw", N, K)
        for s in GA_SIGMAS:
            for K in range(1, N, max(1, N // 32)):
                yield ("ga%g" % s, N, K)


def list_cells(N, frozen):
    """-> cells of the list walks over L = 2, 4, 8, or None when no list size keeps the code on the kernel"""
    out, any_ok = set(), False
    for L in (2, 4, 8):
        _, cells, ok, root = fast_walk(N, frozen, L)
        if ok and not root:
            out |= cells
            any_ok = True
    return out if any_ok else None


@functools.lru_cache(maxsize=None)
def reach():
    """-> {"L1": {code: cells}, "list": {code: cells}} over all_codes(), codes the kernel does not run left out"""
    res = {"L1": {}, "list": {}}
    for code in all_codes():
        fm = frozen_of(code)
        N = code[1]
        _, cells, ok, root = fast_walk(N, fm, 1)
        if ok and not root:
            res["L1"][code] = cells
        lc = list_cells(N, fm)
        if lc is not None:
            res["list"][code] = lc
    return res


def _greedy(cands, want):
    picked, left = [], set(want)
    while left:
        best = max(cands, key=lambda c: (len(cands[c] & left), -c[1]))
        if not cands[best] & left:
            break
        picked.append(best)
        left -= cands[best]
    return picked


@functools.lru_cache(maxsize=None)
def picked(cls):
    """Codes picked greedily until they cover every cell the sweep reaches for the class ("L1" or "list"): first among
    N <= 256 (the emulated decode test runs those), then among the rest for what only longer codes reach."""
    r = reach()[cls]
    every = set().union(*r.values())
    small = _greedy({c: v for c, v in r.items() if c[1] <= 256}, every)
    got = set().union(*(r[c] for c in small))
    return tuple(small + _greedy(r, every - got))


def cell_universe(cls):
    """every cell the walk could meet: each special type the class decodes, 2..512 leaves (the root may not be special)
    on either side, list R1 nodes up to 32 leaves, plus the two list-only R1 cells"""
    types = TYPES if cls == "L1" else TYPES[:3]
    out = set()
    for t in types:
        for lg in range(1, 10):
            temp = 1 << lg
            if cls == "list" and t == "R1" and temp > 32:
                continue
            pos = "top+2" if temp == 2 else "top+1" if temp == 4 else "top" if temp == 8 else "upper"
            out |= {(t, temp, pos, "L"), (t, temp, pos, "R")}
    if cls == "list":
        out |= {("R1", "leaves < L-1"), ("R1", "list not full")}
    return out


def name(code):
    return "%s-%d-%d" % code


TIES = (-1.0, -0.0, 0.0, 1.0)


def decode_cases(max_n):
    """(name, kind, code, ckw) for every picked code with N <= max_n the kernel runs: FastSCLUT, FastSCLLUT and (where
    the 24-bit CRC leaves at least 8 message bits) CAFastSCLLUT at L = 2, 4, 8, each on AWGN + min-sum and on ties"""
    out = []
    codes = sorted(set(picked("L1")) | set(picked("list")), key=lambda c: (c[1], c))
    for code in codes:
        N, K = code[1], code[2]
        if N > max_n:
            continue
        fm = frozen_of(code)
        for kind, Ls in (("FastSCLUTDecoder", (1,)), ("FastSCLLUTDecoder", (2, 4, 8)), ("CAFastSCLLUTDecoder", (2, 4, 8))):
            if kind.startswith("CA") and K - 24 < 8:
                continue
            for L in Ls:
                _, _, ok, root = fast_walk(N, fm, L)
                if not ok or root:
                    continue
                for inputs in ("awgn", "ties"):
                    ckw = dict(N=N, K=K, seed=N + K + L)
                    if L > 1:
                        ckw["L"] = L
                    if kind.startswith("CA"):
                        ckw["A"] = K - 24
                    ckw.update(dict(tables="minsum", ebn0_db=1.5) if inputs == "awgn" else dict(alphabet=TIES))
                    out.append(("%s-%s-l%d-%s" % (kind[:-10], name(code), L, inputs), kind, code, ckw))
    return out
