#!/usr/bin/env python
"""How often a fork of the list decoders changes nothing, counted by the CPU oracle (oracle/polar_oracle.c).
    python tools/fork_stats.py [--config NS|C3|...] [--frames F] [--seed S]
decodes the first F frames of a bench.py configuration (same workload, same seed) and classifies every fork:
  identity   no flip survives and the keeps stay in their slots
  permuted   no flip survives, the keeps are re-ordered
  flip       at least one flip survives
and, for the plain scl_lut_warp walk (32/L frames per warp), the share of (warp, leaf) forks at which every frame of the
warp is an identity fork where the kernel knows the keeps are sorted: the forks that take the kernel's identity exit
(pb_scl_lut.cuh, fork).

The oracle is not changed: a copy of its source with a per-leaf class hook is compiled into a temporary directory.
Test tooling, like oracle/ (tests/test_fork_identity.py predicts the emulator's exit count with it)."""
import argparse
import ctypes as C
import importlib.util
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE = os.path.join(ROOT, "oracle")

# the class hook around the fork of a list leaf (leaf_action): class 1/2/3 as above, | 4 when the path metrics were in
# non-decreasing slot order before the fork; 0 = no fork at that leaf
_ANCHOR = """        fork_select(x, PM2, parent, flip);
        permute_paths(x, parent);
        for (int i = 0; i < L; ++i) x->uc[i][at] = (uint8_t)(flip[i] ? 1 - dec[parent[i]] : dec[parent[i]]);
"""
_HOOK = """        {
            int sorted_before = 1, nof = 1, ident = 1;
            for (int i = 1; i < L; ++i) if (!(x->PM[i - 1] <= x->PM[i])) sorted_before = 0;
            fork_select(x, PM2, parent, flip);
            for (int i = 0; i < L; ++i) { if (flip[i]) nof = 0; if (parent[i] != i) ident = 0; }
            po_fork_class[leaf] = (int8_t)((nof && ident ? 1 : nof ? 2 : 3) | (sorted_before ? 4 : 0));
        }
        permute_paths(x, parent);
        for (int i = 0; i < L; ++i) x->uc[i][at] = (uint8_t)(flip[i] ? 1 - dec[parent[i]] : dec[parent[i]]);
"""
_DECL = "static void leaf_action(po_ctx *x, int leaf) {"
_MAX_N = 65536

_oracle = None


def hooked_oracle():
    """The oracle's Python front-end on a hooked copy of its C source (built once per process)."""
    global _oracle
    if _oracle is not None:
        return _oracle
    src = open(os.path.join(ORACLE, "polar_oracle.c")).read()
    assert src.count(_ANCHOR) == 1 and src.count(_DECL) == 1, "oracle/polar_oracle.c: fork site not found"
    src = src.replace(_ANCHOR, _HOOK).replace(_DECL, "int8_t po_fork_class[%d];\n" % _MAX_N + _DECL)
    tmp = tempfile.mkdtemp(prefix="fork_stats_")
    c_path, so = os.path.join(tmp, "polar_oracle.c"), os.path.join(tmp, "libpolar_oracle_forks.so")
    with open(c_path, "w") as f:
        f.write(src)
    # the flags of oracle/Makefile's port target
    subprocess.check_call(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-fno-fast-math", "-ffp-contract=off", "-o", so, c_path, "-lm"])
    spec = importlib.util.spec_from_file_location("_polar_oracle_forks", os.path.join(ORACLE, "polar_oracle.py"))
    po = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(po)
    po.build_port = lambda force=False: so
    po.lib()
    shutil.rmtree(tmp)   # (loaded: the mapping outlives the file)
    _oracle = po
    return po


def fork_classes(kind, kw, x):
    """-> (bits [B, Kout] as the oracle decodes them, classes int8 [B, N]) for the inputs x [B, N]"""
    po = hooked_oracle()
    dec = po.OracleDecoder(kind, **kw)
    N = int(kw["N"])
    buf = (C.c_int8 * _MAX_N).in_dll(po.lib(), "po_fork_class")
    view = np.ctypeslib.as_array(buf)
    x = np.asarray(x)
    out = np.empty((x.shape[0], dec.kout), np.uint8)
    classes = np.zeros((x.shape[0], N), np.int8)
    for f in range(x.shape[0]):
        view[:N] = 0
        out[f] = dec.decode(x[f:f + 1])[0]
        classes[f] = view[:N]
    return out, classes


def static_sorted(frozen):
    """Leaves at which the plain kernel calls fork with keeps_sorted: an information leaf whose predecessor is one too
    (a frozen leaf may add to the path metrics), and leaf 0 (the initial metrics 0, +inf, ... are sorted)."""
    info = np.asarray(frozen).astype(np.int64) == 0
    prev = np.ones_like(info)
    prev[1:] = info[:-1]
    return info & prev


def warp_identity(classes, frozen, L):
    """-> number of (warp, leaf) forks that take the identity exit of the plain kernel: frame groups of 32/L consecutive
    frames per warp (the last warp's missing frames repeat the last frame, as the kernel does)."""
    B, N = classes.shape
    fpw = 32 // L
    W = -(-B // fpw)
    rows = np.minimum(np.arange(W * fpw), B - 1)
    ident = ((classes[rows] & 3) == 1).reshape(W, fpw, N).all(axis=1)
    return int(ident[:, static_sorted(frozen)].sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="NS")
    ap.add_argument("--frames", type=int, default=2048)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    sys.path.insert(0, ROOT)
    sys.dont_write_bytecode = True
    import bench
    cfg = bench.CONFIGS[args.config]
    L = cfg["L"]
    if L < 2 or L > 8:
        sys.exit(f"{args.config}: L = {L}, the scl_lut_warp fork needs 2 <= L <= 8")
    kw, x, msg = bench.make_workload(cfg, args.frames, seed=args.seed)
    bits, cls = fork_classes(cfg["kind"], kw, x)
    frozen = np.asarray(kw["frozen_bits"])
    forks = cls != 0
    n = int(forks.sum())
    c = cls & 3
    print(f"{args.config}: {cfg['kind']} N={cfg['N']} L={L}, {args.frames} frames (seed {args.seed}), "
          f"{int((bits[:, :msg.shape[1]] != msg).any(axis=1).sum())} block errors, {n // args.frames} forks per frame")
    print("| | share of forks |\n|---|---|")
    for k, name in ((1, "no flip survives, order unchanged (per frame)"), (2, "no flip survives, keeps re-ordered"),
                    (3, "at least one flip survives")):
        print(f"| {name} | {100 * (c == k).sum() / n:.1f} % |")
    fpw = 32 // L
    W = args.frames // fpw
    ss = static_sorted(frozen)
    ident = (c[:W * fpw] == 1).reshape(W, fpw, -1).all(axis=1)
    info = frozen == 0
    print(f"| all {fpw} frames of a warp unchanged at the same leaf | {100 * ident[:, info].mean():.1f} % |")
    print(f"| the same at a leaf where the kernel knows the keeps are sorted: identity exits | "
          f"{100 * ident[:, ss].sum() / (W * info.sum()):.1f} % |")
    q = cfg["N"] // 4
    for k in range(4):
        sel = np.nonzero(info[k * q:(k + 1) * q])[0] + k * q
        rate = f"{100 * ident[:, sel].mean():.1f} %" if len(sel) else "-"
        print(f"leaves {k * q}-{(k + 1) * q - 1}: {len(sel)} forks, warp identity {rate}")
    p = ident[:, info].mean(axis=0)
    print(f"information positions with a warp identity rate >= 99 %: {(p >= 0.99).sum()} of {info.sum()}")


if __name__ == "__main__":
    main()
