#!/usr/bin/env python
"""Device-resident decode rates of the CRC-aided list decoders at list sizes 32 .. 256, one JSON line per shape:

  CASCLDecoder     fp64 LLRs of encode + AWGN frames: few path-metric ties, most forks take the parallel rank
  CASCLLUTDecoder  min-sum LUT tables on quantized frames: integer-valued metrics, many ties, many forks take the serial
                   exact sort (one thread per CTA runs libstdc++'s introsort over the 2L keys)

N in {128, 512, 1024} (A = N/2, K = A + 24), L in {32, 64, 128, 256}.  L = 32 runs on path_warp (one warp per frame) and is
the reference point; L >= 64 runs on path_cta (one CTA per frame).  fps: pd_decode_device repeated on one device batch,
CUDA events over >= WINDOW_S seconds after a warm-up call.  oracle_fps: the C restatement of the reference
(oracle/polar_oracle.c) on one CPU core -- not the compiled reference -- over the first --oracle-frames frames, whose bits
are also compared (oracle_mismatch).

python tools/bench_large_lists.py [--N 128,512,1024] [--L 32,64,128,256] [--ebn0 2.0] [--out FILE]
(writes nothing unless --out is given)"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
WINDOW_S = 1.0


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0],
                              f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), (v.strip() for v in out.split(","))))
    except Exception as e:       # the rates stand without it; say why it is missing
        return {"error": repr(e)}


def batch_for(N, L):
    """enough frames for several waves of either kernel, capped so that the largest shapes stay within seconds"""
    return int(max(2048, min(65536, (1 << 26) // (N * L))))


def measure(q, kind, N, L, ebn0, oracle_frames):
    import torch
    import common
    from quantized_decoder_polar_codes_b200 import capi
    from oracle import polar_oracle as po
    A = N // 2
    K = A + 24
    B = batch_for(N, L)
    t = "minsum" if "LUT" in kind else "channel"
    kw, x, truth = common.make_case(kind, N, K, L=L, A=A, B=B, seed=1, tables=t, ebn0_db=ebn0)
    dec = getattr(q, kind)(**kw)
    lut = "LUT" in kind
    dt = capi.PD_U8 if lut else capi.PD_F64
    xin = torch.from_numpy(x.astype(np.uint8) if lut else x.astype(np.float64)).cuda()
    out = torch.empty((B, A), dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    capi.decode_device(dec, xin.data_ptr(), dt, B, out.data_ptr(), stream)   # warm-up: workspace, module load
    capi.sync_check(dec, stream)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps, elapsed = 1, 0.0
    while True:
        e0.record()
        for _ in range(reps):
            capi.decode_device(dec, xin.data_ptr(), dt, B, out.data_ptr(), stream)
        e1.record()
        e1.synchronize()
        elapsed = e0.elapsed_time(e1) / 1e3
        if elapsed >= WINDOW_S:
            break
        reps = max(reps * 2, int(reps * WINDOW_S / max(elapsed, 1e-6) * 1.2))
    capi.sync_check(dec, stream)
    got = out.cpu().numpy()
    bler = float((got != truth).any(axis=1).mean())
    orc = po.OracleDecoder(kind, **kw)
    nf = min(oracle_frames, B)
    t0 = time.perf_counter()
    want = orc.decode(x[:nf])
    t_or = time.perf_counter() - t0
    return {"kind": kind, "N": N, "K": K, "A": A, "L": L, "kernel": dec.kernel, "batch": B, "ebn0_db": ebn0,
            "fps": B * reps / elapsed, "window_s": round(elapsed, 3), "bler": bler,
            "oracle_parity_frames": nf, "oracle_mismatch": int((got[:nf] != want).any(axis=1).sum()),
            "oracle_fps": nf / t_or}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", default="128,512,1024")
    ap.add_argument("--L", default="32,64,128,256")
    ap.add_argument("--kinds", default="CASCLDecoder,CASCLLUTDecoder")
    ap.add_argument("--ebn0", type=float, default=2.0)
    ap.add_argument("--oracle-frames", type=int, default=2)
    ap.add_argument("--out")
    a = ap.parse_args()
    import quantized_decoder_polar_codes_b200 as q
    info = gpu_info()
    print(json.dumps({"gpu": info}), flush=True)
    rows = []
    for kind in a.kinds.split(","):
        for N in (int(v) for v in a.N.split(",")):
            for L in (int(v) for v in a.L.split(",")):
                r = measure(q, kind, N, L, a.ebn0, a.oracle_frames)
                r["gpu"] = info.get("name")
                r["power_limit"] = info.get("power.limit")
                print(json.dumps(r), flush=True)
                rows.append(r)
    print(json.dumps({"gpu_after": gpu_info()}), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
