#!/usr/bin/env python
"""Rates of the on-device Monte-Carlo loop (simulate.Simulator) for the three channel front ends, one JSON line per shape and
batch size:

  gen_fps     pd_sim_generate alone (message, CRC, encode, AWGN, channel front end), CUDA events over >= 1 s
  run_fps     Simulator.run end to end (generate + pd_decode_device + pd_count_errors per batch), host clock over >= 1 s
  decode_fps  the same decoder on one pre-generated device batch, pd_decode_device repeated, CUDA events over >= 1 s
  host_fps    the same front end in numpy on one host process (rng.integers / normal, CRC, encode, rule), without the copy to
              the device -- how a user makes these frames without the generator

Shapes (bench.py's configurations, Eb/N0 = 2 dB):
  NS  SCLLUTDecoder N=1024 A=K=512 L=8, MinDistortion tables      LLRQuantizer (LLR-domain driver)
  C4  CAFastSCLLUTDecoder N=1024 A=512 K=536 L=8, MMI tables      YQuantizer   (probability-domain driver)
  C5  SCLUniformQuantizedDecoder N=2048 A=K=1024 L=32, GA         UniformLLR   (continuous-domain driver)

python tools/bench_sim.py [--shapes NS,C4,C5] [--out FILE]   (writes nothing unless --out is given)"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
DATA = os.path.join(ROOT, "quantized_decoder_polar_codes_b200", "data")
EB = 2.0
BATCHES = {"NS": (1 << 14, 1 << 16, 1 << 18), "C4": (1 << 14, 1 << 16, 1 << 18), "C5": (1 << 12, 1 << 14)}
WINDOW_S = 1.0


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0],
                              f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), (v.strip() for v in out.split(","))))
    except Exception as e:       # the rates stand without it; say why it is missing
        return {"error": repr(e)}


def setup(q, name):
    """-> decoder, frozen mask, A, crc, channel front end, host generator (rng, B) -> frames in the decoder's dtype"""
    from quantized_decoder_polar_codes_b200 import simulation as sim
    from quantized_decoder_polar_codes_b200.simulate import LLRQuantizer, UniformLLR, YQuantizer
    if name == "C5":
        N, K, v = 2048, 1024, 16
        sigma = sim.awgn_sigma(EB, K / N)
        fm, mm = sim.frozen_mask_ga(N, K, sigma)
        r_f, r_g = sim.uniform_quantizer_steps(N, v, sigma)
        dec = q.SCLUniformQuantizedDecoder(N=N, K=K, L=32, frozen_bits=fm, message_bits=mm, decoder_r_f=r_f, decoder_r_g=r_g, v=v)
        r = r_f[0]
        M = (v // 2 - 0.5) * r

        def host(rng, B):
            llr = sim.awgn_llr(sim.polar_encode(rng.integers(0, 2, (B, K), dtype=np.uint8), fm), sigma, rng)
            return np.where(np.abs(llr) > M, np.sign(llr) * (M - 0.5 * r), (np.floor(llr / r) + 0.5) * r)
        return dec, fm, K, False, UniformLLR(r, v), host
    N, A = 1024, 512
    K = A + 24 if name == "C4" else A
    sigma = sim.awgn_sigma(EB, A / N)
    fm, mm = sim.frozen_mask(N, K)
    z = np.load(os.path.join(DATA, "mmi_n1024_q16_3dB.npz" if name == "C4" else "mindistortion_n1024_q16_3dB.npz"))
    kw = dict(N=N, K=K, L=8, frozen_bits=fm, message_bits=mm, LUT_f=[z["lut_f"][p].astype(np.int32)[None] for p in range(N - 1)],
              LUT_g=[z["lut_g"][p].astype(np.int32)[None] for p in range(N - 1)])
    if name == "C4":
        dec = q.CAFastSCLLUTDecoder(A=A, node_type=sim.identify_nodes(N, fm), virtual_channel_llr=z["llrs"], **kw)
        edges = z["chan_A512_eb2/edges"]

        def host(rng, B):
            cw = sim.polar_encode(sim.crc_attach(rng.integers(0, 2, (B, A), dtype=np.uint8)), fm)
            y = (1.0 - 2.0 * cw) + rng.normal(0.0, sigma, cw.shape)
            return np.where(y <= edges[0], 0, np.where(y >= edges[-1], 15, np.searchsorted(edges, y, side="left") - 1)).astype(np.uint8)
        return dec, fm, A, True, YQuantizer(edges, 16), host
    dec = q.SCLLUTDecoder(virtual_channel_llr=z["llr_quanta"], **kw)
    edges, lut = z["chan_A512_eb2/edges"], z["chan_A512_eb2/lut"]

    def host(rng, B):
        llr = sim.awgn_llr(sim.polar_encode(rng.integers(0, 2, (B, A), dtype=np.uint8), fm), sigma, rng)
        idx = np.clip(np.searchsorted(edges[:-1], llr, side="left") - 1, 0, lut.size - 1)
        return np.where(llr <= edges[0], 0, np.where(llr >= edges[-1], 15, lut[idx])).astype(np.uint8)
    return dec, fm, A, False, LLRQuantizer(edges, lut, 16), host


def event_rate(torch, fn, B):
    """frames/s of fn() (B frames per call): warm-up, then calls in one CUDA-event window of at least WINDOW_S"""
    for _ in range(3):
        fn()
    reps = 1
    while True:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        e1.synchronize()
        s = e0.elapsed_time(e1) / 1e3
        if s >= WINDOW_S:
            return reps * B / s, s
        reps = max(reps * 2, int(reps * 1.2 * WINDOW_S / max(s, 1e-6)) + 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="NS,C4,C5")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    import quantized_decoder_polar_codes_b200 as q
    from quantized_decoder_polar_codes_b200 import capi, simulation as sim
    from quantized_decoder_polar_codes_b200.simulate import Simulator
    lines = []

    def emit(rec):
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    emit({"gpu": torch.cuda.get_device_name(0), "nvidia_smi_before": gpu_info()})
    stream = torch.cuda.current_stream().cuda_stream
    for name in args.shapes.split(","):
        dec, fm, A, crc, channel, host = setup(q, name)
        s = Simulator(dec, fm, A=A, crc=crc, channel_quantizer=channel)
        sigma = sim.awgn_sigma(EB, s.rate)
        dt = capi.PD_U8 if s.quantized else capi.PD_F64
        rng = np.random.default_rng(0)
        host(rng, 64)
        hb, hn, t0 = 2048, 0, time.perf_counter()
        while time.perf_counter() - t0 < WINDOW_S:
            host(rng, hb)
            hn += hb
        host_fps = hn / (time.perf_counter() - t0)
        for B in BATCHES[name]:
            msg = torch.empty((B, A), dtype=torch.uint8, device="cuda")
            out = torch.empty((B, s.N), dtype=torch.uint8 if s.quantized else torch.float64, device="cuda")
            dec_out = torch.empty((B, A), dtype=torch.uint8, device="cuda")
            f0 = [0]

            def gen():
                capi.check(s.lib.pd_sim_generate(s._h, sigma, B, 7, f0[0], msg.data_ptr(), out.data_ptr(), stream))
                f0[0] += B
            gen_fps, gen_s = event_rate(torch, gen, B)
            dec_fps, dec_s = event_rate(torch, lambda: capi.decode_device(dec, out.data_ptr(), dt, B, dec_out.data_ptr(), stream), B)
            s.run(EB, 2 * B, batch=B, seed=1)                       # warm-up
            frames = 2 * B
            while True:
                t0 = time.perf_counter()
                res = s.run(EB, frames, batch=B, seed=1)
                run_s = time.perf_counter() - t0
                if run_s >= WINDOW_S:
                    break
                frames = B * max(2 * frames // B, int(frames / B * 1.2 * WINDOW_S / run_s) + 1)
            emit({"shape": name, "channel": type(channel).__name__, "batch": B, "gen_fps": round(gen_fps), "gen_window_s": round(gen_s, 3),
                  "run_fps": round(res["frames"] / run_s), "run_frames": res["frames"], "run_window_s": round(run_s, 3),
                  "run_bler": res["bler"], "decode_fps": round(dec_fps), "decode_window_s": round(dec_s, 3),
                  "host_numpy_fps": round(host_fps), "gen_over_decode": round(gen_fps / dec_fps, 2)})
            del msg, out, dec_out
        del s, dec
    emit({"nvidia_smi_after": gpu_info()})
    if args.out:
        with open(args.out, "w") as f:
            f.write("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()
