#!/usr/bin/env python
"""Benchmark of the decode hot path.  Default: the north-star shape of BASELINE.json (SCL-LUT, N=1024, A=K=512, L=8,
QDecoder=16); --config C1..C5 selects the other BASELINE.json configurations (synthetic AWGN frames of each shape).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config NS|C1|C2|C3|C4|C5] [--batch F]
                    [--dump-outputs DIR]

A "step" decodes one batch of F frames per GPU (inputs > L2 so no flush is needed).  Prints ONE JSON line:
  value     decoded frames/s over all GPUs, inputs resident in HBM (pd_decode_device), CUDA-event timed, max over ranks
  e2e       the same metric through the reference-facing call with HOST buffers, H2D / D2H copies inside: the pybind
            class's decode((B,N) numpy array) -> C ABI pd_decode, input in pinned host memory in the compact dtype
  e2e_api   the same call exactly as the reference drivers make it: int32 symbols / float64 in PAGEABLE numpy memory
            (the library narrows and stages them: bound by host memory bandwidth, 4-8 bytes read per symbol)
  e2e_cabi  pd_decode on caller-pinned uint8/fp64 buffers (what a C caller that owns its buffers gets)
  roofline  algorithmic bytes (N symbols in + K bits out per frame) / kernel time vs measured HBM peak
  cpu_baseline  the compiled reference (oracle/_ref), one process per host core, on a bounded sample (N=1 only)
`--impl reference` times the reference's own CPU implementation on the same workload instead.
`--dump-outputs DIR` writes what the last timed step computed, for comparing two builds output for output:
  decoded_bits.npy  float32 [frames, A], rank 0's frames only: a fixed seeded sample of the batch that rank 0 decoded in
                    the step (all of it when it fits in 56 MB)
  frame_index.npy   float64 [frames], the rows of rank 0's batch that decoded_bits holds
  error_counts.npy  float64 [2], bit errors and block errors of the step summed over ALL GPUs (with --gpus 1: over the
                    whole batch, not just the sampled rows)
The inputs depend only on the arguments (seeded per rank), so two runs with the same arguments decode the same frames.
Multi-GPU: one process per GPU (torchrun); frames are sharded, no data-path collective; the only exchange is the
NCCL all-reduce of the two error counters (bit / block errors), inside the timed region.
"""
import argparse
import ctypes
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)
PKG = os.path.join(ROOT, "quantized_decoder_polar_codes_b200")


def _sim():
    """simulation.py (plain numpy helpers) loaded by path: the reference arm must not import the package, whose __init__
    loads the CUDA extension"""
    name = "_polar_b200_simulation"
    if name not in sys.modules:
        spec = importlib.util.spec_from_file_location(name, os.path.join(PKG, "simulation.py"))
        m = importlib.util.module_from_spec(spec)
        sys.modules[name] = m
        spec.loader.exec_module(m)
    return sys.modules[name]


# BASELINE.json configurations.  api_dtype = what the reference driver of that configuration hands to decode().
CONFIGS = {
    "NS": dict(kind="SCLLUTDecoder", N=1024, A=512, K=512, L=8, ebn0=2.0, dev_dtype="u8", api_dtype="int32", frames=524288,
               workload="SCL-LUT N=1024 A=K=512 L=8 QDecoder=QChannel=16, MinDistortion LUTs (reference generator, design 3 dB), AWGN Eb/N0=2.0 dB through the driver's channel quantizer, NR-sequence frozen set",
               metric="decoded frames/s (info Gbit/s = frames/s*512/1e9), N=1024 L=8 SCL-LUT"),
    "C1": dict(kind="SCDecoder", N=128, A=64, K=64, L=1, ebn0=2.0, dev_dtype="f64", api_dtype="float64", frames=1 << 19,
               workload="float SC N=128 A=K=64, AWGN Eb/N0=2.0 dB channel LLRs (mainFPDecoder.py), NR-sequence frozen set",
               metric="decoded frames/s, float SC N=128 A=64"),
    "C2": dict(kind="SCLUTDecoder", N=128, A=32, K=32, L=1, ebn0=2.0, dev_dtype="u8", api_dtype="int32", frames=1 << 21,
               workload="SC-LUT N=128 A=K=32 QDecoder=QChannel=16, MinDistortion LUTs (reference generator, design 3 dB), AWGN Eb/N0=2.0 dB",
               metric="decoded frames/s, MinDistortion SC-LUT N=128 A=32"),
    "C3": dict(kind="SCLLUTDecoder", N=128, A=32, K=32, L=8, ebn0=2.0, dev_dtype="u8", api_dtype="int32", frames=1 << 20,
               workload="SCL-LUT N=128 A=K=32 L=8 QDecoder=QChannel=16, MinDistortion LUTs (reference generator, design 3 dB), AWGN Eb/N0=2.0 dB",
               metric="decoded frames/s, MinDistortion SCL-LUT N=128 A=32 L=8"),
    "C4": dict(kind="CAFastSCLLUTDecoder", N=1024, A=512, K=536, L=8, ebn0=2.0, dev_dtype="u8", api_dtype="float64", frames=131072,
               workload="CRC-aided FastSCL-LUT N=1024 A=512 (+CRC-24, K=536) L=8 QDecoder=QChannel=16, MMI LUTs (probability domain, design 3 dB), AWGN Eb/N0=2.0 dB through the MMI channel quantizer",
               metric="decoded frames/s, MMI CA-FastSCL-LUT N=1024 A=512 L=8"),
    "C5": dict(kind="SCLUniformQuantizedDecoder", N=2048, A=1024, K=1024, L=32, ebn0=2.0, dev_dtype="f64", api_dtype="float64", frames=1 << 14,
               workload="uniformly quantized SCL N=2048 A=K=1024 L=32 v=16, GA construction, optimal uniform step sizes (reference design code), AWGN Eb/N0=2.0 dB LLRs through QUniform",
               metric="decoded frames/s, uniformly quantized SCL N=2048 A=1024 L=32"),
}


def make_workload(cfg, frames, seed):
    """-> constructor kwargs (numpy tables), inputs [frames, N] in the device dtype, transmitted message [frames, A]"""
    sim = _sim()
    N, A, K, L, eb, kind = cfg["N"], cfg["A"], cfg["K"], cfg["L"], cfg["ebn0"], cfg["kind"]
    rng = np.random.default_rng(seed)
    if kind == "SCLUniformQuantizedDecoder":                 # C5 (mainQuantizedDecoder_ContinuousDomain.py:95-104,186-192)
        v = 16
        sigma = sim.awgn_sigma(eb, K / N)
        fm, mm = sim.frozen_mask_ga(N, K, sigma)
        r_f, r_g = sim.uniform_quantizer_steps(N, v, sigma)
        msg = rng.integers(0, 2, (frames, K), dtype=np.uint8)
        llr = sim.awgn_llr(sim.polar_encode(msg, fm), sigma, rng)
        r = r_f[0]
        M = (v // 2 - 0.5) * r
        x = np.where(np.abs(llr) > M, np.sign(llr) * (M - 0.5 * r), (np.floor(llr / r) + 0.5) * r)
        return dict(N=N, K=K, L=L, frozen_bits=fm, message_bits=mm, decoder_r_f=r_f, decoder_r_g=r_g, v=v), x, msg
    fm, mm = sim.frozen_mask(N, K)
    msg = rng.integers(0, 2, (frames, A), dtype=np.uint8)
    cw = sim.polar_encode(sim.crc_attach(msg) if K > A else msg, fm)
    sigma = sim.awgn_sigma(eb, A / N)
    kw = dict(N=N, K=K, frozen_bits=fm, message_bits=mm)
    if kind == "SCDecoder":                                  # C1
        return kw, sim.awgn_llr(cw, sigma, rng), msg
    if L > 1:
        kw["L"] = L
    if kind == "CAFastSCLLUTDecoder":                        # C4: MMI tables, symbols cut from y (probability-domain driver)
        z = np.load(os.path.join(PKG, "data", "mmi_n1024_q16_3dB.npz"))
        kw.update(A=A, node_type=sim.identify_nodes(N, fm), virtual_channel_llr=z["llrs"])
        edges = z[f"chan_A{A}_eb{eb:.0f}/edges"]
        y = (1.0 - 2.0 * cw) + rng.normal(0.0, sigma, cw.shape)
        sym = np.where(y <= edges[0], 0, np.where(y >= edges[-1], 15, np.searchsorted(edges, y, side="left") - 1)).astype(np.uint8)
    else:                                                    # NS / C2 / C3: MinDistortion tables, LLR-domain driver's quantizer
        if N == 1024:
            z = np.load(os.path.join(PKG, "data", "mindistortion_n1024_q16_3dB.npz"))
            edges, clut = z[f"chan_A{A}_eb{eb:.0f}/edges"], z[f"chan_A{A}_eb{eb:.0f}/lut"]
            kw["virtual_channel_llr"] = z["llr_quanta"]
        else:
            z = np.load(os.path.join(ROOT, "tests", "golden", "real_lut_n128.npz"))
            edges, clut = z[f"A{A}_eb{eb:.0f}/chan_edges"], z[f"A{A}_eb{eb:.0f}/chan_lut"]
            kw["virtual_channel_llr"] = z["llr_quanta"]
        llr = sim.awgn_llr(cw, sigma, rng)
        idx = np.clip(np.searchsorted(edges[:-1], llr, side="left") - 1, 0, clut.size - 1)
        sym = np.where(llr <= edges[0], 0, np.where(llr >= edges[-1], 15, clut[idx])).astype(np.uint8)
    kw["LUT_f"] = [z["lut_f"][p].astype(np.int32)[None] for p in range(N - 1)]
    kw["LUT_g"] = [z["lut_g"][p].astype(np.int32)[None] for p in range(N - 1)]
    return kw, sym, msg


def tile_frames(sym, msg, frames):
    reps = -(-frames // sym.shape[0])
    return np.tile(sym, (reps, 1))[:frames], np.tile(msg, (reps, 1))[:frames]


# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md): NVML polled every 10 ms from a
    thread (nvidia-smi as a fallback, which is too slow for sub-second regions)."""
    SMI_Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.sm, self.mx, self.reasons = [], 0.0, set()
        self.stop = False
        self.th = None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES when it lists indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = gpu_index
            if vis and all(t.strip().isdigit() for t in vis.split(",")):
                phys = int(vis.split(",")[gpu_index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll_nvml(self):
        n = self.nvml
        bits = {"hw_slowdown": n.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": n.nvmlClocksThrottleReasonHwThermalSlowdown,
                "sw_thermal_slowdown": n.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": n.nvmlClocksThrottleReasonSwPowerCap}
        while not self.stop:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
                self.mx = max(self.mx, float(n.nvmlDeviceGetMaxClockInfo(self.h, n.NVML_CLOCK_SM)))
                r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.01)

    def _poll_smi(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.SMI_Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                r = [t.strip() for t in out.split(",")]
                self.sm.append(float(r[0]))
                self.mx = max(self.mx, float(r[1]))
                for nme, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(nme)
            except Exception:
                pass
            time.sleep(0.05)

    def __enter__(self):
        self.th = threading.Thread(target=self._poll_nvml if self.nvml else self._poll_smi, daemon=True)
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.th.join(timeout=6)

    def summary(self):
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.mx or None,
                "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml" if self.nvml else "nvidia-smi"}


# ---------------------------------------------------------------------------------------------------
def _ref_kwargs(kw):
    """numpy tables -> the nested lists the compiled reference takes, one table per position (tests/common.py: ref_kwargs)"""
    out, N = {}, kw["N"]
    for k, val in kw.items():
        if k in ("LUT_f", "LUT_g"):
            lst = []
            for p_, t in enumerate(val):
                t = np.asarray(t)
                npos = N >> (int(np.floor(np.log2(p_ + 1))) + 1)
                lst.append((np.broadcast_to(t, (npos,) + t.shape[1:]) if t.shape[0] == 1 and npos > 1 else t).tolist())
            out[k] = lst
        else:
            out[k] = val.tolist() if isinstance(val, np.ndarray) else val
    return out


def _ref_worker(args):
    kind, kw, x, core = args
    try:
        os.sched_setaffinity(0, {core})
    except Exception:
        pass
    sys.path.insert(0, ROOT)
    from oracle import polar_oracle as po
    ref = po.load_reference()
    lut = "LUT" in kind
    xx = x.astype(np.int32) if lut else x.astype(np.float64)
    if ref is not None:
        dec = getattr(ref, kind)(**_ref_kwargs(kw))
        t0 = time.perf_counter()
        for i in range(xx.shape[0]):
            dec.decode(xx[i])
        how = "reference"
    else:
        dec = po.OracleDecoder(kind, **kw)
        t0 = time.perf_counter()
        dec.decode(xx)
        how = "port"
    return time.perf_counter() - t0, how


def cpu_reference_throughput(kind, kw, x, frames_per_core, cores=None):
    """The reference's own CPU decode() (oracle/_ref) on `cores` pinned processes, disjoint shards of the same
    pre-generated inputs; frames/s = total frames / slowest process wall time (BASELINE.md section 3)."""
    import multiprocessing as mp
    avail = sorted(os.sched_getaffinity(0))
    cores = cores or len(avail)
    jobs = []
    for c in range(cores):
        shard = x[(c * frames_per_core) % x.shape[0]:][:frames_per_core]
        if shard.shape[0] < frames_per_core:
            shard = np.tile(x, (-(-frames_per_core // x.shape[0]), 1))[:frames_per_core]
        jobs.append((kind, kw, shard, avail[c % len(avail)]))
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        res = pool.map(_ref_worker, jobs)
    wall = max(r[0] for r in res)
    return cores * frames_per_core / wall, cores, res[0][1], wall


def ref_frames_per_core(cfg, args):
    """bounded sample: a few seconds of CPU work per step and core (the reference needs 20 ms per N=1024 L=8 frame, 2 s per C5 frame)"""
    if args.ref_frames > 0:
        return args.ref_frames
    return {"NS": 400, "C4": 400, "C1": 200000, "C2": 100000, "C3": 20000, "C5": 4}[args.config]


# ---------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    fpc = ref_frames_per_core(cfg, args)
    kw, x, _ = make_workload(cfg, min(256 if cfg["N"] >= 1024 else 4096, max(fpc, 16)), seed=0)
    times = []
    for it in range(args.warmup + args.steps):
        fps, cores, how, wall = cpu_reference_throughput(cfg["kind"], kw, x, fpc)
        if it >= args.warmup:
            times.append((fps, wall))
    fps = float(np.mean([t[0] for t in times]))
    ms = float(np.mean([t[1] for t in times]) * 1e3)
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": cfg["dev_dtype"], "data": "synthetic",
        "config": {"workload": cfg["workload"], "name": args.config},
        "run": {"frames_per_step": cores * fpc, "info_gbit_s": fps * cfg["A"] / 1e9},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": how,
                         "sample": f"{fpc} frames per core per step, one pinned process per core, per-frame decode() calls"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(json.dumps(line))


def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    import quantized_decoder_polar_codes_b200 as q
    from quantized_decoder_polar_codes_b200 import capi
    from quantized_decoder_polar_codes_b200 import distributed as D

    cfg = CONFIGS[args.config]
    N, A, kind = cfg["N"], cfg["A"], cfg["kind"]
    lut = cfg["dev_dtype"] == "u8"
    esz = 1 if lut else 8
    pd_dtype = capi.PD_U8 if lut else capi.PD_F64
    if world > 1:      # the ranks of one box share its host cores: size each rank's staging pool accordingly
        os.environ.setdefault("POLAR_B200_HOST_THREADS", str(max(2, (os.cpu_count() or 16) // world)))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    D.init("nccl", dev)
    kw, x0, msg0 = make_workload(cfg, 8192 if N >= 1024 else 65536, seed=rank)
    dec = getattr(q, kind)(device=local_rank, **kw)
    lib = capi.lib()
    Kout = lib.pd_out_len(dec._handle)
    bytes_per_frame = N * esz + Kout               # SURVEY.md 8(d): symbols (or fp64 LLRs) in + one byte per decoded bit out
    # frames per step: --batch, or by default the multiple of the kernel's wave (SMs x resident warps x frames per warp)
    # nearest to the configuration's nominal batch
    F = args.batch
    wave = capi.wave_frames(dec, pd_dtype)
    if F <= 0:
        F = max(1, round(cfg["frames"] / wave)) * wave if wave > 0 else cfg["frames"]
    x, msg = tile_frames(x0, msg0, F)
    stream = torch.cuda.current_stream().cuda_stream

    d_in = torch.from_numpy(x).to(dev)
    d_truth = torch.from_numpy(msg).to(dev)
    d_out = torch.empty((F, Kout), dtype=torch.uint8, device=dev)
    counters = torch.zeros(2, dtype=torch.int64, device=dev)   # run totals (identical on every rank)
    step_cnt = torch.zeros(2, dtype=torch.int64, device=dev)   # this step's local counts -> all-reduced -> added to the totals
    l2_note = "inputs+outputs per step exceed L2 (no flush needed)" if F * bytes_per_frame > 126 * 2 ** 20 else "batch below L2 size"
    assert Kout == A, "the error counters compare A message bits"

    def count_and_reduce():
        step_cnt.zero_()
        capi.check(lib.pd_count_errors(d_out.data_ptr(), d_truth.data_ptr(), F, A, step_cnt.data_ptr(), stream))
        D.allreduce_counters(step_cnt)   # the path's only exchange: 2 x int64 over NCCL/NVLink
        counters.add_(step_cnt)

    def step_device():
        capi.decode_device(dec, d_in.data_ptr(), pd_dtype, F, d_out.data_ptr(), stream)
        count_and_reduce()

    def barrier():
        D.barrier()
        torch.cuda.synchronize()

    def note(msg):
        if args.verbose and rank == 0:
            print(f"[bench] {msg}", file=sys.stderr, flush=True)

    note(f"workload ready: F={F} wave={wave} kernel={dec.kernel}")
    for _ in range(args.warmup):
        counters.zero_()
        step_device()
    barrier()
    note("warm-up done")
    # --- device-resident timing: whole step and the decode kernel alone (roofline) ---
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    counters.zero_()
    with ClockSampler(local_rank) as clk:
        barrier()
        l_before = lib.pd_launch_count()
        ev[0].record()
        for i in range(args.steps):
            kev[i][0].record()
            capi.decode_device(dec, d_in.data_ptr(), pd_dtype, F, d_out.data_ptr(), stream)
            kev[i][1].record()
            count_and_reduce()
        ev[1].record()
        barrier()
        l_after = lib.pd_launch_count()
    capi.sync_check(dec, stream)
    elapsed_ms = ev[0].elapsed_time(ev[1])
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    elapsed_ms = D.max_over_ranks(elapsed_ms, dev)
    kernel_ms = D.max_over_ranks(kernel_ms, dev)
    value = world * F * args.steps / (elapsed_ms / 1e3)
    cnt = counters.cpu().tolist()
    total_frames = world * F * args.steps
    ref_out = d_out.cpu().numpy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ref_out, step_cnt.cpu().numpy())
    note(f"device-resident: {value:.4g} frames/s")

    # --- end to end (1), `e2e`: the reference-facing call -- decode((B,N) array) of the pybind class -- on input in pinned host
    #     memory in the compact dtype (uint8 symbols / float64 LLRs), result a fresh numpy array; H2D and D2H copies inside ---
    h_in_p = lib.pd_host_alloc(F * N * esz)
    h_out_p = lib.pd_host_alloc(F * Kout)
    h_in = np.ctypeslib.as_array(ctypes.cast(h_in_p, ctypes.POINTER(ctypes.c_uint8 if lut else ctypes.c_double)), (F, N))
    h_out = np.ctypeslib.as_array(ctypes.cast(h_out_p, ctypes.POINTER(ctypes.c_uint8)), (F, Kout))
    h_in[:] = x
    for _ in range(2):
        got = dec.decode(h_in)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        got = dec.decode(h_in)
    e2e_s = time.perf_counter() - t0
    e2e_value = world * F * args.steps / D.max_over_ranks(e2e_s, dev)
    same = bool((got == ref_out).all())
    note(f"e2e through decode() on pinned input: {e2e_value:.4g} frames/s")

    # --- end to end (2), `e2e_api`: the same call exactly as the reference drivers make it: input in the drivers' dtype (int32
    #     symbols / float64) in pageable numpy memory; the library narrows and stages it (host-memory bound: 4-8 B per symbol) ---
    x_api = x.astype(cfg["api_dtype"])
    for _ in range(2):
        got = dec.decode(x_api)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        got = dec.decode(x_api)
    e2e_api_s = time.perf_counter() - t0
    e2e_api = world * F * args.steps / D.max_over_ranks(e2e_api_s, dev)
    same_api = bool((got == ref_out).all())
    del x_api
    note(f"e2e through decode() as the drivers call it: {e2e_api:.4g} frames/s")

    # --- end to end (3), `e2e_cabi`: the C ABI's host-buffer call on the same pinned buffers ---
    for _ in range(2):
        capi.decode_host(dec, h_in_p, pd_dtype, F, h_out_p)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        capi.decode_host(dec, h_in_p, pd_dtype, F, h_out_p)
    torch.cuda.synchronize()
    e2e_c_s = time.perf_counter() - t0
    e2e_cabi = world * F * args.steps / D.max_over_ranks(e2e_c_s, dev)
    same = same and bool((h_out == ref_out).all())
    del h_in, h_out
    lib.pd_host_free(h_in_p)
    lib.pd_host_free(h_out_p)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = bytes_per_frame * F / (kernel_ms / 1e3) / 1e9
        traffic = None
        try:   # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this kernel, per frame
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if tj.get("kernel") == dec.kernel and tj.get("config", "NS") == args.config:
                traffic = tj["dram_bytes_per_frame"] * F
        except Exception:
            pass
        n_launch = int(l_after - l_before)
        line = {
            "metric": cfg["metric"], "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": cfg["dev_dtype"], "data": "synthetic",
            "config": {"workload": cfg["workload"], "name": args.config},
            "run": {"frames_per_step_per_gpu": F, "wave_frames": wave, "info_gbit_s": value * A / 1e9, "kernel": dec.kernel, "l2": l2_note,
                    "bit_errors": cnt[0], "block_errors": cnt[1], "frames_counted": total_frames,
                    "unique_frames": int(x0.shape[0]), "e2e_outputs_equal_device_output": same and same_api},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback",
                         "kernel_ms": kernel_ms, "bytes_per_frame": bytes_per_frame,
                         "per": f"decode call of one step ({(n_launch // args.steps) - 1} {dec.kernel} launches); algorithmic bytes, kernel_ms and traffic all refer to that call",
                         "note": "HBM-nominal codec path; the kernel is SM-issue bound, not HBM bound (see DESIGN.md 4.1, profiles/)"},
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": F * N * esz, "d2h_bytes_per_step": F * Kout,
                    "call": f"{kind}.decode(({F},{N}) {'uint8' if lut else 'float64'} numpy array in pinned host memory) -> pd_decode -> fresh ({F},{Kout}) uint8 array"},
            "e2e_api": {"value": e2e_api, "unit": "frames/s",
                        "call": f"{kind}.decode(({F},{N}) {cfg['api_dtype']} numpy array, pageable) as the reference drivers call it; {F * N * np.dtype(cfg['api_dtype']).itemsize} host bytes read and narrowed per step"},
            "e2e_cabi": {"value": e2e_cabi, "unit": "frames/s", "call": "pd_decode on pd_host_alloc'ed buffers in the device dtype"},
            "gpu_launches": n_launch,
            "clocks": clk.summary(),
        }
        if world == 1 and not args.no_cpu_baseline:
            try:
                fpc = ref_frames_per_core(cfg, args)
                fps, cores, how, wall = cpu_reference_throughput(kind, kw, x0[:256 if N >= 1024 else 4096], fpc)
                line["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": cores, "kind": how,
                                        "sample": f"{fpc} frames per core ({wall:.1f} s), one pinned process per core, per-frame decode() calls of the compiled reference"}
            except Exception as e:  # pragma: no cover
                line["cpu_baseline"] = {"value": None, "unit": "frames/s", "cores": 0, "kind": "reference", "sample": f"failed: {e}"}
        emit(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_BYTES = 56 << 20     # decoded_bits.npy stays below this; the two small arrays fit in the rest of 64 MB


def dump_outputs(path, bits, step_counts):
    """decoded bits of the last timed step (a seeded sample of its frames when the batch is larger than DUMP_BYTES allows)
    and that step's error counters, as float .npy files under `path`"""
    F, A = bits.shape
    n = min(F, DUMP_BYTES // (4 * A))
    rows = np.arange(F) if n == F else np.sort(np.random.default_rng(0).choice(F, n, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "decoded_bits.npy"), bits[rows].astype(np.float32))
    np.save(os.path.join(path, "frame_index.npy"), rows.astype(np.float64))
    np.save(os.path.join(path, "error_counts.npy"), np.asarray(step_counts, np.float64))


_REAL_STDOUT = None


def protect_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner on stdout when
    NCCL_DEBUG is set): keep a private handle on the real stdout for the result and point fd 1 at stderr for everyone else."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(text):
    out = _REAL_STDOUT or sys.stdout
    out.write(text + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="NS", choices=sorted(CONFIGS), help="BASELINE.json configuration (NS = the north-star shape)")
    ap.add_argument("--batch", type=int, default=0, help="frames per step per GPU (default: the whole number of kernel waves nearest to the configuration's nominal batch)")
    ap.add_argument("--ref-frames", type=int, default=0, help="CPU reference: frames per core per step (default: a few seconds of work)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--verbose", action="store_true", help="progress notes on stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the outputs of the last timed step as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours (the reference arm keeps no outputs)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "ours" and args.gpus > 1 and "RANK" not in os.environ:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29531", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    protect_stdout()
    if args.verbose:
        import faulthandler
        faulthandler.dump_traceback_later(90, repeat=True, file=sys.stderr)   # where it hangs, if it hangs
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
