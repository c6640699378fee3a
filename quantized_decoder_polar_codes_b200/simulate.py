"""Batched Monte-Carlo front-end on the GPU (SURVEY.md 8f, row f1): what the reference drivers' frame loop does
(mainQuantizedDecoder_LLRDomain.py:130-192) -- random message, [CRC], polar encode, BPSK + AWGN, LLR, channel
quantizer, decode, BER/BLER counters -- without ever leaving the device.  One process per GPU; with
torch.distributed initialised the two counters are all-reduced (NCCL) at the end of each Eb/N0 point.

The channel front end is one of the reference drivers' (csrc/pb_sim.cuh); `set_channel` swaps it between Eb/N0 points, which
is how the drivers' outer loop runs (a new channel quantizer per point, same code and CRC):

    # LLR-domain driver, MinDistortion tables: symbol = lut[bisect of the LLR over the uniform cells]
    sim = Simulator(decoder, frozen_bits, A=512, crc=False, channel_quantizer=(edges, lut, 16))
    for eb in (1.0, 2.0, 3.0):
        edges, lut = lutgen.llr_channel_quantizer(awgn_sigma(eb, 512 / 1024))
        sim.set_channel(LLRQuantizer(edges, lut, 16))
        res = sim.run(ebn0_db=eb, frames=1 << 22, max_block_errors=1000)    # {'ber':..., 'bler':..., 'frames':..., ...}

    # probability-domain driver, MMI tables: y cut at the MMI channel quantizer's edges, symbol = cell index
    _, interval_x, channel_lut = lutgen.mmi_channel_quantizer(sigma)
    sim.set_channel(YQuantizer(interval_x[channel_lut], 16))

    # continuous-domain driver, uniformly quantized decoders: QUniform of the LLR with the root step, fp64
    r_f, r_g = simulation.uniform_quantizer_steps(N, 16, sigma)
    sim.set_channel(UniformLLR(r_f[0], 16))

`set_channel(None)` gives fp64 LLRs (the float decoders).
"""
import ctypes as C
from typing import NamedTuple

import numpy as np
import torch

from . import capi
from . import distributed as D
from .simulation import CRC24_LOC, awgn_sigma


class LLRQuantizer(NamedTuple):
    """LLR-domain driver (mainQuantizedDecoder_LLRDomain.py:167-176): 0 if llr <= edges[0], q_channel-1 if llr >= edges[-1],
    else lut[bisect_left(edges[:-1], llr) - 1].  edges: interval_x [M+1], lut: channel_lut [M].  uint8 symbols."""
    edges: np.ndarray
    lut: np.ndarray
    q_channel: int


class YQuantizer(NamedTuple):
    """Probability-domain driver (mainQuantizedDecoder_ProbabilityDomain.py:153-177): y (not the LLR) cut at the MMI channel
    quantizer's edges interval_x[channel_lut] [q_channel+1]: 0 if y <= edges[0], q_channel-1 if y >= edges[-1], else
    searchsorted(edges, y, 'left') - 1.  uint8 symbols."""
    edges: np.ndarray
    q_channel: int


class UniformLLR(NamedTuple):
    """Continuous-domain driver's QUniform (mainQuantizedDecoder_ContinuousDomain.py:29-32) with step r = decoder_r_f[0] and
    v levels: M = (v//2 - 0.5) r, sign(llr) (M - r/2) if |llr| > M, else (floor(llr/r) + 0.5) r.  fp64."""
    r: float
    v: int


def _ptr(a):
    return None if a is None else a.ctypes.data


class Simulator:
    """channel_quantizer: None (fp64 LLRs), an (edges, lut, q_channel) tuple or LLRQuantizer, a YQuantizer or a UniformLLR."""

    def __init__(self, decoder, frozen_bits, A, crc=False, channel_quantizer=None, device=None, crc_n=24, crc_loc=CRC24_LOC):
        self.dec = decoder
        self.lib = capi.lib()
        self.N = self.lib.pd_code_len(decoder._handle)
        self.kout = self.lib.pd_out_len(decoder._handle)
        self.A = int(A)
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        fb = np.ascontiguousarray(frozen_bits, dtype=np.int32)
        K = int((fb == 0).sum())
        cfg = capi.SimConfig()
        cfg.N, cfg.K, cfg.A, cfg.device = self.N, K, self.A, self.device.index
        cfg.frozen_bits = fb.ctypes.data
        loc = np.ascontiguousarray(crc_loc, dtype=np.int32)
        if crc:
            cfg.crc_n, cfg.crc_loc, cfg.crc_loc_len = crc_n, loc.ctypes.data, loc.size
        later = None
        if isinstance(channel_quantizer, (YQuantizer, UniformLLR)):     # front ends pd_sim_config has no fields for
            later, channel_quantizer = channel_quantizer, None
        self.channel = None
        if channel_quantizer is not None:
            edges, lut, qc = channel_quantizer
            edges = np.ascontiguousarray(edges, dtype=np.float64)
            lut = np.ascontiguousarray(lut, dtype=np.uint8)
            assert lut.size == edges.size - 1
            cfg.edges, cfg.n_edges, cfg.chan_lut, cfg.q_channel = edges.ctypes.data, edges.size, lut.ctypes.data, int(qc)
            self.channel = LLRQuantizer(edges, lut, int(qc))
        h = C.c_void_p()
        capi.check(self.lib.pd_sim_create(C.byref(cfg), C.byref(h)))
        self._h = h
        self.rate = self.A / self.N
        if later is not None:
            self.set_channel(later)

    @property
    def quantized(self):
        """True when the channel front end emits uint8 symbols (LLRQuantizer, YQuantizer), False for fp64 output."""
        return isinstance(self.channel, (LLRQuantizer, YQuantizer))

    def set_channel(self, channel):
        """Replaces the channel front end (pd_sim_set_channel): None, LLRQuantizer, YQuantizer or UniformLLR.  The code and CRC
        stay; frames already enqueued by generate() keep the tables they were launched with.  Raises ValueError on a bad
        quantizer."""
        ch = capi.SimChannel()
        edges = lut = None
        if channel is None:
            ch.mode = capi.PD_SIM_LLR
        elif isinstance(channel, LLRQuantizer):
            edges = None if channel.edges is None else np.ascontiguousarray(channel.edges, dtype=np.float64)
            if channel.lut is not None:
                lut = np.asarray(channel.lut)
                if lut.size and (lut.min() < 0 or lut.max() > 255):
                    raise ValueError("channel lut entries must be in [0,255]")
                lut = np.ascontiguousarray(lut, dtype=np.uint8)
                if edges is not None and lut.size != edges.size - 1:
                    raise ValueError(f"the lut has {lut.size} entries for {edges.size} edges (need one per cell)")
            ch.mode, ch.q_channel = capi.PD_SIM_LLR_QUANT, int(channel.q_channel)
        elif isinstance(channel, YQuantizer):
            edges = None if channel.edges is None else np.ascontiguousarray(channel.edges, dtype=np.float64)
            ch.mode, ch.q_channel = capi.PD_SIM_Y_QUANT, int(channel.q_channel)
        elif isinstance(channel, UniformLLR):
            ch.mode, ch.r, ch.v = capi.PD_SIM_LLR_UNIFORM, float(channel.r), int(channel.v)
        else:
            raise TypeError(f"unknown channel front end {type(channel).__name__}")
        ch.edges, ch.chan_lut = _ptr(edges), _ptr(lut)
        ch.n_edges = 0 if edges is None else edges.size
        capi.check(self.lib.pd_sim_set_channel(self._h, C.byref(ch)))
        self.channel = channel

    def __del__(self):
        try:
            self.lib.pd_sim_destroy(self._h)
        except Exception:
            pass

    def generate(self, sigma, frames, seed=0, first_frame=0):
        """-> (msg [B,A] uint8, channel output [B,N] uint8 symbols or fp64 LLRs) as device tensors."""
        msg = torch.empty((frames, self.A), dtype=torch.uint8, device=self.device)
        out = torch.empty((frames, self.N), dtype=torch.uint8 if self.quantized else torch.float64, device=self.device)
        s = torch.cuda.current_stream(self.device).cuda_stream
        capi.check(self.lib.pd_sim_generate(self._h, float(sigma), frames, seed, first_frame, msg.data_ptr(), out.data_ptr(), s))
        return msg, out

    def run(self, ebn0_db, frames, batch=1 << 16, seed=0, max_block_errors=None, rank=0, world=1):
        """Decodes `frames` frames (this rank's contiguous share of them) at one Eb/N0 point.  `max_block_errors`
        reproduces the drivers' early stop (> 1000 block errors, :184), checked between batches."""
        if self.kout != self.A:
            raise ValueError(f"the decoder returns {self.kout} bits per frame but the messages have A={self.A}: with a CRC use a "
                             "CRC-aided class (it returns the A message bits); pd_count_errors compares [B][A] rows")
        sigma = awgn_sigma(ebn0_db, self.rate)
        lo, hi = D.shard_range(frames, rank, world)
        s = torch.cuda.current_stream(self.device).cuda_stream
        counters = torch.zeros(3, dtype=torch.int64, device=self.device)   # bit errors, block errors, frames
        dec_out = torch.empty((min(batch, max(hi - lo, 1)), self.kout), dtype=torch.uint8, device=self.device)
        dt = capi.PD_U8 if self.quantized else capi.PD_F64
        f0 = lo
        while f0 < hi:
            nb = min(batch, hi - f0)
            msg, x = self.generate(sigma, nb, seed, f0)
            capi.decode_device(self.dec, x.data_ptr(), dt, nb, dec_out.data_ptr(), s)
            capi.check(self.lib.pd_count_errors(dec_out.data_ptr(), msg.data_ptr(), nb, self.A, counters.data_ptr(), s))
            counters[2] += nb
            f0 += nb
            if max_block_errors is not None and int(counters[1].item()) > max_block_errors:
                break
        capi.sync_check(self.dec, s)
        D.allreduce_counters(counters)
        be, ble, n = (int(v) for v in counters.cpu().tolist())
        return {"ebn0_db": ebn0_db, "frames": n, "bit_errors": be, "block_errors": ble,
                "ber": be / max(1, n * self.A), "bler": ble / max(1, n)}
