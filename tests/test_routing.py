"""Which kernel family a decoder runs on, read through the host emulator (tools/emu, like test_packed_walk.py): for every
decoder class over a grid of code lengths and list sizes, with POLAR_B200_FORCE_GENERIC unset, =1 and =2, the kernel
name, whether a kernel note is given, and the frames per wave for each input dtype the decoder accepts.  The expected
values are literals: a change to the host's routing or launch sizing shows up here as a changed row.  The emulator
models a device of 2 SMs, so the wave sizes are those of that device."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tools", "emu")

# decoders built inside a child process: the emulated pybind module must not meet the real package's types
_PROBE = r"""
import ctypes, json, os, sys
sys.path.insert(0, os.path.join(%(root)r, "tools", "emu"))
import check, common
import numpy as np
emu = check.load_emu()
lib = ctypes.CDLL(os.path.join(%(root)r, "tools", "emu", "build", "libpolar_b200.so"))
lib.pd_kernel_name.restype = lib.pd_kernel_note.restype = ctypes.c_char_p
lib.pd_wave_frames.restype = ctypes.c_int64


def ctor(kind, N, L, Q=16):
    K = N // 2
    extra = {"A": K - 4} if kind in common.CA_KINDS else {}
    kw, x, _ = common.make_case(kind, N, K, L=L, B=16, Q=Q, seed=11, **extra)
    if kind == "CASCLDecoder":
        kw.update(crc_n=4, crc_p=[4, 1, 0])   # four CRC bits: a CRC-24 does not fit K = 8 at N = 16
    return kw, x


out = {}
for kind, N, L, Q in %(cases)r:
    kw, _ = ctor(kind, N, L, Q)
    dec = getattr(emu, kind)(**kw)   # (kept alive: the handle is freed with the object)
    h = ctypes.c_void_p(dec._handle)
    dtypes = (0, 1, 2) if "LUT" in kind else (2,)
    out["%%s %%d %%s %%d" %% (kind, N, L, Q)] = [lib.pd_kernel_name(h).decode(), int(lib.pd_kernel_note(h) != b"")] + \
        [lib.pd_wave_frames(h, t) for t in dtypes]

# pd_decode_device with an input that starts one byte into its allocation: not 16-byte aligned, so scl_lut_warp hands
# the call to another kernel, which must give the same bits
from oracle import polar_oracle as po
kind = "SCLLUTDecoder"
kw, x = ctor(kind, 128, 4)
dec = emu.SCLLUTDecoder(**kw)
h = ctypes.c_void_p(dec._handle)
buf = np.zeros(x.size + 1, np.uint8)
buf[1:] = x.ravel()
bits = np.zeros((x.shape[0], kw["K"]), np.uint8)
rc = lib.pd_decode_device(h, ctypes.c_void_p(buf.ctypes.data + 1), 0, ctypes.c_int64(x.shape[0]),
                          ctypes.c_void_p(bits.ctypes.data), None)
rc = rc or lib.pd_check(h, None)
out["misaligned"] = dict(kernel=dec.kernel, rc=rc,
                         mismatching=int((bits != po.OracleDecoder(kind, **kw).decode(x)).any(axis=1).sum()))
print(json.dumps(out))
"""

KINDS = ["SCDecoder", "FastSCDecoder", "SCLDecoder", "FastSCLDecoder", "CASCLDecoder", "SCLUTDecoder",
         "FastSCLUTDecoder", "SCLLUTDecoder", "FastSCLLUTDecoder", "CASCLLUTDecoder", "CAFastSCLLUTDecoder",
         "SCUniformQuantizedDecoder", "SCLUniformQuantizedDecoder", "SCLloydQuantizedDecoder",
         "SCLLloydQuantizedDecoder"]
LIST_KINDS = {"SCLDecoder", "FastSCLDecoder", "CASCLDecoder", "SCLLUTDecoder", "FastSCLLUTDecoder", "CASCLLUTDecoder",
              "CAFastSCLLUTDecoder", "SCLUniformQuantizedDecoder", "SCLLloydQuantizedDecoder"}
# (kind, N, L, Q): L is "-" for the SC classes, Q is the LUT table size (Q x Q; 32 is wider than scl_lut_warp takes)
CASES = [(k, N, L, 16) for k in KINDS for N in (16, 32, 128, 1024)
         for L in ((1, 2, 3, 8, 32, 64) if k in LIST_KINDS else ("-",)) if not (L == 64 and N < 32)]
CASES += [("SCLLUTDecoder", 128, 8, 32), ("SCLUTDecoder", 1024, "-", 32)]

# kind N L Q | FORCE_GENERIC unset | =1 | =2; each column: kernel name ("+note" when pd_kernel_note is not empty), then the
# frames per wave for PD_U8, PD_I32 and PD_F64 symbols (LUT classes) or PD_F64 LLRs (the others)
EXPECTED = """
SCDecoder 16 - 16                     | generic 0                     | generic 0              | generic 0
SCDecoder 32 - 16                     | path_warp 2048                | generic 0              | path_warp 2048
SCDecoder 128 - 16                    | path_warp 2048                | generic 0              | path_warp 2048
SCDecoder 1024 - 16                   | path_warp 1856                | generic 0              | path_warp 1856
FastSCDecoder 16 - 16                 | generic 0                     | generic 0              | generic 0
FastSCDecoder 32 - 16                 | path_warp 2048                | generic 0              | path_warp 2048
FastSCDecoder 128 - 16                | path_warp 2048                | generic 0              | path_warp 2048
FastSCDecoder 1024 - 16               | path_warp 1856                | generic 0              | path_warp 1856
SCLDecoder 16 1 16                    | generic 0                     | generic 0              | generic 0
SCLDecoder 16 2 16                    | generic 0                     | generic 0              | generic 0
SCLDecoder 16 3 16                    | generic 0                     | generic 0              | generic 0
SCLDecoder 16 8 16                    | generic 0                     | generic 0              | generic 0
SCLDecoder 16 32 16                   | generic 0                     | generic 0              | generic 0
SCLDecoder 32 1 16                    | generic 0                     | generic 0              | generic 0
SCLDecoder 32 2 16                    | path_warp 1024                | generic 0              | path_warp 1024
SCLDecoder 32 3 16                    | generic 0                     | generic 0              | generic 0
SCLDecoder 32 8 16                    | path_warp 256                 | generic 0              | path_warp 256
SCLDecoder 32 32 16                   | path_warp 64                  | generic 0              | path_warp 64
SCLDecoder 32 64 16                   | path_cta 50                   | path_cta 50            | path_cta 50
SCLDecoder 128 1 16                   | generic 0                     | generic 0              | generic 0
SCLDecoder 128 2 16                   | path_warp 1024                | generic 0              | path_warp 1024
SCLDecoder 128 3 16                   | generic 0                     | generic 0              | generic 0
SCLDecoder 128 8 16                   | path_warp 256                 | generic 0              | path_warp 256
SCLDecoder 128 32 16                  | path_warp 64                  | generic 0              | path_warp 64
SCLDecoder 128 64 16                  | path_cta 46                   | path_cta 46            | path_cta 46
SCLDecoder 1024 1 16                  | generic 0                     | generic 0              | generic 0
SCLDecoder 1024 2 16                  | path_warp 736                 | generic 0              | path_warp 736
SCLDecoder 1024 3 16                  | generic 0                     | generic 0              | generic 0
SCLDecoder 1024 8 16                  | path_warp 224                 | generic 0              | path_warp 224
SCLDecoder 1024 32 16                 | path_warp 58                  | generic 0              | path_warp 58
SCLDecoder 1024 64 16                 | path_cta 26                   | path_cta 26            | path_cta 26
FastSCLDecoder 16 1 16                | generic 0                     | generic 0              | generic 0
FastSCLDecoder 16 2 16                | generic 0                     | generic 0              | generic 0
FastSCLDecoder 16 3 16                | generic 0                     | generic 0              | generic 0
FastSCLDecoder 16 8 16                | generic 0                     | generic 0              | generic 0
FastSCLDecoder 16 32 16               | generic 0                     | generic 0              | generic 0
FastSCLDecoder 32 1 16                | generic 0                     | generic 0              | generic 0
FastSCLDecoder 32 2 16                | path_warp 1024                | generic 0              | path_warp 1024
FastSCLDecoder 32 3 16                | generic 0                     | generic 0              | generic 0
FastSCLDecoder 32 8 16                | path_warp 256                 | generic 0              | path_warp 256
FastSCLDecoder 32 32 16               | path_warp 64                  | generic 0              | path_warp 64
FastSCLDecoder 32 64 16               | path_cta 50                   | path_cta 50            | path_cta 50
FastSCLDecoder 128 1 16               | generic 0                     | generic 0              | generic 0
FastSCLDecoder 128 2 16               | path_warp 1024                | generic 0              | path_warp 1024
FastSCLDecoder 128 3 16               | generic 0                     | generic 0              | generic 0
FastSCLDecoder 128 8 16               | path_warp 256                 | generic 0              | path_warp 256
FastSCLDecoder 128 32 16              | path_warp 64                  | generic 0              | path_warp 64
FastSCLDecoder 128 64 16              | path_cta 46                   | path_cta 46            | path_cta 46
FastSCLDecoder 1024 1 16              | generic 0                     | generic 0              | generic 0
FastSCLDecoder 1024 2 16              | path_warp 736                 | generic 0              | path_warp 736
FastSCLDecoder 1024 3 16              | generic 0                     | generic 0              | generic 0
FastSCLDecoder 1024 8 16              | path_warp 224                 | generic 0              | path_warp 224
FastSCLDecoder 1024 32 16             | path_warp 58                  | generic 0              | path_warp 58
FastSCLDecoder 1024 64 16             | path_cta 26                   | path_cta 26            | path_cta 26
CASCLDecoder 16 1 16                  | generic 0                     | generic 0              | generic 0
CASCLDecoder 16 2 16                  | generic 0                     | generic 0              | generic 0
CASCLDecoder 16 3 16                  | generic 0                     | generic 0              | generic 0
CASCLDecoder 16 8 16                  | generic 0                     | generic 0              | generic 0
CASCLDecoder 16 32 16                 | generic 0                     | generic 0              | generic 0
CASCLDecoder 32 1 16                  | generic 0                     | generic 0              | generic 0
CASCLDecoder 32 2 16                  | path_warp 1024                | generic 0              | path_warp 1024
CASCLDecoder 32 3 16                  | generic 0                     | generic 0              | generic 0
CASCLDecoder 32 8 16                  | path_warp 256                 | generic 0              | path_warp 256
CASCLDecoder 32 32 16                 | path_warp 64                  | generic 0              | path_warp 64
CASCLDecoder 32 64 16                 | path_cta 50                   | path_cta 50            | path_cta 50
CASCLDecoder 128 1 16                 | generic 0                     | generic 0              | generic 0
CASCLDecoder 128 2 16                 | path_warp 1024                | generic 0              | path_warp 1024
CASCLDecoder 128 3 16                 | generic 0                     | generic 0              | generic 0
CASCLDecoder 128 8 16                 | path_warp 256                 | generic 0              | path_warp 256
CASCLDecoder 128 32 16                | path_warp 64                  | generic 0              | path_warp 64
CASCLDecoder 128 64 16                | path_cta 46                   | path_cta 46            | path_cta 46
CASCLDecoder 1024 1 16                | generic 0                     | generic 0              | generic 0
CASCLDecoder 1024 2 16                | path_warp 736                 | generic 0              | path_warp 736
CASCLDecoder 1024 3 16                | generic 0                     | generic 0              | generic 0
CASCLDecoder 1024 8 16                | path_warp 224                 | generic 0              | path_warp 224
CASCLDecoder 1024 32 16               | path_warp 58                  | generic 0              | path_warp 58
CASCLDecoder 1024 64 16               | path_cta 26                   | path_cta 26            | path_cta 26
SCLUTDecoder 16 - 16                  | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
SCLUTDecoder 32 - 16                  | scl_lut_warp 4096 4096 2048   | generic 0 0 0          | path_warp 2048 2048 2048
SCLUTDecoder 128 - 16                 | scl_lut_warp 3456 3456 2048   | generic 0 0 0          | path_warp 2048 2048 2048
SCLUTDecoder 1024 - 16                | scl_lut_warp 1792 1792 2048   | generic 0 0 0          | path_warp 2048 2048 2048
FastSCLUTDecoder 16 - 16              | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
FastSCLUTDecoder 32 - 16              | scl_lut_warp 4096 4096 2048   | generic 0 0 0          | path_warp 2048 2048 2048
FastSCLUTDecoder 128 - 16             | scl_lut_warp 3328 3328 2048   | generic 0 0 0          | path_warp 2048 2048 2048
FastSCLUTDecoder 1024 - 16            | scl_lut_warp 1792 1792 2048   | generic 0 0 0          | path_warp 2048 2048 2048
SCLLUTDecoder 16 1 16                 | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
SCLLUTDecoder 16 2 16                 | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
SCLLUTDecoder 16 3 16                 | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
SCLLUTDecoder 16 8 16                 | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
SCLLUTDecoder 16 32 16                | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
SCLLUTDecoder 32 1 16                 | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
SCLLUTDecoder 32 2 16                 | scl_lut_warp 2048 2048 1024   | generic 0 0 0          | path_warp 1024 1024 1024
SCLLUTDecoder 32 3 16                 | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
SCLLUTDecoder 32 8 16                 | scl_lut_warp 512 512 256      | generic 0 0 0          | path_warp 256 256 256
SCLLUTDecoder 32 32 16                | path_warp+note 64 64 64       | generic+note 0 0 0     | path_warp+note 64 64 64
SCLLUTDecoder 32 64 16                | path_cta+note 64 64 64        | path_cta+note 64 64 64 | path_cta+note 64 64 64
SCLLUTDecoder 128 1 16                | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
SCLLUTDecoder 128 2 16                | scl_lut_warp 1728 1728 1024   | generic 0 0 0          | path_warp 1024 1024 1024
SCLLUTDecoder 128 3 16                | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
SCLLUTDecoder 128 8 16                | scl_lut_warp 432 432 256      | generic 0 0 0          | path_warp 256 256 256
SCLLUTDecoder 128 32 16               | path_warp+note 64 64 64       | generic+note 0 0 0     | path_warp+note 64 64 64
SCLLUTDecoder 128 64 16               | path_cta+note 64 64 64        | path_cta+note 64 64 64 | path_cta+note 64 64 64
SCLLUTDecoder 1024 1 16               | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
SCLLUTDecoder 1024 2 16               | scl_lut_warp 704 704 896      | generic 0 0 0          | path_warp 896 896 896
SCLLUTDecoder 1024 3 16               | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
SCLLUTDecoder 1024 8 16               | scl_lut_warp 224 224 256      | generic 0 0 0          | path_warp 256 256 256
SCLLUTDecoder 1024 32 16              | path_warp+note 64 64 64       | generic+note 0 0 0     | path_warp+note 64 64 64
SCLLUTDecoder 1024 64 16              | path_cta+note 32 32 32        | path_cta+note 32 32 32 | path_cta+note 32 32 32
FastSCLLUTDecoder 16 1 16             | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
FastSCLLUTDecoder 16 2 16             | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
FastSCLLUTDecoder 16 3 16             | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
FastSCLLUTDecoder 16 8 16             | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
FastSCLLUTDecoder 16 32 16            | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
FastSCLLUTDecoder 32 1 16             | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
FastSCLLUTDecoder 32 2 16             | scl_lut_warp 384 384 1024     | generic 0 0 0          | path_warp 1024 1024 1024
FastSCLLUTDecoder 32 3 16             | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
FastSCLLUTDecoder 32 8 16             | scl_lut_warp 96 96 256        | generic 0 0 0          | path_warp 256 256 256
FastSCLLUTDecoder 32 32 16            | path_warp+note 64 64 64       | generic+note 0 0 0     | path_warp+note 64 64 64
FastSCLLUTDecoder 32 64 16            | path_cta+note 64 64 64        | path_cta+note 64 64 64 | path_cta+note 64 64 64
FastSCLLUTDecoder 128 1 16            | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
FastSCLLUTDecoder 128 2 16            | scl_lut_warp 384 384 1024     | generic 0 0 0          | path_warp 1024 1024 1024
FastSCLLUTDecoder 128 3 16            | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
FastSCLLUTDecoder 128 8 16            | scl_lut_warp 96 96 256        | generic 0 0 0          | path_warp 256 256 256
FastSCLLUTDecoder 128 32 16           | path_warp+note 64 64 64       | generic+note 0 0 0     | path_warp+note 64 64 64
FastSCLLUTDecoder 128 64 16           | path_cta+note 64 64 64        | path_cta+note 64 64 64 | path_cta+note 64 64 64
FastSCLLUTDecoder 1024 1 16           | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
FastSCLLUTDecoder 1024 2 16           | scl_lut_warp 384 384 896      | generic 0 0 0          | path_warp 896 896 896
FastSCLLUTDecoder 1024 3 16           | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
FastSCLLUTDecoder 1024 8 16           | scl_lut_warp 96 96 256        | generic 0 0 0          | path_warp 256 256 256
FastSCLLUTDecoder 1024 32 16          | path_warp+note 64 64 64       | generic+note 0 0 0     | path_warp+note 64 64 64
FastSCLLUTDecoder 1024 64 16          | path_cta+note 32 32 32        | path_cta+note 32 32 32 | path_cta+note 32 32 32
CASCLLUTDecoder 16 1 16               | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CASCLLUTDecoder 16 2 16               | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CASCLLUTDecoder 16 3 16               | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CASCLLUTDecoder 16 8 16               | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CASCLLUTDecoder 16 32 16              | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CASCLLUTDecoder 32 1 16               | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CASCLLUTDecoder 32 2 16               | scl_lut_warp 2048 2048 1024   | generic 0 0 0          | path_warp 1024 1024 1024
CASCLLUTDecoder 32 3 16               | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CASCLLUTDecoder 32 8 16               | scl_lut_warp 512 512 256      | generic 0 0 0          | path_warp 256 256 256
CASCLLUTDecoder 32 32 16              | path_warp+note 64 64 64       | generic+note 0 0 0     | path_warp+note 64 64 64
CASCLLUTDecoder 32 64 16              | path_cta+note 64 64 64        | path_cta+note 64 64 64 | path_cta+note 64 64 64
CASCLLUTDecoder 128 1 16              | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CASCLLUTDecoder 128 2 16              | scl_lut_warp 1728 1728 1024   | generic 0 0 0          | path_warp 1024 1024 1024
CASCLLUTDecoder 128 3 16              | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CASCLLUTDecoder 128 8 16              | scl_lut_warp 432 432 256      | generic 0 0 0          | path_warp 256 256 256
CASCLLUTDecoder 128 32 16             | path_warp+note 64 64 64       | generic+note 0 0 0     | path_warp+note 64 64 64
CASCLLUTDecoder 128 64 16             | path_cta+note 64 64 64        | path_cta+note 64 64 64 | path_cta+note 64 64 64
CASCLLUTDecoder 1024 1 16             | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CASCLLUTDecoder 1024 2 16             | scl_lut_warp 704 704 896      | generic 0 0 0          | path_warp 896 896 896
CASCLLUTDecoder 1024 3 16             | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CASCLLUTDecoder 1024 8 16             | scl_lut_warp 224 224 256      | generic 0 0 0          | path_warp 256 256 256
CASCLLUTDecoder 1024 32 16            | path_warp+note 64 64 64       | generic+note 0 0 0     | path_warp+note 64 64 64
CASCLLUTDecoder 1024 64 16            | path_cta+note 32 32 32        | path_cta+note 32 32 32 | path_cta+note 32 32 32
CAFastSCLLUTDecoder 16 1 16           | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CAFastSCLLUTDecoder 16 2 16           | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CAFastSCLLUTDecoder 16 3 16           | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CAFastSCLLUTDecoder 16 8 16           | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CAFastSCLLUTDecoder 16 32 16          | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CAFastSCLLUTDecoder 32 1 16           | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CAFastSCLLUTDecoder 32 2 16           | scl_lut_warp 384 384 1024     | generic 0 0 0          | path_warp 1024 1024 1024
CAFastSCLLUTDecoder 32 3 16           | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CAFastSCLLUTDecoder 32 8 16           | scl_lut_warp 96 96 256        | generic 0 0 0          | path_warp 256 256 256
CAFastSCLLUTDecoder 32 32 16          | path_warp+note 64 64 64       | generic+note 0 0 0     | path_warp+note 64 64 64
CAFastSCLLUTDecoder 32 64 16          | path_cta+note 64 64 64        | path_cta+note 64 64 64 | path_cta+note 64 64 64
CAFastSCLLUTDecoder 128 1 16          | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CAFastSCLLUTDecoder 128 2 16          | scl_lut_warp 384 384 1024     | generic 0 0 0          | path_warp 1024 1024 1024
CAFastSCLLUTDecoder 128 3 16          | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CAFastSCLLUTDecoder 128 8 16          | scl_lut_warp 96 96 256        | generic 0 0 0          | path_warp 256 256 256
CAFastSCLLUTDecoder 128 32 16         | path_warp+note 64 64 64       | generic+note 0 0 0     | path_warp+note 64 64 64
CAFastSCLLUTDecoder 128 64 16         | path_cta+note 64 64 64        | path_cta+note 64 64 64 | path_cta+note 64 64 64
CAFastSCLLUTDecoder 1024 1 16         | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CAFastSCLLUTDecoder 1024 2 16         | scl_lut_warp 384 384 896      | generic 0 0 0          | path_warp 896 896 896
CAFastSCLLUTDecoder 1024 3 16         | generic+note 0 0 0            | generic+note 0 0 0     | generic+note 0 0 0
CAFastSCLLUTDecoder 1024 8 16         | scl_lut_warp 96 96 256        | generic 0 0 0          | path_warp 256 256 256
CAFastSCLLUTDecoder 1024 32 16        | path_warp+note 64 64 64       | generic+note 0 0 0     | path_warp+note 64 64 64
CAFastSCLLUTDecoder 1024 64 16        | path_cta+note 32 32 32        | path_cta+note 32 32 32 | path_cta+note 32 32 32
SCUniformQuantizedDecoder 16 - 16     | generic 0                     | generic 0              | generic 0
SCUniformQuantizedDecoder 32 - 16     | path_warp 2048                | generic 0              | path_warp 2048
SCUniformQuantizedDecoder 128 - 16    | path_warp 2048                | generic 0              | path_warp 2048
SCUniformQuantizedDecoder 1024 - 16   | path_warp 1856                | generic 0              | path_warp 1856
SCLUniformQuantizedDecoder 16 1 16    | generic 0                     | generic 0              | generic 0
SCLUniformQuantizedDecoder 16 2 16    | generic 0                     | generic 0              | generic 0
SCLUniformQuantizedDecoder 16 3 16    | generic 0                     | generic 0              | generic 0
SCLUniformQuantizedDecoder 16 8 16    | generic 0                     | generic 0              | generic 0
SCLUniformQuantizedDecoder 16 32 16   | generic 0                     | generic 0              | generic 0
SCLUniformQuantizedDecoder 32 1 16    | generic 0                     | generic 0              | generic 0
SCLUniformQuantizedDecoder 32 2 16    | path_warp 1024                | generic 0              | path_warp 1024
SCLUniformQuantizedDecoder 32 3 16    | generic 0                     | generic 0              | generic 0
SCLUniformQuantizedDecoder 32 8 16    | path_warp 256                 | generic 0              | path_warp 256
SCLUniformQuantizedDecoder 32 32 16   | path_warp 64                  | generic 0              | path_warp 64
SCLUniformQuantizedDecoder 32 64 16   | path_cta 50                   | path_cta 50            | path_cta 50
SCLUniformQuantizedDecoder 128 1 16   | generic 0                     | generic 0              | generic 0
SCLUniformQuantizedDecoder 128 2 16   | path_warp 1024                | generic 0              | path_warp 1024
SCLUniformQuantizedDecoder 128 3 16   | generic 0                     | generic 0              | generic 0
SCLUniformQuantizedDecoder 128 8 16   | path_warp 256                 | generic 0              | path_warp 256
SCLUniformQuantizedDecoder 128 32 16  | path_warp 64                  | generic 0              | path_warp 64
SCLUniformQuantizedDecoder 128 64 16  | path_cta 46                   | path_cta 46            | path_cta 46
SCLUniformQuantizedDecoder 1024 1 16  | generic 0                     | generic 0              | generic 0
SCLUniformQuantizedDecoder 1024 2 16  | path_warp 736                 | generic 0              | path_warp 736
SCLUniformQuantizedDecoder 1024 3 16  | generic 0                     | generic 0              | generic 0
SCLUniformQuantizedDecoder 1024 8 16  | path_warp 224                 | generic 0              | path_warp 224
SCLUniformQuantizedDecoder 1024 32 16 | path_warp 58                  | generic 0              | path_warp 58
SCLUniformQuantizedDecoder 1024 64 16 | path_cta 26                   | path_cta 26            | path_cta 26
SCLloydQuantizedDecoder 16 - 16       | generic 0                     | generic 0              | generic 0
SCLloydQuantizedDecoder 32 - 16       | path_warp 2048                | generic 0              | path_warp 2048
SCLloydQuantizedDecoder 128 - 16      | path_warp 2048                | generic 0              | path_warp 2048
SCLloydQuantizedDecoder 1024 - 16     | path_warp 1856                | generic 0              | path_warp 1856
SCLLloydQuantizedDecoder 16 1 16      | generic 0                     | generic 0              | generic 0
SCLLloydQuantizedDecoder 16 2 16      | generic 0                     | generic 0              | generic 0
SCLLloydQuantizedDecoder 16 3 16      | generic 0                     | generic 0              | generic 0
SCLLloydQuantizedDecoder 16 8 16      | generic 0                     | generic 0              | generic 0
SCLLloydQuantizedDecoder 16 32 16     | generic 0                     | generic 0              | generic 0
SCLLloydQuantizedDecoder 32 1 16      | generic 0                     | generic 0              | generic 0
SCLLloydQuantizedDecoder 32 2 16      | path_warp 1024                | generic 0              | path_warp 1024
SCLLloydQuantizedDecoder 32 3 16      | generic 0                     | generic 0              | generic 0
SCLLloydQuantizedDecoder 32 8 16      | path_warp 256                 | generic 0              | path_warp 256
SCLLloydQuantizedDecoder 32 32 16     | path_warp 64                  | generic 0              | path_warp 64
SCLLloydQuantizedDecoder 32 64 16     | path_cta 50                   | path_cta 50            | path_cta 50
SCLLloydQuantizedDecoder 128 1 16     | generic 0                     | generic 0              | generic 0
SCLLloydQuantizedDecoder 128 2 16     | path_warp 1024                | generic 0              | path_warp 1024
SCLLloydQuantizedDecoder 128 3 16     | generic 0                     | generic 0              | generic 0
SCLLloydQuantizedDecoder 128 8 16     | path_warp 256                 | generic 0              | path_warp 256
SCLLloydQuantizedDecoder 128 32 16    | path_warp 64                  | generic 0              | path_warp 64
SCLLloydQuantizedDecoder 128 64 16    | path_cta 46                   | path_cta 46            | path_cta 46
SCLLloydQuantizedDecoder 1024 1 16    | generic 0                     | generic 0              | generic 0
SCLLloydQuantizedDecoder 1024 2 16    | path_warp 736                 | generic 0              | path_warp 736
SCLLloydQuantizedDecoder 1024 3 16    | generic 0                     | generic 0              | generic 0
SCLLloydQuantizedDecoder 1024 8 16    | path_warp 224                 | generic 0              | path_warp 224
SCLLloydQuantizedDecoder 1024 32 16   | path_warp 58                  | generic 0              | path_warp 58
SCLLloydQuantizedDecoder 1024 64 16   | path_cta 26                   | path_cta 26            | path_cta 26
SCLLUTDecoder 128 8 32                | path_warp+note 256 256 256    | generic+note 0 0 0     | path_warp+note 256 256 256
SCLUTDecoder 1024 - 32                | path_warp+note 2048 2048 2048 | generic+note 0 0 0     | path_warp+note 2048 2048 2048
"""


def _expected():
    rows = {}
    for line in EXPECTED.strip().splitlines():
        key, *cols = [c.strip() for c in line.split("|")]
        rows[" ".join(key.split())] = [c.split() for c in cols]
    return rows


def _row(r):
    name, note, *waves = r
    return [name + ("+note" if note else "")] + [str(w) for w in waves]


@pytest.fixture(scope="module")
def probes():
    r = subprocess.run(["bash", os.path.join(EMU, "build.sh")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    out = []
    for force in (None, "1", "2"):
        env = {k: v for k, v in os.environ.items() if not k.startswith(("POLAR_B200_", "PB_EMU_"))}
        env["POLAR_B200_QUIET"] = "1"
        if force:
            env["POLAR_B200_FORCE_GENERIC"] = force
        r = subprocess.run([sys.executable, "-c", _PROBE % dict(root=ROOT, cases=CASES)], capture_output=True, text=True,
                           timeout=900, cwd=EMU, env=env)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        out.append(json.loads(r.stdout.strip().splitlines()[-1]))
    return out


def test_kernel_note_and_wave_per_case(probes):
    want = _expected()
    got = {key: [_row(p[key]) for p in probes] for key in probes[0] if key != "misaligned"}
    assert set(got) == set(want)
    bad = {key: (got[key], want[key]) for key in got if got[key] != want[key]}
    assert not bad, bad


def test_misaligned_device_input_decodes_like_the_oracle(probes):
    for p in probes:
        m = p["misaligned"]
        assert m["rc"] == 0 and m["mismatching"] == 0, m
    assert probes[0]["misaligned"]["kernel"] == "scl_lut_warp"
