"""ctypes prototypes of the C ABI (include/polar_b200.h) for callers that already hold device pointers
(bench.py, the torch.distributed front-end, tests).  Decoder objects are created through the pybind11
classes; their `_handle` attribute is the `pd_decoder*` these functions take."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpolar_b200.so")

PD_U8, PD_I32, PD_F64 = 0, 1, 2
PD_OK, PD_EINVAL, PD_ECUDA, PD_ERANGE, PD_ENOMEM = 0, 1, 2, 3, 4
PD_SIM_LLR, PD_SIM_LLR_QUANT, PD_SIM_Y_QUANT, PD_SIM_LLR_UNIFORM = 0, 1, 2, 3      # pd_sim_channel.mode

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is not built (python -m quantized_decoder_polar_codes_b200.build); no CPU fallback exists")
        L = C.CDLL(LIB_PATH)
        L.pd_last_error.restype = C.c_char_p
        L.pd_version.restype = C.c_char_p
        L.pd_kernel_name.restype = C.c_char_p
        L.pd_kernel_name.argtypes = [C.c_void_p]
        L.pd_kernel_note.restype = C.c_char_p
        L.pd_kernel_note.argtypes = [C.c_void_p]
        L.pd_launch_count.restype = C.c_int64
        L.pd_out_len.argtypes = [C.c_void_p]
        L.pd_code_len.argtypes = [C.c_void_p]
        L.pd_wave_frames.restype = C.c_int64
        L.pd_wave_frames.argtypes = [C.c_void_p, C.c_int]
        L.pd_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p]
        L.pd_decode_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p]
        L.pd_check.argtypes = [C.c_void_p, C.c_void_p]
        L.pd_set_debug_outputs.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.pd_count_errors.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]
        L.pd_schedule_stats.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.pd_host_alloc.restype = C.c_void_p
        L.pd_host_alloc.argtypes = [C.c_size_t]
        L.pd_host_free.argtypes = [C.c_void_p]
        L.pd_destroy.argtypes = [C.c_void_p]
        L.pd_sim_create.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        L.pd_sim_destroy.argtypes = [C.c_void_p]
        L.pd_sim_generate.argtypes = [C.c_void_p, C.c_double, C.c_int64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
        L.pd_sim_set_channel.argtypes = [C.c_void_p, C.c_void_p]
        L.pd_sim_encode.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p]
        L.pd_sim_encode_device.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
        L.pd_decode_bd.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.pd_decode_bd_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.pd_mmi_slice_sums.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32]
        L.pd_mmi_design.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32]
        L.pd_optls_quantize.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]
        _lib = L
    return _lib


class PolarError(RuntimeError):
    pass


def check(rc):
    if rc != PD_OK:
        msg = lib().pd_last_error().decode()
        raise (ValueError if rc in (PD_EINVAL, PD_ERANGE) else PolarError)(msg)


def decode_device(decoder, dev_in_ptr, dtype, B, dev_out_ptr, stream=0):
    """Asynchronous decode of B device-resident frames (pd_decode_device)."""
    check(lib().pd_decode_device(decoder._handle, dev_in_ptr, dtype, B, dev_out_ptr, stream))


def decode_host(decoder, host_in_ptr, dtype, B, host_out_ptr):
    check(lib().pd_decode(decoder._handle, host_in_ptr, dtype, B, host_out_ptr))


def wave_frames(decoder, dtype):
    """Frames one full wave of the persistent decode kernel holds (pd_wave_frames); 0 = CTA-per-frame kernel."""
    return int(lib().pd_wave_frames(decoder._handle, dtype))


def sync_check(decoder, stream=0):
    check(lib().pd_check(decoder._handle, stream))


def schedule_stats(decoder):
    a, b, c = C.c_int64(), C.c_int64(), C.c_int64()
    check(lib().pd_schedule_stats(decoder._handle, C.byref(a), C.byref(b), C.byref(c)))
    return {"steps": a.value, "elem_ops_per_path": b.value, "sorts": c.value}


class SimConfig(C.Structure):
    _fields_ = [("N", C.c_int32), ("K", C.c_int32), ("A", C.c_int32), ("device", C.c_int32),
                ("frozen_bits", C.c_void_p), ("crc_n", C.c_int32), ("crc_loc", C.c_void_p), ("crc_loc_len", C.c_int32),
                ("edges", C.c_void_p), ("n_edges", C.c_int32), ("chan_lut", C.c_void_p), ("q_channel", C.c_int32)]


class SimChannel(C.Structure):
    _fields_ = [("mode", C.c_int32), ("edges", C.c_void_p), ("n_edges", C.c_int32), ("chan_lut", C.c_void_p),
                ("q_channel", C.c_int32), ("r", C.c_double), ("v", C.c_int32)]
