"""ctypes loader of the C-ABI library libsdrg.so (include/sdrg.h).

The product path has no CPU fallback: if the library is missing, or a call fails (e.g. no CUDA
device), an exception is raised -- ConfigError for SDRG_ERR_CONFIG, RuntimeError otherwise, the
same split libsdr makes (src/exception.hh:10-45).
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsdrg.so")

OK, ERR_CONFIG, ERR_RUNTIME, ERR_CUDA, ERR_ARG = 0, 1, 2, 3, 4

(T_UNDEFINED, T_U8, T_S8, T_U16, T_S16, T_F32, T_F64,
 T_CU8, T_CS8, T_CU16, T_CS16, T_CF32, T_CF64) = range(13)

DEMOD_NONE, DEMOD_FM, DEMOD_AM, DEMOD_USB = 0, 1, 2, 3


class SDRError(Exception):
    pass


class ConfigError(SDRError):
    pass


class RuntimeError_(SDRError, RuntimeError):
    pass


class Config(C.Structure):
    """sdr::Config (src/node.hh:35-105)."""
    _fields_ = [("type", C.c_int), ("sample_rate", C.c_double), ("buffer_size", C.c_size_t),
                ("num_buffers", C.c_size_t)]

    def __repr__(self):
        return "Config(type=%d, sample_rate=%g, buffer_size=%d, num_buffers=%d)" % (
            self.type, self.sample_rate, self.buffer_size, self.num_buffers)


class IqbbInfo(C.Structure):
    _fields_ = [("order", C.c_size_t), ("sub_sample", C.c_size_t), ("lut_inc", C.c_size_t),
                ("negative_shift", C.c_int), ("samples_consumed", C.c_uint64), ("outputs_produced", C.c_uint64)]


_V, _SZ, _I, _D = C.c_void_p, C.c_size_t, C.c_int, C.c_double
_PSZ, _PV, _PCFG = C.POINTER(C.c_size_t), C.POINTER(C.c_void_p), C.POINTER(Config)

# every symbol include/sdrg.h declares: name -> argtypes (restype is int unless noted)
SIGNATURES = {
    "sdrg_abi_version": [],
    "sdrg_build_has_experiments": [],
    "sdrg_last_error": [],
    "sdrg_device_count": [C.POINTER(C.c_int)],
    "sdrg_set_device": [_I],
    "sdrg_get_device": [C.POINTER(C.c_int)],
    "sdrg_device_synchronize": [],
    "sdrg_buffer_alloc": [_SZ, _PV],
    "sdrg_buffer_free": [_V],
    "sdrg_buffer_is_managed": [_V, C.POINTER(C.c_int)],
    "sdrg_buffer_device_ptr": [_V, _PV],
    "sdrg_buffer_mark_device_valid": [_V, _SZ, _V],
    "sdrg_buffer_device_valid": [_V, _SZ, C.POINTER(C.c_int)],
    "sdrg_buffer_invalidate_device": [_V],
    "sdrg_buffer_sync_to_host": [_V, _SZ],
    "sdrg_buffer_to_device": [_V, _SZ, _V, _PV],
    "sdrg_stream_default": [_PV],
    "sdrg_stream_synchronize": [_V],
    "sdrg_scratch": [_SZ, _PV],
    "sdrg_scratch_out": [_SZ, _PV],
    "sdrg_memcpy_h2d_async": [_V, _V, _SZ, _V],
    "sdrg_memcpy_d2h_async": [_V, _V, _SZ, _V],
    "sdrg_iqbb_create": [_I, _D, _D, _D, _SZ, _SZ, _D, _PV],
    "sdrg_iqbb_create_real": [_I, _D, _D, _D, _SZ, _SZ, _PV],
    "sdrg_iqbb_destroy": [_V],
    "sdrg_iqbb_set_center_frequency": [_V, _D],
    "sdrg_iqbb_set_filter_frequency": [_V, _D],
    "sdrg_iqbb_set_filter_width": [_V, _D],
    "sdrg_iqbb_set_order": [_V, _SZ],
    "sdrg_iqbb_set_subsample": [_V, _SZ],
    "sdrg_iqbb_set_output_sample_rate": [_V, _D],
    "sdrg_iqbb_configure": [_V, _PCFG, _PCFG],
    "sdrg_iqbb_set_float_path": [_V, _I],
    "sdrg_iqbb_last_float_kernel": [_V, C.POINTER(C.c_int)],
    "sdrg_iqbb_set_input_type": [_V, _I],
    "sdrg_autocast_out_bytes": [_I, _I, _SZ, _PSZ],
    "sdrg_autocast_process": [_I, _I, _V, _SZ, _V],
    "sdrg_autocast_process_dev": [_I, _I, _V, _SZ, _V, _V],
    "sdrg_fmdeemph_create": [_SZ, _PV],
    "sdrg_fmdeemph_destroy": [_V],
    "sdrg_fmdeemph_configure": [_V, _PCFG, _PCFG],
    "sdrg_fmdeemph_process": [_V, _V, _SZ, _SZ, _V],
    "sdrg_fmdeemph_process_dev": [_V, _V, _SZ, _SZ, _V, _V],
    "sdrg_iqbb_design": [_V, _PCFG, _PCFG],
    "sdrg_iqbb_get_info": [_V, C.POINTER(IqbbInfo), _V, _V],
    "sdrg_iqbb_process": [_V, _V, _SZ, _V, _SZ, _PSZ],
    "sdrg_iqbb_process_dev": [_V, _V, _SZ, _V, _SZ, _PSZ, _V],
    "sdrg_iqbb_outputs_for": [_V, _SZ, _PSZ],
    "sdrg_fmdemod_create": [_I, _PV],
    "sdrg_fmdemod_destroy": [_V],
    "sdrg_fmdemod_configure": [_V, _PCFG, _PCFG],
    "sdrg_fmdemod_process": [_V, _V, _SZ, _V, _I],
    "sdrg_fmdemod_process_dev": [_V, _V, _SZ, _V, _I, _V],
    "sdrg_amdemod_configure": [_I, _PCFG, _PCFG],
    "sdrg_usbdemod_configure": [_I, _PCFG, _PCFG],
    "sdrg_amdemod_process": [_I, _V, _SZ, _V],
    "sdrg_amdemod_process_dev": [_I, _V, _SZ, _V, _V],
    "sdrg_usbdemod_process": [_I, _V, _SZ, _V],
    "sdrg_usbdemod_process_dev": [_I, _V, _SZ, _V, _V],
    "sdrg_rxchain_create": [_V, _I, _PV],
    "sdrg_rxchain_destroy": [_V],
    "sdrg_rxchain_reset": [_V],
    "sdrg_rxchain_process_dev": [_V, _V, _SZ, _SZ, _V, _V, _SZ, _PSZ, _PSZ, _V],
    "sdrg_rxchain_process": [_V, _V, _SZ, _SZ, _V, _V, _SZ, _PSZ, _PSZ],
    "sdrg_fft_create": [_SZ, _I, _PV],
    "sdrg_fft_destroy": [_V],
    "sdrg_fft_exec": [_V, _V, _V, _SZ],
    "sdrg_fft_exec_dev": [_V, _V, _V, _SZ, _V],
    "sdrg_fft64_create": [_SZ, _I, _PV],
    "sdrg_fft64_destroy": [_V],
    "sdrg_fft64_exec": [_V, _V, _V, _SZ],
    "sdrg_fft64_exec_dev": [_V, _V, _V, _SZ, _V],
    "sdrg_filter_create": [_SZ, _PV],
    "sdrg_filter_destroy": [_V],
    "sdrg_filter_add": [_V, _D, _D, _PSZ],
    "sdrg_filter_set_freq": [_V, _SZ, _D, _D],
    "sdrg_filter_count": [_V, _PSZ],
    "sdrg_filter_configure": [_V, _PCFG, _PCFG],
    "sdrg_filter_get_design": [_V, _SZ, _V, _V],
    "sdrg_filter_outputs_for": [_V, _SZ, _PSZ],
    "sdrg_filter_process": [_V, _V, _SZ, _V, _SZ, _PSZ],
    "sdrg_filter_process_dev": [_V, _V, _SZ, _V, _SZ, _PSZ, _V],
    "sdrg_bank_create": [_I, _SZ, C.POINTER(C.c_double), C.POINTER(C.c_double), _D, _SZ, _SZ, _D, _PV],
    "sdrg_bank_destroy": [_V],
    "sdrg_bank_configure": [_V, _PCFG, _PCFG],
    "sdrg_bank_get_info": [_V, _PSZ, _PSZ, _SZ, C.POINTER(IqbbInfo), _V],
    "sdrg_bank_outputs_for": [_V, _SZ, _PSZ],
    "sdrg_bank_process": [_V, _V, _SZ, _SZ, _V, _V, _V, _V, _SZ, _PSZ],
    "sdrg_bank_process_dev": [_V, _V, _SZ, _SZ, _V, _V, _V, _V, _SZ, _PSZ, _V],
    "sdrg_bank_sharded_create": [_I, _SZ, C.POINTER(C.c_double), C.POINTER(C.c_double), _D, _SZ, _SZ, _D,
                                 C.POINTER(C.c_int), _SZ, _PV],
    "sdrg_bank_sharded_destroy": [_V],
    "sdrg_bank_sharded_configure": [_V, _PCFG, _PCFG],
    "sdrg_bank_sharded_info": [_V, _PSZ, _PSZ, _SZ, C.POINTER(C.c_int), _PSZ, _PSZ, C.POINTER(C.c_int)],
    "sdrg_bank_sharded_outputs_for": [_V, _SZ, _PSZ],
    "sdrg_bank_sharded_process": [_V, _V, _SZ, _SZ, _V, _V, _V, _V, _SZ, _PSZ],
    "sdrg_bank_sharded_process_dev": [_V, _V, _SZ, _SZ, _V, _V, _V, _V, _SZ, _PSZ, _V],
    "sdrg_peer_window_create": [_SZ, _PV, _V],
    "sdrg_peer_window_open": [_V, _PV],
    "sdrg_peer_window_close": [_V],
    "sdrg_peer_window_destroy": [_V],
    "sdrg_peer_signal": [_V, C.c_uint64, _V],
    "sdrg_peer_wait": [_V, _SZ, C.c_uint64, C.c_uint, _V],
    "sdrg_peer_wait_timed_out": [C.POINTER(C.c_int)],
    "sdrg_memcpy_d2d_async": [_V, _V, _SZ, _V],
    "sdrg_host_alloc": [_SZ, _I, _PV, C.POINTER(C.c_int)],
    "sdrg_host_free": [_V],
    "sdrg_kernel_launch_count": [C.POINTER(C.c_uint64)],
    "sdrg_profile_enable": [_I],
    "sdrg_profile_read": [_I, C.POINTER(C.c_double), C.POINTER(C.c_uint64)],
}

_lib = None


def load():
    """Load libsdrg.so (once). Raises if it has not been built -- there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("%s is missing: run `python -m libsdr_b200.build` (nvcc, sm_100a). "
                          "libsdr_b200 has no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_char_p if name == "sdrg_last_error" else C.c_int
    _lib = lib
    return lib


def check(rc):
    if rc == OK:
        return
    msg = load().sdrg_last_error().decode("utf-8", "replace")
    if rc == ERR_CONFIG:
        raise ConfigError(msg)
    raise RuntimeError_("sdrg error %d: %s" % (rc, msg))


def call(name, *args):
    check(getattr(load(), name)(*args))


KERNEL_IQBB_ACCUM, KERNEL_IQBB_FINALIZE, KERNEL_OLA, KERNEL_BANK = 1, 2, 3, 4


def profile_enable(on):
    call("sdrg_profile_enable", int(bool(on)))


def profile_read(kind):
    """(total device ms, launches) of the kernels of `kind` since the last read."""
    ms, n = C.c_double(0), C.c_uint64(0)
    call("sdrg_profile_read", int(kind), C.byref(ms), C.byref(n))
    return ms.value, n.value


def kernel_launch_count():
    n = C.c_uint64(0)
    call("sdrg_kernel_launch_count", C.byref(n))
    return n.value
